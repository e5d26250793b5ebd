// sbd.cu - libsbd.so: context, launch logic and the C ABI of include/sbd.h.
// Hand-written CUDA for sm_100a, fp64.  No CPU fallback anywhere in this file:
// every numerical result is produced by the kernels in tv.cuh / fft.cuh /
// sapg.cuh / psf.cuh; the host code only sequences launches and post-processes
// scalar trajectories (running means, Guassian.m:218-247).
#include "common.cuh"
#include "philox.cuh"
#include "psf.cuh"
#include "tv.cuh"
#include "tv_multi.cuh"
#include "tv_coop.cuh"
#include "fft.cuh"
#include "fft2.cuh"
#include "fft_any.cuh"
#include "sapg.cuh"

#include <dlfcn.h>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <limits>
#include <map>

using namespace sbd;

// ---------------------------------------------------------------------------
// NCCL through dlopen (keeps libsbd.so loadable without NCCL; multi-GPU calls
// fail loudly with SBD_E_COMM if it cannot be found).
// ---------------------------------------------------------------------------
namespace {
typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm;
struct NcclApi {
    void* h = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm*, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, nccl_comm, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool load() {
        if (h) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) return false;
        GetUniqueId = (int (*)(nccl_uid*))dlsym(h, "ncclGetUniqueId");
        CommInitRank = (int (*)(nccl_comm*, int, nccl_uid, int))dlsym(h, "ncclCommInitRank");
        CommDestroy = (int (*)(nccl_comm))dlsym(h, "ncclCommDestroy");
        AllGather = (int (*)(const void*, void*, size_t, int, nccl_comm, cudaStream_t))dlsym(h, "ncclAllGather");
        GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && CommDestroy && AllGather;
    }
};
NcclApi g_nccl;
constexpr int NCCL_FLOAT64 = 8;     // ncclDouble
std::string g_create_error;
}  // namespace

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
struct sbd_ctx {
    int device = 0;
    int nx = 0, ny = 0;             // rows (fast) / cols (slow)
    int t = 7, model = 0;
    double phi = 0.0;
    int max_batch = 1;
    bool pow2 = false;              // FFT passes of fft.cuh / fft2.cuh
    bool smooth = false;            // every other size the FFT operators take: fft_any.cuh (fft_plan.h)
    std::string fft_err;            // why the FFT operators refuse this size ("" when they take it)
    AnyPlan plan_x = {}, plan_y = {};   // smooth: plans of the rows (length nx) and column (length ny) passes
    size_t npix = 0;
    int sp = 0, nk = 0;             // half-spectrum pitch / number of bins (nx/2+1)
    size_t spec_elems = 0;          // per image, in double2
    cudaStream_t stream = nullptr;
    long long launches = 0;
    std::string err;

    // geometry
    int tvV = 1, tv_gx = 1, tv_gy = 1, tv_seg = 8, tv_parts = 1;
    int sm_count = 148, fft_pf = 1;                                     // L2 prefetch distance of the FFT passes
    int cmT = 5, cm_strips = 1, cm_gx = 1, cm_gy = 1, cm_seg = 128;     // fused Chambolle geometry
    bool cm_pipe = false, cm_emit = true, cm_plan33 = true;
    double salsa_mu = 0.0;
    int cm_minb = 3;
    int rowsLP = 1, rowsT = 32, colsC = 2, colsLogC = 1, colsT = 32, ntiles = 1;
    int colsKC = 2, colsLogKC = 1;     // columns per block of the column pass (<= colsC, the layout tile width)
    size_t rows_smem = 0, cols_smem = 0;
    // v2 passes (fft2.cuh): column-contiguous spectrum, bulk / tensor copies.  Tensor maps of the spectra buffers
    // the rows passes write (S1, Y^) or read (S2, S1), built when the buffers are allocated.
    bool v2 = false;
    CUtensorMap tm_S1, tm_S2, tm_yhat;
    int geom_batch = -1;
    // launch-geometry overrides (sbd_set_option; -1 = automatic).  Seeded from the SBD_* environment at sbd_create.
    int opt_chamb_seg = -1, opt_chamb_T = -1, opt_tv_seg = -1, opt_chamb_emit = -1, opt_chamb_plan33 = -1;
    int opt_chamb_errsub = -1;      // sampled stop test of the fused Chambolle kernel: -1 automatic, 0 never, 1 whenever allowed
    // The segment lengths fix the summation order of the TV-norm and err_k partial sums, so they must not depend
    // on how many of a run's chains happen to live on this GPU: inside a SAPG run the geometry is derived from
    // the TOTAL number of chains over all ranks (0 = use the batch of the call).
    int geom_total = 0;
    // per-context (= per-device) caches of kernel attributes: cudaFuncSetAttribute is per device
    std::map<const void*, size_t> smem_optin;
    std::map<std::pair<const void*, size_t>, int> resident_cache;

    // device buffers
    double2 *tw_nx = nullptr, *tw_ny = nullptr;
    double* taps = nullptr;         // [3][t*t]
    double2* coef = nullptr;        // [3][nx][MAXT]
    Control* ctl = nullptr;
    ChambState* chst = nullptr;
    unsigned int *cnt_tv = nullptr, *cnt_col = nullptr, *cnt_sq = nullptr;
    double *stats = nullptr, *allstats = nullptr;
    double *part_tv = nullptr, *part_ch = nullptr, *part_col = nullptr, *part_sq = nullptr;
    double *in_y = nullptr, *in_x0 = nullptr, *in_xt = nullptr;         // staging images of the host-pointer entries
    double* psi_dev = nullptr;      // [2] override for operator calls
    // workspaces (sized for ws_batch images)
    int ws_batch = 0;
    double *X = nullptr, *P = nullptr, *Gf = nullptr, *px0 = nullptr, *py0 = nullptr, *px1 = nullptr, *py1 = nullptr;
    double2 *S1 = nullptr, *S2 = nullptr, *yhat = nullptr;
    double *ximg = nullptr;         // 1-image staging (y, x_true)
    double *post = nullptr;
    int post_batch = 0;
    // posterior statistics (sbd_set_posterior / sbd_posterior_stats, DESIGN.md "Posterior statistics")
    int post_levels = 0;                    // sticky request: block sizes 1 .. 2^(post_levels-1), 0 = off
    double* post_m2 = nullptr;              // pixel-scale M2 next to `post`, [post_m2_batch][npix]
    int post_m2_batch = 0;
    double* post_blk = nullptr; size_t post_blk_cap = 0;    // m and M2 of the levels >= 1, [2][sum_j n_chains*nb_j]
    double* post_out = nullptr; size_t post_out_cap = 0;    // mean, within, between of every level of the last run
    int stat_levels = 0, stat_n = 0, stat_chains = 0;       // what post_out holds (stat_levels 0: nothing)
    // batch means and split halves (sbd_set_posterior_diagnostics / sbd_posterior_diagnostics, DiagAcc in sapg.cuh)
    int post_diag = 0;                      // sticky request: 0 off, -1 batch length floor(sqrt(n)), b >= 1
    double* diag_pix = nullptr; int diag_pix_batch = 0;     // pixel scale: 7 images per chain (DiagAcc layout)
    double* diag_blk = nullptr; size_t diag_blk_cap = 0;    // levels >= 1: [7][sum_j n_chains*nb_j]
    double* diag_out = nullptr; size_t diag_out_cap = 0;    // per level: batch mean/within/between, half mean/within/between
    int diag_levels = 0, diag_b = 0, diag_nbatch = 0, diag_h = 0;   // what diag_out holds (diag_levels 0: nothing)
    // credible intervals and median (sbd_set_posterior_quantiles / sbd_posterior_quantiles, QuantAcc in sapg.cuh)
    double post_ci = 0.0;                   // sticky request: 0 off, else the credible level alpha in (0, 1)
    double* quant_q = nullptr; int* quant_n = nullptr; size_t quant_cap = 0;   // P^2 state [9][E], [7][E]
    double* quant_blk = nullptr; size_t quant_blk_cap = 0;  // block means of the current sample, post_blk layout
    double* quant_out = nullptr; size_t quant_out_cap = 0;  // lower, median, upper of every level of the last run
    int quant_levels = 0; double quant_alpha = 0.0; long long quant_count = 0;   // what quant_out holds

    // per-run scratch kept across calls (a cudaMalloc / cudaFree per sbd_sapg_run costs up to 0.6 s: a free tears down
    // whatever the driver deferred, e.g. the graphs of the run)
    double* trace_d = nullptr; size_t trace_d_cap = 0;      // 13 double arrays + delta + err_psf, `trace_len` each
    int* trace_i = nullptr; size_t trace_i_cap = 0;
    int allstats_cap = 0;
    double *sal_aty = nullptr, *sal_u = nullptr, *sal_bu = nullptr, *sal_xt = nullptr;   // SALSA images
    cudaStream_t copy_stream = nullptr;                     // device -> host copy of the last samples, overlapped
    cudaEvent_t ev_langevin = nullptr;
    cudaStream_t prox_stream = nullptr;                     // the prox of an iteration runs here, next to the analysis
    cudaEvent_t ev_fork = nullptr, ev_reset = nullptr, ev_join = nullptr;
    int opt_overlap = -1;                                   // -1 automatic (on unless profiling), 0 off
    int opt_pdl = 1;                                        // programmatic dependent launch of the Chambolle kernels
    int opt_chamb_coop = -1;                                // cooperative single-launch prox (tv_coop.cuh): -1 auto (small problems), 0 never, 1 whenever it fits
    int cc_cap = 0;                                         // co-resident blocks of k_chamb_coop on this device
    unsigned int* cc_bar = nullptr;                         // its per-image barrier counters
    bool arm_ev_reset = false;

    // comm
    nccl_comm comm = nullptr;
    int nranks = 1, rank = 0;

    // profiling
    bool profile = false;
    double phase_ms[SBD_N_PHASES] = {0};
    long long phase_calls[SBD_N_PHASES] = {0};
    bool phase_main_only = true;
    std::vector<cudaEvent_t> ev;
    std::vector<int> ev_phase;
};

namespace {

const char* kPhaseNames[SBD_N_PHASES] = {"spectral_inverse", "langevin", "chambolle_sweeps", "chambolle_other",
                                         "tvnorm", "spectral_forward", "scalar_update", "allgather"};

template <typename T>
T* dalloc(size_t n) {
    T* p = nullptr;
    SBD_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
    return p;
}
template <typename T>
void dfree(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

void make_twiddles(int n, double2* d, cudaStream_t s) {
    std::vector<double2> h(n);
    for (int m = 0; m < n; ++m) {
        // exact octant symmetry keeps e.g. W^(n/4) = -i exactly
        const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)m / (long double)n;
        h[m].x = (double)cosl(a);
        h[m].y = (double)sinl(a);
    }
    if (n % 4 == 0) { h[n / 4] = make_double2(0.0, -1.0); h[n / 2] = make_double2(-1.0, 0.0); h[3 * n / 4] = make_double2(0.0, 1.0); }
    else if (n % 2 == 0) h[n / 2] = make_double2(-1.0, 0.0);
    SBD_CUDA(cudaMemcpyAsync(d, h.data(), sizeof(double2) * n, cudaMemcpyHostToDevice, s));
    SBD_CUDA(cudaStreamSynchronize(s));
}

void free_ws(sbd_ctx* c) {
    dfree(c->X); dfree(c->P); dfree(c->Gf); dfree(c->px0); dfree(c->py0); dfree(c->px1); dfree(c->py1);
    dfree(c->S1); dfree(c->S2);
    dfree(c->cc_bar); dfree(c->chst); dfree(c->cnt_tv); dfree(c->cnt_col); dfree(c->cnt_sq); dfree(c->stats);
    dfree(c->part_tv); dfree(c->part_ch); dfree(c->part_col); dfree(c->part_sq);
    c->ws_batch = 0;
}

// 3-D tensor map of a spectrum buffer as doubles {2*ny (q, re/im), nk (k), batch}; box = 2 complex x 256 bins
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
CUtensorMap make_spec_tmap(sbd_ctx* c, double2* base, int batch) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        SBD_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr));
        SBD_REQUIRE(fn && qr == cudaDriverEntryPointSuccess, SBD_E_CUDA, "cuTensorMapEncodeTiled not available in this driver");
        encode = (EncodeTiledFn)fn;
    }
    CUtensorMap tm;
    const cuuint64_t gdim[3] = {(cuuint64_t)2 * c->ny, (cuuint64_t)c->nk, (cuuint64_t)batch};
    const cuuint64_t gstr[2] = {(cuuint64_t)c->ny * 16, (cuuint64_t)c->spec_elems * 16};
    const cuuint32_t box[3] = {4, (cuuint32_t)TMA_KBOX, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    // SWIZZLE_32B: the shared-memory side of a box row (32 bytes) is stored with its halves exchanged in every other
    // group of four rows - the bank-conflict-free slab layout of fft2.cuh (slab())
    const CUresult r = encode(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw Error{SBD_E_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"};
    return tm;
}
const CUtensorMap& spec_tmap(sbd_ctx* c, const double2* buf) {
    if (buf == c->S1) return c->tm_S1;
    if (buf == c->S2) return c->tm_S2;
    if (buf == c->yhat) return c->tm_yhat;
    throw Error{SBD_E_INVALID, "rows pass: spectrum buffer without a tensor map"};
}

// choose launch geometry for a batch of `batch` images
void set_geometry(sbd_ctx* c, int batch_local) {
    const int batch = std::max(batch_local, c->geom_total);
    if (c->geom_batch == batch) return;
    const int nx = c->nx, ny = c->ny;
    c->tvV = (nx % 2 == 0 && nx >= 64) ? 2 : 1;
    const int strips = (nx + 32 * c->tvV - 1) / (32 * c->tvV);
    c->tv_gx = (strips + TV_WARPS - 1) / TV_WARPS;
    int seg = 64;
    while (seg > 8 && (long long)c->tv_gx * ((ny + seg - 1) / seg) * batch < 4 * 148) seg /= 2;
    if (c->opt_tv_seg > 0) seg = c->opt_tv_seg;
    c->tv_seg = seg;
    c->tv_gy = (ny + seg - 1) / seg;
    c->tv_parts = c->tv_gx * c->tv_gy;
    {   // fused multi-sweep Chambolle kernel (tv_multi.cuh): T levels, strips of 64 - 2*HL output pixels
        int T = 4;
        if (c->opt_chamb_T > 0) T = c->opt_chamb_T;
        if (nx % 2 != 0 || nx < 8) T = 1;           // pairs of pixels must be 16-byte aligned
        c->cmT = (T == 3 || T == 4) ? T : 1;
        const int HL = (c->cmT + 1) & ~1, WO = 64 - 2 * HL;
        c->cm_strips = (nx + WO - 1) / WO;
        c->cm_gx = (c->cm_strips + TV_WARPS - 1) / TV_WARPS;
        int sg = 128;
        // small problems are latency-bound (one warp per SM): shorter segments trade redundant halo rows for
        // parallelism (256^2, one chain: 4-row segments are 10 % faster than 8-row ones)
        // (tools/seg_sweep.py, 8 chains: 1024^2 - 32 rows 6340, 64 rows 7170, 128 rows 7100 chain-steps/s; 2048^2 x 2 -
        // 32 rows 1755, 64 rows 1840, 128 rows 1725: four blocks per SM are enough, halo rows cost more than the tail)
        while (sg > 8 && (long long)c->cm_gx * ((ny + sg - 1) / sg) * batch < 4 * 148) sg /= 2;
        if (sg == 8 && (long long)c->cm_gx * ((ny + 7) / 8) * batch < 2 * 148) sg = 4;      // less than two blocks per SM
        // very large batches (64 chains at 4096^2): longer segments cut the share of the vertical halo rows; only while
        // the grid still has >= 20 waves of 3 blocks per SM, so that the tail wave stays negligible (4096^2 x 64 chains:
        // 80.9 -> 78.2 ms per prox step from 128 to 512 rows)
        while (sg >= 128 && sg < 512 && (long long)c->cm_gx * ((ny + 2 * sg - 1) / (2 * sg)) * batch >= 20LL * 3 * 148) sg *= 2;
        if (c->opt_chamb_seg > 0) sg = c->opt_chamb_seg;
        if (c->opt_chamb_emit >= 0) c->cm_emit = c->opt_chamb_emit != 0;
        if (c->opt_chamb_plan33 >= 0) c->cm_plan33 = c->opt_chamb_plan33 != 0;
        c->cm_seg = sg;
        c->cm_gy = (ny + sg - 1) / sg;
    }
    if (c->pow2) {
        // rows pass: LP line pairs per block, shared memory <= ~74 KB so that 3 blocks fit an SM
        const size_t le_x = (size_t)nx + nx / (nx >= 1024 || nx == 256 || nx == 128 ? 16 : (nx == 16 ? 4 : 8));
        int LP = 1;
        while (2 * LP <= ny / 2 && (size_t)(2 * LP) * le_x * 16 <= 74 * 1024 && 2 * LP * nx <= 4096) LP *= 2;
        while (LP > 1 && (long long)(ny / 2 / LP) * batch < 2 * 148) LP /= 2;
        c->rowsLP = LP;
        c->rowsT = std::max(32, LP * nx / 16);
        c->rows_smem = (size_t)LP * le_x * 16;
        c->colsT = std::max(32, c->colsKC * ny / 16);
    }
    c->geom_batch = batch;
}

void ensure_ws(sbd_ctx* c, int batch) {
    if (batch <= c->ws_batch) { set_geometry(c, batch); return; }
    free_ws(c);
    const size_t n = (size_t)batch * c->npix;
    c->X = dalloc<double>(n); c->P = dalloc<double>(n); c->Gf = dalloc<double>(n);
    c->px0 = dalloc<double>(n); c->py0 = dalloc<double>(n); c->px1 = dalloc<double>(n); c->py1 = dalloc<double>(n);
    if (c->pow2 || c->smooth) {
        c->S1 = dalloc<double2>((size_t)batch * c->spec_elems);
        c->S2 = dalloc<double2>((size_t)batch * c->spec_elems);
        if (c->v2) { c->tm_S1 = make_spec_tmap(c, c->S1, batch); c->tm_S2 = make_spec_tmap(c, c->S2, batch); }
    }
    c->chst = dalloc<ChambState>(batch);
    c->cc_bar = dalloc<unsigned int>(batch);
    SBD_CUDA(cudaMemsetAsync(c->cc_bar, 0, sizeof(unsigned int) * batch, c->stream));
    c->cnt_tv = dalloc<unsigned int>(batch); c->cnt_col = dalloc<unsigned int>(batch); c->cnt_sq = dalloc<unsigned int>(batch);
    c->stats = dalloc<double>((size_t)batch * NSTAT);
    SBD_CUDA(cudaMemsetAsync(c->cnt_tv, 0, sizeof(unsigned int) * batch, c->stream));
    SBD_CUDA(cudaMemsetAsync(c->cnt_col, 0, sizeof(unsigned int) * batch, c->stream));
    SBD_CUDA(cudaMemsetAsync(c->cnt_sq, 0, sizeof(unsigned int) * batch, c->stream));
    SBD_CUDA(cudaMemsetAsync(c->stats, 0, sizeof(double) * batch * NSTAT, c->stream));
    SBD_CUDA(cudaMemsetAsync(c->chst, 0, sizeof(ChambState) * batch, c->stream));
    // partial buffers sized for the finest geometry (seg = 1 worst case is never used; seg >= 1)
    c->geom_batch = -1;
    set_geometry(c, batch);
    const int strips = (c->nx + 31) / 32;
    const size_t maxparts = (size_t)((strips + TV_WARPS - 1) / TV_WARPS) * c->ny;    // seg = 1 bound
    c->part_tv = dalloc<double>((size_t)batch * maxparts);
    c->part_ch = dalloc<double>((size_t)batch * maxparts * 5);     // up to T = 5 levels per launch
    c->part_col = dalloc<double>((size_t)batch * (c->nk + 8) * 4);
    c->part_sq = dalloc<double>((size_t)batch * 1024);
    c->ws_batch = batch;
}

// launches issued inside the scope go to another stream of the context
struct StreamScope {
    sbd_ctx* c; cudaStream_t old;
    StreamScope(sbd_ctx* c_, cudaStream_t s) : c(c_), old(c_->stream) { c->stream = s; }
    ~StreamScope() { c->stream = old; }
};

// Phase timing without perturbing the run: event pairs are only RECORDED while
// the iteration is being enqueued and resolved after the run has finished.
struct PhaseTimer {
    sbd_ctx* c; int phase; cudaEvent_t a = nullptr, b = nullptr;
    PhaseTimer(sbd_ctx* c_, int p) : c(c_), phase(p) {
        if (!c->profile) return;
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, c->stream);
    }
    ~PhaseTimer() {
        if (!c->profile) return;
        cudaEventRecord(b, c->stream);
        c->ev.push_back(a); c->ev.push_back(b); c->ev_phase.push_back(phase);
    }
};

void resolve_phase_events(sbd_ctx* c) {
    for (size_t i = 0; i < c->ev_phase.size(); ++i) {
        float ms = 0.f;
        cudaEventSynchronize(c->ev[2 * i + 1]);
        cudaEventElapsedTime(&ms, c->ev[2 * i], c->ev[2 * i + 1]);
        c->phase_ms[c->ev_phase[i]] += ms;
        c->phase_calls[c->ev_phase[i]] += 1;
        cudaEventDestroy(c->ev[2 * i]); cudaEventDestroy(c->ev[2 * i + 1]);
    }
    c->ev.clear(); c->ev_phase.clear();
}

// ---- launch helpers --------------------------------------------------------
#define LAUNCH_CHECK(c) do { (c)->launches++; SBD_CUDA(cudaGetLastError()); } while (0)

void tvnorm(sbd_ctx* c, const double* x, double* out, int out_stride, int batch) {
    dim3 g(c->tv_gx, c->tv_gy, batch);
    if (c->tvV == 2)
        k_tvnorm<2><<<g, TV_THREADS, 0, c->stream>>>(x, c->nx, c->ny, c->tv_seg, c->npix, c->part_tv, c->cnt_tv, out, out_stride);
    else
        k_tvnorm<1><<<g, TV_THREADS, 0, c->stream>>>(x, c->nx, c->ny, c->tv_seg, c->npix, c->part_tv, c->cnt_tv, out, out_stride);
    LAUNCH_CHECK(c);
}

// prox with the options stored in ctl (prox_lambda_theta, tau, tol, maxiter).
// `maxiter` is the host copy used to size the launch sequence.  The dual pair
// starts from px0/py0 (caller zeroes or fills them).
void zero_duals(sbd_ctx* c, int batch) {
    SBD_CUDA(cudaMemsetAsync(c->px0, 0, sizeof(double) * batch * c->npix, c->stream));
    SBD_CUDA(cudaMemsetAsync(c->py0, 0, sizeof(double) * batch * c->npix, c->stream));
}

template <int T, bool PIPE, int MINB, int EMIT = 0, bool ERRSUB = false>
void chamb_multi_launch(sbd_ctx* c, const double* g, const double* pxi, const double* pyi, double* pxo,
                        double* pyo, int batch, int redo, int zero_in, double* f = nullptr) {
    // strip geometry depends on the number of fused levels (lateral halo HL)
    constexpr int HL = (T + 1) & ~1, WO = 64 - 2 * HL;
    const int strips = (c->nx + WO - 1) / WO;
    dim3 grid((strips + TV_WARPS - 1) / TV_WARPS, c->cm_gy, batch);
    // programmatic stream serialization: the launch is staged while the previous kernel of the stream still runs and
    // starts the moment that one has completed (the kernel waits with griddepcontrol.wait before reading anything)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(TV_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = c->opt_pdl ? 1 : 0;
    const int nx = c->nx, ny = c->ny, seg = c->cm_seg;
    const size_t npix = c->npix;
    const Control* ctl = c->ctl;
    if (zero_in)
        SBD_CUDA(cudaLaunchKernelEx(&cfg, k_chamb_multi<T, PIPE, MINB, true, EMIT, ERRSUB>, g, pxi, pyi, pxo, pyo, nx, ny, seg, strips, npix,
                                    ctl, c->chst, c->part_ch, redo, f));
    else
        SBD_CUDA(cudaLaunchKernelEx(&cfg, k_chamb_multi<T, PIPE, MINB, false, EMIT, ERRSUB>, g, pxi, pyi, pxo, pyo, nx, ny, seg, strips, npix,
                                    ctl, c->chst, c->part_ch, redo, f));
}

// Does the prox of `batch` images run as the cooperative single-launch kernel, and with which partition?  The partition
// (blocks per image, units per warp) fixes the order of the err_k partial sums, so like the rest of the launch geometry it
// is a function of the TOTAL chain count, not of the chains on this rank.
bool coop_plan(sbd_ctx* c, int batch, int& bpi, int& upw) {
    if (c->opt_chamb_coop == 0 || c->nx % 2 != 0 || c->nx < 2 || c->ny < 2) return false;
    const int total = std::max(batch, c->geom_total);
    const long long units = (long long)c->ny * ((c->nx + 63) / 64);
    if (c->opt_chamb_coop < 0) {
        // automatic: small problems only (measured with tools/coop_crossover.py: ahead up to 2^21 pixels x chains - 1.7x at
        // 256^2 x 1, 1.55x at 512^2 x 8, 1.1x at 1024^2 x 2 - behind from 2^22), and never when an option addresses the
        // fused kernel explicitly
        if ((long long)c->npix * total > (1LL << 21)) return false;
        if (c->opt_chamb_seg > 0 || c->opt_chamb_T > 0 || c->opt_chamb_errsub >= 0 || c->opt_chamb_emit >= 0 || c->opt_chamb_plan33 >= 0) return false;
    }
    if (!c->cc_cap) {
        int per_sm = 0;
        SBD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_chamb_coop, CC_THREADS, 0));
        c->cc_cap = std::max(1, per_sm) * c->sm_count;
    }
    for (upw = 1; upw <= 256; upw *= 2) {
        bpi = (int)((units + (long long)CC_WARPS * upw - 1) / ((long long)CC_WARPS * upw));
        if ((long long)bpi * total <= c->cc_cap) return true;
    }
    return false;
}

// zero_start: the dual pair starts from zero (px0/py0 are then neither read nor need to be cleared
// when the fused kernel runs; the single-sweep path clears them itself)
// want_err == false: the caller never reads the VALUE of err_k (only the sweep count), which allows the sampled stop
// test of tv_multi.cuh (ERRSUB) on large problems: same k, same p, same f, 12 % fewer fp64 instructions per sweep
// trace/ntrace: where the sweep count of chain 0 is recorded at the end of a main-loop prox (k_chamb_record); the
// cooperative kernel does that itself, every other path leaves it to the caller - returns true when it was recorded
bool chambolle(sbd_ctx* c, const double* g, double* f, int batch, int maxiter, bool zero_start, bool keep_duals = true,
               bool want_err = true, int* trace = nullptr, int ntrace = 0) {
    SBD_REQUIRE(maxiter >= 1, SBD_E_INVALID, "chambolle: maxiter must be >= 1");       // the block plan below relies on it
    k_chamb_reset<<<(batch + 127) / 128, 128, 0, c->stream>>>(c->chst, batch, c->ctl, c->cc_bar);
    LAUNCH_CHECK(c);
    if (c->arm_ev_reset) SBD_CUDA(cudaEventRecord(c->ev_reset, c->stream));     // the lambda*theta snapshot is taken
    {
        int bpi = 0, upw = 0;
        if (coop_plan(c, batch, bpi, upw)) {
            // small problem: all sweeps, the stop test and f = g - lambda div p in ONE cooperative launch (tv_coop.cuh)
            PhaseTimer pt2(c, 2);
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(batch * bpi)); cfg.blockDim = dim3(CC_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = c->stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeCooperative;
            attr[0].val.cooperative = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            const int nx = c->nx, ny = c->ny, zs = zero_start ? 1 : 0;
            const size_t npix = c->npix;
            const Control* ctl = c->ctl;
            SBD_CUDA(cudaLaunchKernelEx(&cfg, k_chamb_coop, g, c->px0, c->py0, c->px1, c->py1, f, nx, ny, npix, bpi, upw, zs, maxiter,
                                        ctl, c->chst, c->part_ch, c->cc_bar, c->ctl, trace, ntrace));
            LAUNCH_CHECK(c);
            return trace != nullptr;
        }
    }
    dim3 grid(c->tv_gx, c->tv_gy, batch);
    PhaseTimer* pt = new PhaseTimer(c, 2);
    if (c->cmT > 1) {
        // blocks of fused sweeps; each block = main launch + redo launch (a no-op unless the reference's
        // stop test fired inside the block).  4-level blocks are the most efficient; the block planned
        // last is an odd one (3 or 1 levels), because odd blocks have a pixel of lateral validity to
        // spare and can write the prox output themselves (EMIT, tv_multi.cuh).  K = 4k+1 runs as 4 x(k-2), 3 x3
        // rather than 4 x k, 1: the one-level tail is a full memory pass for a single sweep (K = 25: 10.12 vs
        // 10.22 ms per prox of 8 chains at 4096^2; SBD_CHAMB_PLAN33=0 restores the other plan).
        std::vector<int> plan;
        if (c->cmT == 4) {
            const int a = maxiter / 4, r = maxiter % 4;
            if (r == 1 && a >= 2 && c->cm_plan33) { plan.assign(a - 2, 4); plan.insert(plan.end(), 3, 3); }   // 4k+1 = 4(k-2) + 3*3
            else if (r == 1 || r == 3) { plan.assign(a, 4); plan.push_back(r); }
            else if (r == 2) { if (a > 0) { plan.assign(a - 1, 4); plan.push_back(3); plan.push_back(3); } else plan.push_back(3); }
            else { plan.assign(a - 1, 4); plan.push_back(3); plan.push_back(1); }      // maxiter >= 4 here
        } else {
            for (int k = 0; k < maxiter; k += c->cmT) plan.push_back(std::min(c->cmT, maxiter - k));
            if (plan.back() % 2 == 0 && plan.back() > 1) { plan.back() -= 1; plan.push_back(1); }
        }
        // sampled stop test: only where the exact fallback launch (one more no-op per block) is noise, i.e. large grids
        const bool errsub = !want_err && c->opt_chamb_errsub != 0 &&
                            (c->opt_chamb_errsub > 0 || (long long)c->npix * std::max(batch, c->geom_total) >= (1LL << 22));
        for (size_t b = 0; b < plan.size(); ++b) {
            const int T = plan[b];
            if (pt && T != 4) { delete pt; pt = nullptr; }      // phase 2 = the 4-level launches only
            const double* pxi = (b & 1) ? c->px1 : c->px0;
            const double* pyi = (b & 1) ? c->py1 : c->py0;
            double* pxo = (b & 1) ? c->px0 : c->px1;
            double* pyo = (b & 1) ? c->py0 : c->py1;
            const int zin = (zero_start && b == 0) ? 1 : 0;
            const bool last = b + 1 == plan.size();
            const int emit = (last && c->cm_emit && (T & 1)) ? (keep_duals ? 1 : 2) : 0;
            // launches of a block: main [, exact: behind a sampled main launch] [, redo: a one-level block cannot stop
            // "inside"].  The sampled variants exist for the blocks of the SAPG prox: (4, EMIT 0), (3, EMIT 0), (3, EMIT 2).
            const bool sub = errsub && (T == 4 || (T == 3 && emit != 1));
            const int seq[3] = {0, sub ? 2 : -1, T > 1 ? 1 : -1};
            for (int q = 0; q < 3; ++q) {
                const int redo = seq[q];
                if (redo < 0) continue;
                const int em = (redo == 1) ? 0 : emit;
                const bool sm = sub && redo == 0;
#define SBD_CM(T_, MINB_) \
                if (em == 1) chamb_multi_launch<T_, false, MINB_, 1>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin, f); \
                else if (em == 2) chamb_multi_launch<T_, false, MINB_, 2>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin, f); \
                else chamb_multi_launch<T_, false, MINB_, 0>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin);
                if (T == 1) { SBD_CM(1, 4) }
                else if (T == 3) {
                    if (sm && em == 2) chamb_multi_launch<3, false, 3, 2, true>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin, f);
                    else if (sm) chamb_multi_launch<3, false, 3, 0, true>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin);
                    else { SBD_CM(3, 3) }
                }
                else if (sm) chamb_multi_launch<4, false, 3, 0, true>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin);
                else chamb_multi_launch<4, false, 3, 0>(c, g, pxi, pyi, pxo, pyo, batch, redo, zin);
#undef SBD_CM
                LAUNCH_CHECK(c);
            }
        }
    } else {
        if (zero_start) zero_duals(c, batch);
        for (int s = 0; s < maxiter; ++s) {
            const double* pxi = (s & 1) ? c->px1 : c->px0;
            const double* pyi = (s & 1) ? c->py1 : c->py0;
            double* pxo = (s & 1) ? c->px0 : c->px1;
            double* pyo = (s & 1) ? c->py0 : c->py1;
            if (c->tvV == 2)
                k_chamb_sweep<2><<<grid, TV_THREADS, 0, c->stream>>>(g, pxi, pyi, pxo, pyo, c->nx, c->ny, c->tv_seg, c->npix, c->ctl, c->chst, c->part_ch);
            else
                k_chamb_sweep<1><<<grid, TV_THREADS, 0, c->stream>>>(g, pxi, pyi, pxo, pyo, c->nx, c->ny, c->tv_seg, c->npix, c->ctl, c->chst, c->part_ch);
            LAUNCH_CHECK(c);
        }
    }
    if (pt) delete pt;
    if (c->tvV == 2)
        k_chamb_out<2><<<grid, TV_THREADS, 0, c->stream>>>(g, c->px0, c->py0, c->px1, c->py1, f, c->nx, c->ny, c->tv_seg, c->npix, c->ctl, c->chst);
    else
        k_chamb_out<1><<<grid, TV_THREADS, 0, c->stream>>>(g, c->px0, c->py0, c->px1, c->py1, f, c->nx, c->ny, c->tv_seg, c->npix, c->ctl, c->chst);
    LAUNCH_CHECK(c);
    return false;
}

template <typename K>
void set_smem(sbd_ctx* c, K kernel, size_t bytes) {
    // opt in to > 48 KB of dynamic shared memory, once per (context = device, kernel, size)
    std::map<const void*, size_t>& done = c->smem_optin;
    const void* key = reinterpret_cast<const void*>(kernel);
    auto it = done.find(key);
    if (it != done.end() && it->second >= bytes) return;
    if (bytes > 48 * 1024)
        SBD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done[key] = bytes;
}

// blocks of `kernel` resident on the whole device = the L2 prefetch distance of the FFT passes
template <typename K>
int resident_blocks(sbd_ctx* c, K kernel, int threads, size_t smem) {
    std::map<std::pair<const void*, size_t>, int>& cache = c->resident_cache;
    const auto key = std::make_pair(reinterpret_cast<const void*>(kernel), smem * 4096 + (size_t)threads);
    auto it = cache.find(key);
    if (it != cache.end()) return c->fft_pf ? it->second : 0;
    int per_sm = 1;
    SBD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    cache[key] = std::max(1, per_sm) * c->sm_count;
    return c->fft_pf ? cache[key] : 0;
}

#define SBD_FFT_SIZES(X) X(16) X(32) X(64) X(128) X(256) X(512) X(1024) X(2048) X(4096)

SpecGeom spec_geom(const sbd_ctx* c) {
    SpecGeom g;
    g.C = c->colsC; g.logC = c->colsLogC; g.ny = c->ny;
    return g;
}

#define SBD_FFT2_SIZES(X) X(1024) X(2048) X(4096)

// The mixed-radix kernels serve every size with one instantiation, and the dynamic shared-memory limit is a property of
// the kernel on the device, not of a context: each opts in once to the largest line any size needs (ANY_MAXN double2),
// so that no context can lower the limit under another one that uses a longer line.
constexpr size_t ANY_SMEM_OPTIN = (size_t)ANY_MAXN * sizeof(double2);

void rows_fwd(sbd_ctx* c, const double* x, double2* spec, int batch) {
    if (c->smooth) {
        const size_t smem = (size_t)c->nx * 16;
        set_smem(c, k_rows_any_fwd, ANY_SMEM_OPTIN);
        k_rows_any_fwd<<<dim3((c->ny + 1) / 2, batch), c->plan_x.T, smem, c->stream>>>(x, spec, c->plan_x, c->ny, c->npix,
                                                                                       c->spec_elems, c->tw_nx);
        LAUNCH_CHECK(c);
        return;
    }
    if (c->v2) {
        const size_t smem2 = (size_t)c->nx * 16;
        dim3 g2(c->ny / 2, batch);
        const CUtensorMap& tm = spec_tmap(c, spec);
        switch (c->nx) {
#define X(N) case N: set_smem(c, k_rows2_fwd<N>, smem2); \
            k_rows2_fwd<N><<<g2, N / 16, smem2, c->stream>>>(x, spec, tm, c->ny, c->npix, c->spec_elems, c->tw_nx); break;
            SBD_FFT2_SIZES(X)
#undef X
            default: throw Error{SBD_E_UNSUPPORTED, "rows_fwd (v2): unsupported size"};
        }
        LAUNCH_CHECK(c);
        return;
    }
    const size_t smem = c->rows_smem;
    dim3 g(c->ny / 2 / c->rowsLP, batch);
    const SpecGeom sg = spec_geom(c);
    switch (c->nx) {
#define X(N) case N: set_smem(c, k_rows_fwd<N>, smem); \
        k_rows_fwd<N><<<g, c->rowsT, smem, c->stream>>>(x, spec, sg, c->rowsLP, c->npix, c->spec_elems, c->tw_nx, \
                                                        resident_blocks(c, k_rows_fwd<N>, c->rowsT, smem)); break;
        SBD_FFT_SIZES(X)
#undef X
        default: throw Error{SBD_E_UNSUPPORTED, "rows_fwd: unsupported size"};
    }
    LAUNCH_CHECK(c);
}

void rows_inv(sbd_ctx* c, const double2* spec, double* out, int batch) {
    if (c->smooth) {
        const size_t smem = (size_t)c->nx * 16;
        set_smem(c, k_rows_any_inv, ANY_SMEM_OPTIN);
        k_rows_any_inv<<<dim3((c->ny + 1) / 2, batch), c->plan_x.T, smem, c->stream>>>(spec, out, c->plan_x, c->ny, c->npix,
                                                                                       c->spec_elems, c->tw_nx);
        LAUNCH_CHECK(c);
        return;
    }
    if (c->v2) {
        const size_t smem2 = (size_t)c->nx * 16;
        dim3 g2(c->ny / 2, batch);
        const CUtensorMap& tm = spec_tmap(c, spec);
        switch (c->nx) {
#define X(N) case N: set_smem(c, k_rows2_inv<N>, smem2); \
            k_rows2_inv<N><<<g2, N / 16, smem2, c->stream>>>(spec, out, tm, c->ny, c->npix, c->spec_elems, c->tw_nx); break;
            SBD_FFT2_SIZES(X)
#undef X
            default: throw Error{SBD_E_UNSUPPORTED, "rows_inv (v2): unsupported size"};
        }
        LAUNCH_CHECK(c);
        return;
    }
    const size_t smem = c->rows_smem;
    dim3 g(c->ny / 2 / c->rowsLP, batch);
    const SpecGeom sg = spec_geom(c);
    switch (c->nx) {
#define X(N) case N: set_smem(c, k_rows_inv<N>, smem); \
        k_rows_inv<N><<<g, c->rowsT, smem, c->stream>>>(spec, out, sg, c->rowsLP, c->npix, c->spec_elems, c->tw_nx); break;
        SBD_FFT_SIZES(X)
#undef X
        default: throw Error{SBD_E_UNSUPPORTED, "rows_inv: unsupported size"};
    }
    LAUNCH_CHECK(c);
}

template <int MODE>
void cols(sbd_ctx* c, const double2* in, double2* out, int batch, int opsel = 0) {
    ColArgs a;
    a.in = in; a.out = out; a.yhat = c->yhat; a.coef = c->coef; a.tw = c->tw_ny; a.tw_x = c->tw_nx; a.ctl = c->ctl;
    a.partials = c->part_col; a.counters = c->cnt_col; a.stats = c->stats;
    a.spec_stride = c->spec_elems; a.nk = c->nk; a.nxfull = c->nx; a.t = c->t;
    a.npsi = (c->model == SBD_LAPLACE) ? 1 : 2; a.C = c->colsKC; a.logC = c->colsLogKC; a.LC = c->colsC;
    a.nsub = c->colsC / c->colsKC; a.ntiles = c->ntiles; a.opsel = opsel;
    a.opscale = 1.0 / ((double)c->nx * (double)c->ny);
    a.mu = c->salsa_mu;
    if (c->smooth) {
        const size_t smem = (size_t)c->ny * 16;
        set_smem(c, k_cols_any<MODE>, ANY_SMEM_OPTIN);
        k_cols_any<MODE><<<dim3(batch, c->nk), c->plan_y.T, smem, c->stream>>>(a, c->plan_y);
        LAUNCH_CHECK(c);
        return;
    }
    if (c->v2) {
        const size_t smem2 = (size_t)c->ny * 16;
        dim3 g2(batch, c->nk);
        a.pf = 0;
        switch (c->ny) {
#define X(N) case N: set_smem(c, k_cols2<N, MODE>, smem2); k_cols2<N, MODE><<<g2, N / 16, smem2, c->stream>>>(a); break;
            SBD_FFT2_SIZES(X)
#undef X
            default: throw Error{SBD_E_UNSUPPORTED, "cols (v2): unsupported size"};
        }
        LAUNCH_CHECK(c);
        return;
    }
    const size_t smem = c->cols_smem;
    dim3 g(batch, c->ntiles * (c->colsC / c->colsKC));
    switch (c->ny) {
#define X(N) case N: \
        if (c->t == 7) { set_smem(c, k_cols<N, MODE, true>, smem); a.pf = resident_blocks(c, k_cols<N, MODE, true>, c->colsT, smem); \
                         k_cols<N, MODE, true><<<g, c->colsT, smem, c->stream>>>(a); } \
        else { set_smem(c, k_cols<N, MODE, false>, smem); a.pf = resident_blocks(c, k_cols<N, MODE, false>, c->colsT, smem); \
               k_cols<N, MODE, false><<<g, c->colsT, smem, c->stream>>>(a); } \
        break;
        SBD_FFT_SIZES(X)
#undef X
        default: throw Error{SBD_E_UNSUPPORTED, "cols: unsupported size"};
    }
    LAUNCH_CHECK(c);
}

// PSF taps (from ctl->psi or an override on device) + column coefficients for nkc bins
void psf_refresh_coef(sbd_ctx* c, int nkc) {
    const int total = 3 * nkc * c->t;
    k_psf_colcoef<<<(total + 127) / 128, 128, 0, c->stream>>>(c->t, c->nx, nkc, c->taps, c->tw_nx, c->coef);
    LAUNCH_CHECK(c);
}
void psf_from_host(sbd_ctx* c, const double psi[2], int nkc) {
    SBD_CUDA(cudaMemcpyAsync(c->psi_dev, psi, 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    k_psf_taps<<<1, 256, 0, c->stream>>>(c->model, c->t, c->phi, c->ctl, c->psi_dev, c->taps);
    LAUNCH_CHECK(c);
    if (nkc > 0) psf_refresh_coef(c, nkc);
}

void require_fft(sbd_ctx* c) {
    SBD_REQUIRE(c->pow2 || c->smooth, SBD_E_UNSUPPORTED, c->fft_err);
}

// elements of one image at block size 2^level: ceil(rows / s) x ceil(cols / s)
size_t post_blocks(const sbd_ctx* c, int level) {
    const int s = 1 << level;
    return (size_t)((c->nx + s - 1) / s) * (size_t)((c->ny + s - 1) / s);
}

int fail(sbd_ctx* c, const Error& e) {
    if (c) c->err = e.msg; else g_create_error = e.msg;
    return e.code;
}

}  // namespace

#define SBD_TRY(ctx) try {
#define SBD_CATCH(ctx)                                                     \
    } catch (const Error& e) { return fail((ctx), e); }                    \
      catch (const std::exception& e) { return fail((ctx), Error{SBD_E_INVALID, e.what()}); } \
    return SBD_OK;

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int sbd_version(void) { return SBD_VERSION; }

const char* sbd_last_error(const sbd_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

long long sbd_launch_count(const sbd_ctx* ctx) { return ctx ? ctx->launches : 0; }

const char* sbd_phase_name(int i) { return (i >= 0 && i < SBD_N_PHASES) ? kPhaseNames[i] : ""; }

int sbd_phase_times(const sbd_ctx* ctx, double ms[SBD_N_PHASES], long long calls[SBD_N_PHASES]) {
    if (!ctx || !ms) return SBD_E_INVALID;
    for (int i = 0; i < SBD_N_PHASES; ++i) {
        ms[i] = ctx->phase_ms[i];
        if (calls) calls[i] = ctx->phase_calls[i];
    }
    return SBD_OK;
}

int sbd_set_profile(sbd_ctx* ctx, int on) {
    if (!ctx) return SBD_E_INVALID;
    ctx->profile = on != 0;
    return SBD_OK;
}

int sbd_set_posterior(sbd_ctx* c, int levels) {
    if (!c) return SBD_E_INVALID;
    if (levels < 0 || levels > POST_MAXL) {
        c->err = "sbd_set_posterior: levels must be in 0..7 (block sizes 1 .. 2^(levels-1))";
        return SBD_E_INVALID;
    }
    c->post_levels = levels;
    return SBD_OK;
}

int sbd_posterior_stats(const sbd_ctx* ctx, int level, double* mean, double* within, double* between, int* n,
                        int* chains) {
    if (!ctx) return SBD_E_INVALID;
    sbd_ctx* c = const_cast<sbd_ctx*>(ctx);     // only the error text and the stream are touched
    SBD_TRY(c)
    SBD_REQUIRE(c->stat_levels > 0, SBD_E_INVALID,
                "sbd_posterior_stats: the last SAPG run on this context accumulated no statistics (sbd_set_posterior)");
    SBD_REQUIRE(level >= 0 && level < c->stat_levels, SBD_E_INVALID,
                "sbd_posterior_stats: level " + std::to_string(level) + " outside 0.." + std::to_string(c->stat_levels - 1) +
                " of the last run");
    SBD_CUDA(cudaSetDevice(c->device));
    size_t off = 0;
    for (int j = 0; j < level; ++j) off += 3 * post_blocks(c, j);
    const size_t nb = post_blocks(c, level);
    double* dst[3] = {mean, within, between};
    for (int q = 0; q < 3; ++q)
        if (dst[q]) SBD_CUDA(cudaMemcpyAsync(dst[q], c->post_out + off + q * nb, nb * sizeof(double), cudaMemcpyDeviceToHost,
                                             c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    if (n) *n = c->stat_n;
    if (chains) *chains = c->stat_chains;
    SBD_CATCH(c)
}

int sbd_set_posterior_diagnostics(sbd_ctx* c, int batch_len) {
    if (!c) return SBD_E_INVALID;
    if (batch_len < -1) {
        c->err = "sbd_set_posterior_diagnostics: batch_len must be 0 (off), -1 (floor(sqrt(n))) or a length >= 1";
        return SBD_E_INVALID;
    }
    c->post_diag = batch_len;
    return SBD_OK;
}

int sbd_posterior_diagnostics(const sbd_ctx* ctx, int level, double* batch_mean, double* batch_within,
                              double* batch_between, double* half_mean, double* half_within, double* half_between,
                              int* batch_len, int* n_batches, int* half_n) {
    if (!ctx) return SBD_E_INVALID;
    sbd_ctx* c = const_cast<sbd_ctx*>(ctx);     // only the error text and the stream are touched
    SBD_TRY(c)
    SBD_REQUIRE(c->diag_levels > 0, SBD_E_INVALID,
                "sbd_posterior_diagnostics: the last SAPG run on this context accumulated no diagnostics "
                "(sbd_set_posterior_diagnostics)");
    SBD_REQUIRE(level >= 0 && level < c->diag_levels, SBD_E_INVALID,
                "sbd_posterior_diagnostics: level " + std::to_string(level) + " outside 0.." +
                std::to_string(c->diag_levels - 1) + " of the last run");
    SBD_CUDA(cudaSetDevice(c->device));
    size_t off = 0;
    for (int j = 0; j < level; ++j) off += 6 * post_blocks(c, j);
    const size_t nb = post_blocks(c, level);
    double* dst[6] = {batch_mean, batch_within, batch_between, half_mean, half_within, half_between};
    for (int q = 0; q < 6; ++q)
        if (dst[q]) SBD_CUDA(cudaMemcpyAsync(dst[q], c->diag_out + off + q * nb, nb * sizeof(double),
                                             cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    if (batch_len) *batch_len = c->diag_b;
    if (n_batches) *n_batches = c->diag_nbatch;
    if (half_n) *half_n = c->diag_h;
    SBD_CATCH(c)
}

int sbd_set_posterior_quantiles(sbd_ctx* c, double alpha) {
    if (!c) return SBD_E_INVALID;
    if (!(alpha >= 0.0 && alpha < 1.0)) {
        c->err = "sbd_set_posterior_quantiles: alpha must be 0 (off) or a credible level in (0, 1)";
        return SBD_E_INVALID;
    }
    c->post_ci = alpha;
    return SBD_OK;
}

int sbd_posterior_quantiles(const sbd_ctx* ctx, int level, double* lower, double* median, double* upper,
                            double* alpha, long long* count) {
    if (!ctx) return SBD_E_INVALID;
    sbd_ctx* c = const_cast<sbd_ctx*>(ctx);     // only the error text and the stream are touched
    SBD_TRY(c)
    SBD_REQUIRE(c->quant_levels > 0, SBD_E_INVALID,
                "sbd_posterior_quantiles: the last SAPG run on this context accumulated no quantiles "
                "(sbd_set_posterior_quantiles)");
    SBD_REQUIRE(level >= 0 && level < c->quant_levels, SBD_E_INVALID,
                "sbd_posterior_quantiles: level " + std::to_string(level) + " outside 0.." +
                std::to_string(c->quant_levels - 1) + " of the last run");
    SBD_CUDA(cudaSetDevice(c->device));
    size_t off = 0;
    for (int j = 0; j < level; ++j) off += 3 * post_blocks(c, j);
    const size_t nb = post_blocks(c, level);
    double* dst[3] = {lower, median, upper};
    for (int q = 0; q < 3; ++q)
        if (dst[q]) SBD_CUDA(cudaMemcpyAsync(dst[q], c->quant_out + off + q * nb, nb * sizeof(double),
                                             cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    if (alpha) *alpha = c->quant_alpha;
    if (count) *count = c->quant_count;
    SBD_CATCH(c)
}

int sbd_set_option(sbd_ctx* c, const char* name, int value) {
    if (!c || !name) return SBD_E_INVALID;
    const std::string n(name);
    if (n == "chamb_seg") c->opt_chamb_seg = value;
    else if (n == "chamb_levels") c->opt_chamb_T = value;
    else if (n == "tv_seg") c->opt_tv_seg = value;
    else if (n == "chamb_emit") c->opt_chamb_emit = value;
    else if (n == "chamb_plan33") c->opt_chamb_plan33 = value;
    else if (n == "chamb_errsub") c->opt_chamb_errsub = value;
    else if (n == "overlap") c->opt_overlap = value;
    else if (n == "pdl") c->opt_pdl = value != 0;
    else if (n == "chamb_coop") c->opt_chamb_coop = value;
    else if (n == "geom_chains") c->geom_total = std::max(value, 0);
    else { c->err = "sbd_set_option: unknown option '" + n + "'"; return SBD_E_INVALID; }
    c->geom_batch = -1;             // recomputed by the next call
    return SBD_OK;
}

int sbd_get_geometry(sbd_ctx* c, int batch, int out[SBD_N_GEOM]) {
    if (!c || !out || batch < 1) return SBD_E_INVALID;
    set_geometry(c, batch);
    out[0] = c->cmT; out[1] = c->cm_seg; out[2] = c->cm_gx; out[3] = c->cm_gy;
    out[4] = c->tv_seg; out[5] = c->tv_gx; out[6] = c->tv_gy; out[7] = c->rowsLP;
    try {
        int bpi = 0, upw = 0;
        const bool coop = coop_plan(c, batch, bpi, upw);
        out[8] = coop ? bpi : 0; out[9] = coop ? upw : 0;
    } catch (const Error& e) { c->err = e.msg; return e.code; }
    return SBD_OK;
}

int sbd_create(sbd_ctx** out, int rows, int cols, int psf_size, int model, double phi,
               int max_batch, int device) {
    sbd_ctx* c = nullptr;
    try {
        SBD_REQUIRE(out, SBD_E_INVALID, "sbd_create: out is NULL");
        *out = nullptr;
        SBD_REQUIRE(rows >= 2 && cols >= 2, SBD_E_INVALID, "sbd_create: rows and cols must be >= 2");
        SBD_REQUIRE(psf_size >= 1 && psf_size <= MAXT, SBD_E_INVALID, "sbd_create: psf_size must be in [1,15]");
        SBD_REQUIRE(psf_size <= rows && psf_size <= cols, SBD_E_INVALID, "sbd_create: PSF larger than the image");
        SBD_REQUIRE(model >= 0 && model <= 2, SBD_E_INVALID, "sbd_create: unknown PSF model");
        SBD_REQUIRE(max_batch >= 1, SBD_E_INVALID, "sbd_create: max_batch must be >= 1");
        // FFT size class from the size alone (no device needed).  A size the FFT operators refuse still makes a context:
        // the TV entry points take any size >= 2; the FFT entry points then fail with this message.
        const std::string fft_err = fft_size_error(rows, cols);
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw Error{SBD_E_NODEVICE, std::string("sbd_create: no CUDA device (") + cudaGetErrorString(e) +
                                         "); libsbd has no CPU fallback"};
        SBD_REQUIRE(device >= 0 && device < ndev, SBD_E_INVALID, "sbd_create: bad device index");
        SBD_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        SBD_CUDA(cudaGetDeviceProperties(&prop, device));
        SBD_REQUIRE(prop.major == 10, SBD_E_NODEVICE,
                    "sbd_create: libsbd is built for sm_100a (Blackwell B200) only");
        c = new sbd_ctx();
        c->device = device; c->nx = rows; c->ny = cols; c->t = psf_size; c->model = model; c->phi = phi;
        c->max_batch = max_batch;
        c->npix = (size_t)rows * cols;
        c->pow2 = is_pow2(rows) && is_pow2(cols) && rows >= 16 && cols >= 16 && rows <= 4096 && cols <= 4096;
        c->smooth = !c->pow2 && fft_err.empty();
        c->fft_err = fft_err;
        c->nk = rows / 2 + 1;
        c->sp = 0;
        if (c->pow2) {
            // column pass: C bins per block (tile-major half spectrum); padded line of ny elements
            const size_t le_y = (size_t)cols + cols / (cols >= 1024 || cols == 256 || cols == 128 ? 16 : (cols == 16 ? 4 : 8));
            // large images with the 7 x 7 PSF of the reference demos: the bulk / tensor-copy passes of fft2.cuh, which
            // use the column-contiguous layout (tile width 1).  SBD_FFT_V2=0 keeps the tiled passes of fft.cuh.
            c->v2 = rows >= 1024 && cols >= 1024 && psf_size == 7 && !(getenv("SBD_FFT_V2") && atoi(getenv("SBD_FFT_V2")) == 0);
            int C = 8;
            const size_t cap = (cols >= 2048) ? 144 * 1024 : 74 * 1024;
            while (C > 1 && (size_t)C * le_y * 16 > cap) C /= 2;
            if (c->v2) C = 1;
            if (const char* e = getenv("SBD_COLS_C")) {
                const int v = atoi(e);
                if ((v == 1 || v == 2 || v == 4 || v == 8) && !c->v2) C = v;
            }
            c->colsC = C;
            c->colsLogC = (C == 8) ? 3 : (C == 4) ? 2 : (C == 2) ? 1 : 0;
            c->ntiles = (c->nk + C - 1) / C;
            // columns per block (<= tile width): bounded by threads (<= 512, the launch bound of k_cols) and shared memory
            int KC = C;
            if (const char* e = getenv("SBD_COLS_KC")) {
                const int v = atoi(e);
                if ((v == 1 || v == 2 || v == 4 || v == 8) && v <= C) KC = v;
            }
            while (KC > 1 && ((size_t)KC * cols / 16 > 512 || (size_t)KC * le_y * 16 > 220 * 1024)) KC /= 2;
            c->colsKC = KC;
            c->colsLogKC = (KC == 8) ? 3 : (KC == 4) ? 2 : (KC == 2) ? 1 : 0;
            c->cols_smem = (size_t)KC * le_y * 16;
        }
        c->spec_elems = (size_t)c->ntiles * cols * c->colsC;
        if (c->smooth) {                // column-contiguous spec[img][k][q]
            any_plan(rows, &c->plan_x);
            any_plan(cols, &c->plan_y);
            c->spec_elems = (size_t)c->nk * cols;
        }
        {
            auto env_int = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
            c->opt_chamb_seg = env_int("SBD_CHAMB_SEG", -1); c->opt_chamb_T = env_int("SBD_CHAMB_T", -1);
            c->opt_tv_seg = env_int("SBD_TV_SEG", -1); c->opt_chamb_emit = env_int("SBD_CHAMB_EMIT", -1);
            c->opt_chamb_plan33 = env_int("SBD_CHAMB_PLAN33", -1);
            c->opt_chamb_errsub = env_int("SBD_CHAMB_ERRSUB", -1);
        }
        c->profile = getenv("SBD_PROFILE") && atoi(getenv("SBD_PROFILE")) != 0;
        SBD_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        SBD_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        SBD_CUDA(cudaEventCreateWithFlags(&c->ev_langevin, cudaEventDisableTiming));
        SBD_CUDA(cudaStreamCreateWithFlags(&c->prox_stream, cudaStreamNonBlocking));
        SBD_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        SBD_CUDA(cudaEventCreateWithFlags(&c->ev_reset, cudaEventDisableTiming));
        SBD_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        if (const char* e = getenv("SBD_OVERLAP")) c->opt_overlap = atoi(e);
        if (const char* e = getenv("SBD_PDL")) c->opt_pdl = atoi(e) != 0;
        if (const char* e = getenv("SBD_CHAMB_COOP")) c->opt_chamb_coop = atoi(e);
        {
            int dev = 0;
            SBD_CUDA(cudaGetDevice(&dev));
            SBD_CUDA(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, dev));
            if (const char* e = getenv("SBD_FFT_PF")) c->fft_pf = atoi(e);
        }
        c->taps = dalloc<double>(3 * MAXT * MAXT);
        c->ctl = dalloc<Control>(1);
        c->psi_dev = dalloc<double>(2);
        c->ximg = dalloc<double>(c->npix);
        c->in_y = dalloc<double>(c->npix);          // staging image of the host-pointer entries (not allocated per call)
        SBD_CUDA(cudaMemsetAsync(c->ctl, 0, sizeof(Control), c->stream));
        if (c->pow2 || c->smooth) {
            c->tw_nx = dalloc<double2>(rows); c->tw_ny = dalloc<double2>(cols);
            make_twiddles(rows, c->tw_nx, c->stream);
            make_twiddles(cols, c->tw_ny, c->stream);
            c->coef = dalloc<double2>((size_t)3 * rows * MAXT);
            c->yhat = dalloc<double2>(c->spec_elems);
            if (c->v2) c->tm_yhat = make_spec_tmap(c, c->yhat, 1);
        }
        SBD_CUDA(cudaStreamSynchronize(c->stream));
        *out = c;
        return SBD_OK;
    } catch (const Error& e) {
        if (c) { sbd_destroy(c); }
        return fail(nullptr, e);
    }
}

int sbd_destroy(sbd_ctx* c) {
    if (!c) return SBD_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    free_ws(c);
    dfree(c->in_y); dfree(c->in_x0); dfree(c->in_xt);
    dfree(c->tw_nx); dfree(c->tw_ny); dfree(c->taps); dfree(c->coef); dfree(c->ctl); dfree(c->psi_dev);
    dfree(c->ximg); dfree(c->yhat); dfree(c->allstats); dfree(c->post);
    dfree(c->post_m2); dfree(c->post_blk); dfree(c->post_out);
    dfree(c->diag_pix); dfree(c->diag_blk); dfree(c->diag_out);
    dfree(c->quant_q); dfree(c->quant_n); dfree(c->quant_blk); dfree(c->quant_out);
    dfree(c->trace_d); dfree(c->trace_i); dfree(c->sal_aty); dfree(c->sal_u); dfree(c->sal_bu); dfree(c->sal_xt);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    if (c->ev_langevin) cudaEventDestroy(c->ev_langevin);
    if (c->prox_stream) { cudaStreamSynchronize(c->prox_stream); cudaStreamDestroy(c->prox_stream); }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_reset) cudaEventDestroy(c->ev_reset);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return SBD_OK;
}

int sbd_synchronize(sbd_ctx* c) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_CUDA(cudaSetDevice(c->device));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    SBD_CATCH(c)
}

// ---------------------------------------------------------------- PSF
int sbd_psf_taps(sbd_ctx* c, const double psi[2], int which, double* out) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(psi && out && which >= 0 && which <= 2, SBD_E_INVALID, "sbd_psf_taps: bad argument");
    SBD_CUDA(cudaSetDevice(c->device));
    psf_from_host(c, psi, 0);
    SBD_CUDA(cudaMemcpyAsync(out, c->taps + (size_t)which * c->t * c->t, sizeof(double) * c->t * c->t,
                             cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    SBD_CATCH(c)
}

int sbd_psf_spectrum(sbd_ctx* c, const double psi[2], int which, double* re, double* im) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(psi && re && im && which >= 0 && which <= 2, SBD_E_INVALID, "sbd_psf_spectrum: bad argument");
    require_fft(c);
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, 1);
    psf_from_host(c, psi, c->nx);
    double* dre = c->X; double* dim_ = c->P;
    k_psf_spectrum<<<(unsigned)((c->npix + 255) / 256), 256, 0, c->stream>>>(c->t, c->nx, c->ny, which, c->coef, c->tw_ny, dre, dim_);
    LAUNCH_CHECK(c);
    SBD_CUDA(cudaMemcpyAsync(re, dre, sizeof(double) * c->npix, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaMemcpyAsync(im, dim_, sizeof(double) * c->npix, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    SBD_CATCH(c)
}

// ---------------------------------------------------------------- blur
int sbd_blur_dev(sbd_ctx* c, const double* d_x, const double psi[2], int op, double* d_out, int batch) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(d_x && d_out && psi && op >= 0 && op <= 3 && batch >= 1, SBD_E_INVALID, "sbd_blur: bad argument");
    SBD_REQUIRE(batch <= c->max_batch, SBD_E_INVALID, "sbd_blur: batch exceeds max_batch");
    SBD_REQUIRE(!(op == SBD_OP_D1 && c->model == SBD_LAPLACE), SBD_E_INVALID, "sbd_blur: Laplace PSF has one parameter");
    require_fft(c);
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, batch);
    psf_from_host(c, psi, c->nk);
    rows_fwd(c, d_x, c->S1, batch);
    cols<COL_OP>(c, c->S1, c->S1, batch, op);
    rows_inv(c, c->S1, d_out, batch);
    SBD_CATCH(c)
}

int sbd_blur(sbd_ctx* c, const double* x, const double psi[2], int op, double* out, int batch) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(x && out && batch >= 1 && batch <= c->max_batch, SBD_E_INVALID, "sbd_blur: bad argument");
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, batch);
    const size_t bytes = sizeof(double) * batch * c->npix;
    SBD_CUDA(cudaMemcpyAsync(c->X, x, bytes, cudaMemcpyHostToDevice, c->stream));
    int rc = sbd_blur_dev(c, c->X, psi, op, c->Gf, batch);
    if (rc) return rc;
    SBD_CUDA(cudaMemcpyAsync(out, c->Gf, bytes, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    SBD_CATCH(c)
}

// ---------------------------------------------------------------- TV
int sbd_tvnorm(sbd_ctx* c, const double* x, double* out, int batch) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(x && out && batch >= 1 && batch <= c->max_batch, SBD_E_INVALID, "sbd_tvnorm: bad argument");
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, batch);
    SBD_CUDA(cudaMemcpyAsync(c->X, x, sizeof(double) * batch * c->npix, cudaMemcpyHostToDevice, c->stream));
    tvnorm(c, c->X, c->stats, NSTAT, batch);
    std::vector<double> h((size_t)batch * NSTAT);
    SBD_CUDA(cudaMemcpyAsync(h.data(), c->stats, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    for (int b = 0; b < batch; ++b) out[b] = h[(size_t)b * NSTAT];
    SBD_CATCH(c)
}

int sbd_diff(sbd_ctx* c, const double* x, int axis, double* out, int batch) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(x && out && (axis == 0 || axis == 1) && batch >= 1 && batch <= c->max_batch, SBD_E_INVALID, "sbd_diff: bad argument");
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, batch);
    const size_t n = (size_t)batch * c->npix;
    SBD_CUDA(cudaMemcpyAsync(c->X, x, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    k_diff<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->X, c->P, c->nx, c->ny, axis, n);
    LAUNCH_CHECK(c);
    SBD_CUDA(cudaMemcpyAsync(out, c->P, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    SBD_CATCH(c)
}

static void set_chamb_options(sbd_ctx* c, double lambda, int maxiter, double tol, double tau) {
    Control h;
    SBD_CUDA(cudaMemcpyAsync(&h, c->ctl, sizeof(Control), cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    h.prox_lambda_theta = lambda; h.maxiter = maxiter; h.tol = tol; h.tau = tau;
    SBD_CUDA(cudaMemcpyAsync(c->ctl, &h, sizeof(Control), cudaMemcpyHostToDevice, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
}

static void fetch_chamb_state(sbd_ctx* c, int batch, int* iters, double* err) {
    if (!iters && !err) return;
    std::vector<ChambState> h(batch);
    SBD_CUDA(cudaMemcpyAsync(h.data(), c->chst, sizeof(ChambState) * batch, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    for (int b = 0; b < batch; ++b) {
        if (iters) iters[b] = h[b].k;
        if (err) err[b] = h[b].err;
    }
}

int sbd_tvprox_dev(sbd_ctx* c, const double* d_g, double lambda, int maxiter, double tol, double tau,
                   double* d_f, int* iters, double* err, int batch) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(d_g && d_f && batch >= 1 && batch <= c->max_batch, SBD_E_INVALID, "sbd_tvprox: bad argument");
    SBD_REQUIRE(maxiter >= 1, SBD_E_INVALID,
                "sbd_tvprox: 'maxiter' is required (the reference leaves MaxIter undefined without it)");
    {   // the tail block writes f while other blocks still read g (and its halo): no in-place use
        const char *g0 = (const char*)d_g, *f0 = (const char*)d_f;
        const size_t bytes = sizeof(double) * (size_t)batch * c->npix;
        SBD_REQUIRE(f0 + bytes <= g0 || g0 + bytes <= f0, SBD_E_INVALID, "sbd_tvprox_dev: d_f must not overlap d_g");
    }
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, batch);
    set_chamb_options(c, lambda, maxiter, tol, tau);
    chambolle(c, d_g, d_f, batch, maxiter, true, false, err != nullptr);
    fetch_chamb_state(c, batch, iters, err);
    SBD_CATCH(c)
}

int sbd_tvprox(sbd_ctx* c, const double* g, double lambda, int maxiter, double tol, double tau,
               const double* dual_px, const double* dual_py, double* f, double* px, double* py,
               int* iters, double* err, int batch) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(g && f && batch >= 1 && batch <= c->max_batch, SBD_E_INVALID, "sbd_tvprox: bad argument");
    SBD_REQUIRE(maxiter >= 1, SBD_E_INVALID,
                "sbd_tvprox: 'maxiter' is required (the reference leaves MaxIter undefined without it)");
    SBD_REQUIRE((dual_px == nullptr) == (dual_py == nullptr), SBD_E_INVALID, "sbd_tvprox: give both dual arrays or none");
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, batch);
    const size_t bytes = sizeof(double) * batch * c->npix;
    set_chamb_options(c, lambda, maxiter, tol, tau);
    SBD_CUDA(cudaMemcpyAsync(c->X, g, bytes, cudaMemcpyHostToDevice, c->stream));
    if (dual_px) {
        SBD_CUDA(cudaMemcpyAsync(c->px0, dual_px, bytes, cudaMemcpyHostToDevice, c->stream));
        SBD_CUDA(cudaMemcpyAsync(c->py0, dual_py, bytes, cudaMemcpyHostToDevice, c->stream));
    }
    chambolle(c, c->X, c->P, batch, maxiter, dual_px == nullptr, px != nullptr || py != nullptr);
    SBD_CUDA(cudaMemcpyAsync(f, c->P, bytes, cudaMemcpyDeviceToHost, c->stream));
    std::vector<ChambState> h(batch);
    SBD_CUDA(cudaMemcpyAsync(h.data(), c->chst, sizeof(ChambState) * batch, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    for (int b = 0; b < batch; ++b) {
        if (iters) iters[b] = h[b].k;
        if (err) err[b] = h[b].err;
        const bool odd = h[b].buf != 0;
        if (px) SBD_CUDA(cudaMemcpyAsync(px + (size_t)b * c->npix, (odd ? c->px1 : c->px0) + (size_t)b * c->npix,
                                         sizeof(double) * c->npix, cudaMemcpyDeviceToHost, c->stream));
        if (py) SBD_CUDA(cudaMemcpyAsync(py + (size_t)b * c->npix, (odd ? c->py1 : c->py0) + (size_t)b * c->npix,
                                         sizeof(double) * c->npix, cudaMemcpyDeviceToHost, c->stream));
    }
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    SBD_CATCH(c)
}

// ---------------------------------------------------------------- likelihood closures
static void set_params_device(sbd_ctx* c, double theta, double sigma2, const double psi[2], double prox_lambda,
                              int maxiter, double tol, double tau) {
    Control h;
    memset(&h, 0, sizeof h);
    h.theta = theta; h.sigma2 = sigma2; h.psi[0] = psi[0]; h.psi[1] = psi[1];
    h.prox_lambda_theta = prox_lambda * theta;
    h.inv_scale = 1.0 / (sigma2 * (double)c->npix);
    h.tau = tau; h.tol = tol; h.maxiter = maxiter;
    h.ii = 2; h.draw = 0; h.phase = 0; h.post_n = 0;
    SBD_CUDA(cudaMemcpyAsync(c->ctl, &h, sizeof(Control), cudaMemcpyHostToDevice, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
}

int sbd_likelihood(sbd_ctx* c, const double* x, const double* y, const double psi[2], double sigma2,
                   double theta, double scal[6], double* gradF) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(x && y && psi && scal, SBD_E_INVALID, "sbd_likelihood: bad argument");
    require_fft(c);
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, 1);
    const size_t bytes = sizeof(double) * c->npix;
    set_params_device(c, theta, sigma2, psi, 1.0, 1, 1e-3, 0.249);
    SBD_CUDA(cudaMemcpyAsync(c->ximg, y, bytes, cudaMemcpyHostToDevice, c->stream));
    rows_fwd(c, c->ximg, c->yhat, 1);
    cols<COL_FWD>(c, c->yhat, c->yhat, 1);
    SBD_CUDA(cudaMemcpyAsync(c->X, x, bytes, cudaMemcpyHostToDevice, c->stream));
    psf_from_host(c, psi, c->nk);
    tvnorm(c, c->X, c->stats, NSTAT, 1);
    rows_fwd(c, c->X, c->S1, 1);
    cols<COL_FWD_REDUCE>(c, c->S1, c->S1, 1);
    if (gradF) {
        cols<COL_MUL_INV>(c, c->S1, c->S2, 1);
        rows_inv(c, c->S2, c->Gf, 1);
        SBD_CUDA(cudaMemcpyAsync(gradF, c->Gf, bytes, cudaMemcpyDeviceToHost, c->stream));
    }
    double st[NSTAT];
    SBD_CUDA(cudaMemcpyAsync(st, c->stats, sizeof st, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    const double dimX = (double)c->npix, tv = st[0], rss = st[1];
    scal[0] = rss / (2.0 * sigma2);
    scal[1] = st[2] / sigma2;
    scal[2] = st[3] / sigma2;
    scal[3] = rss / (2.0 * (sigma2 * sigma2)) - dimX / (2.0 * sigma2);
    scal[4] = tv;
    scal[5] = -scal[0] - theta * tv;
    SBD_CATCH(c)
}

// ---------------------------------------------------------------- setup stage
static double image_sumsq_vs(sbd_ctx* c, const double* d_x, const double* d_ref) {
    k_sqdiff<<<dim3(256, 1), 256, 0, c->stream>>>(d_x, d_ref, c->npix, c->part_sq, c->cnt_sq, c->stats);
    LAUNCH_CHECK(c);
    double st[NSTAT];
    SBD_CUDA(cudaMemcpyAsync(st, c->stats, sizeof st, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    return st[4];
}

int sbd_max_eigenval(sbd_ctx* c, const double psi[2], const double* x0, double tol, int max_iter,
                     uint64_t seed, double* val, int* iters) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(psi && val && max_iter >= 1, SBD_E_INVALID, "sbd_max_eigenval: bad argument");
    require_fft(c);
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, 1);
    const size_t n = c->npix, bytes = sizeof(double) * n;
    const unsigned gb = (unsigned)((n + 255) / 256), gp = (unsigned)(((n + 1) / 2 + 255) / 256);
    double* zero = c->ximg;                                         // all-zero image for the norms
    SBD_CUDA(cudaMemsetAsync(zero, 0, bytes, c->stream));
    if (x0) SBD_CUDA(cudaMemcpyAsync(c->X, x0, bytes, cudaMemcpyHostToDevice, c->stream));
    else { k_philox_image<<<gp, 256, 0, c->stream>>>(c->X, n, seed, 0xFFFF0001u); LAUNCH_CHECK(c); }
    double nrm = std::sqrt(image_sumsq_vs(c, c->X, zero));
    k_div<<<gb, 256, 0, c->stream>>>(c->X, n, nrm); LAUNCH_CHECK(c);    // x = x/norm(x(:))          :5
    psf_from_host(c, psi, c->nk);
    double init_val = 1.0, v = 0.0;                                     // :6
    int k = 0;
    for (k = 1; k <= max_iter; ++k) {                                   // :8
        rows_fwd(c, c->X, c->S1, 1); cols<COL_OP>(c, c->S1, c->S1, 1, SBD_OP_A); rows_inv(c, c->S1, c->P, 1);    // y = A(x)   :9
        rows_fwd(c, c->P, c->S1, 1); cols<COL_OP>(c, c->S1, c->S1, 1, SBD_OP_AT); rows_inv(c, c->S1, c->X, 1);   // x = At(y)  :10
        v = std::sqrt(image_sumsq_vs(c, c->X, zero));                   // val = norm(x(:))           :11
        const double rel_var = std::fabs(v - init_val) / init_val;      // :12
        if (rel_var < tol) break;                                       // :16-18
        init_val = v;                                                   // :19
        k_div<<<gb, 256, 0, c->stream>>>(c->X, n, v); LAUNCH_CHECK(c);  // x = x/val                  :20
    }
    *val = v;
    if (iters) *iters = std::min(k, max_iter);
    SBD_CATCH(c)
}

int sbd_observe(sbd_ctx* c, const double* x, const double psi[2], double bsnr, const double* noise,
                uint64_t seed, double* y, double* sigma, double* ax_norm) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(x && psi && y, SBD_E_INVALID, "sbd_observe: bad argument");
    require_fft(c);
    SBD_CUDA(cudaSetDevice(c->device));
    ensure_ws(c, 1);
    const size_t n = c->npix, bytes = sizeof(double) * n;
    const unsigned gb = (unsigned)((n + 255) / 256), gp = (unsigned)(((n + 1) / 2 + 255) / 256);
    SBD_CUDA(cudaMemcpyAsync(c->X, x, bytes, cudaMemcpyHostToDevice, c->stream));
    psf_from_host(c, psi, c->nk);
    rows_fwd(c, c->X, c->S1, 1); cols<COL_OP>(c, c->S1, c->S1, 1, SBD_OP_A); rows_inv(c, c->S1, c->P, 1);        // Ax  :145
    k_sum<<<256, 256, 0, c->stream>>>(c->P, n, c->part_sq, c->cnt_sq, c->stats + 5);
    LAUNCH_CHECK(c);
    double st[NSTAT];
    SBD_CUDA(cudaMemcpyAsync(st, c->stats, sizeof st, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    const double mean = st[5] / (double)n;                              // mean(mean(Ax))             :148
    k_fill<<<gb, 256, 0, c->stream>>>(c->ximg, n, mean); LAUNCH_CHECK(c);
    const double nrm = std::sqrt(image_sumsq_vs(c, c->P, c->ximg));     // norm(Ax-mean,'fro')
    const double sg = nrm / std::sqrt((double)n * std::pow(10.0, bsnr / 10.0));      // :148
    double* d_noise = nullptr;
    if (noise) {
        d_noise = c->Gf;
        SBD_CUDA(cudaMemcpyAsync(d_noise, noise, bytes, cudaMemcpyHostToDevice, c->stream));
    }
    k_add_noise<<<gp, 256, 0, c->stream>>>(c->P, d_noise, sg, c->X, n, seed, 0xFFFF0002u);   // y = Ax + sigma*noise  :166-168
    LAUNCH_CHECK(c);
    SBD_CUDA(cudaMemcpyAsync(y, c->X, bytes, cudaMemcpyDeviceToHost, c->stream));
    SBD_CUDA(cudaStreamSynchronize(c->stream));
    if (sigma) *sigma = sg;
    if (ax_norm) *ax_norm = nrm;
    SBD_CATCH(c)
}

// ---------------------------------------------------------------- SALSA MAP (post-SAPG)
int sbd_salsa_tv(sbd_ctx* c, const double* y, const double psi[2], double tau, double mu, int maxiter,
                 double tolA, int tv_iters, const double* x_true, double* x, double* objective,
                 double* distance, double* mses, int* n_outer) {
    if (!c) return SBD_E_INVALID;
    double *d_aty = nullptr, *d_u = nullptr, *d_bu = nullptr, *d_xt = nullptr;
    int rc = SBD_OK;
    try {
        SBD_REQUIRE(y && psi && x && maxiter >= 1 && tv_iters >= 1 && mu > 0.0, SBD_E_INVALID, "sbd_salsa_tv: bad argument");
        require_fft(c);
        SBD_CUDA(cudaSetDevice(c->device));
        ensure_ws(c, 1);
        cudaStream_t s = c->stream;
        const size_t n = c->npix, bytes = sizeof(double) * n;
        const unsigned gb = (unsigned)((n + 255) / 256);
        const double P = (double)n;
        if (!c->sal_aty) { c->sal_aty = dalloc<double>(n); c->sal_u = dalloc<double>(n); c->sal_bu = dalloc<double>(n); }
        d_aty = c->sal_aty; d_u = c->sal_u; d_bu = c->sal_bu;
        if (x_true) {
            if (!c->sal_xt) c->sal_xt = dalloc<double>(n);
            d_xt = c->sal_xt;
            SBD_CUDA(cudaMemcpyAsync(d_xt, x_true, bytes, cudaMemcpyHostToDevice, s));
        }
        // Y^, ATy = AT(y)                                                        SALSA_v2.m:287
        SBD_CUDA(cudaMemcpyAsync(c->ximg, y, bytes, cudaMemcpyHostToDevice, s));
        psf_from_host(c, psi, c->nk);
        rows_fwd(c, c->ximg, c->yhat, 1);
        cols<COL_FWD>(c, c->yhat, c->yhat, 1);
        // COL_OP takes the rows-pass output (it does the forward column transform itself)
        rows_fwd(c, c->ximg, c->S1, 1);
        cols<COL_OP>(c, c->S1, c->S1, 1, SBD_OP_AT);
        rows_inv(c, c->S1, d_aty, 1);
        // x = AT(0) = 0, u = x, bu = 0, pux = puy = 0                            :368, :391-392, :418-419
        double* d_x = c->X;
        SBD_CUDA(cudaMemsetAsync(d_x, 0, bytes, s));
        SBD_CUDA(cudaMemsetAsync(d_u, 0, bytes, s));
        SBD_CUDA(cudaMemsetAsync(d_bu, 0, bytes, s));
        SBD_CUDA(cudaMemsetAsync(c->px0, 0, bytes, s));
        SBD_CUDA(cudaMemsetAsync(c->py0, 0, bytes, s));
        // prev_f = 0.5*||y - A(0)||^2 + tau*phi(0) ; mses(1)                      :398-400, :414
        SBD_CUDA(cudaMemsetAsync(c->Gf, 0, bytes, s));
        double st[NSTAT];
        const double yy = image_sumsq_vs(c, c->ximg, c->Gf);
        double prev_obj = 0.5 * yy;
        if (objective) objective[0] = prev_obj;
        if (mses && x_true) mses[0] = image_sumsq_vs(c, d_xt, c->Gf) / P;
        const double threshold = tau / mu;                                        // :393
        set_chamb_options(c, threshold, tv_iters, 1e-3, 0.249);
        c->salsa_mu = mu;
        int outer = 0;
        for (outer = 1; outer <= maxiter; ++outer) {                              // :422
            k_salsa_pre<<<gb, 256, 0, s>>>(d_x, d_bu, c->P, n); LAUNCH_CHECK(c);                 // PTx - bu
            chambolle(c, c->P, d_u, 1, tv_iters, false);                          // :428 (warm start from px0/py0)
            k_salsa_r<<<gb, 256, 0, s>>>(d_aty, d_u, d_bu, mu, c->Gf, n); LAUNCH_CHECK(c);       // :433
            rows_fwd(c, c->Gf, c->S1, 1);
            cols<COL_FILTER>(c, c->S1, c->S1, 1);                                 // x = invLS(r), rss = ||y - A x||^2   :435, :441
            rows_inv(c, c->S1, d_x, 1);
            k_salsa_post<<<256, 256, 0, s>>>(d_x, d_u, d_bu, d_xt, n, c->part_sq, c->cnt_sq, c->stats + 2);   // :439
            LAUNCH_CHECK(c);
            tvnorm(c, d_u, c->stats, NSTAT, 1);                                   // phi(u)
            ChambState hs;
            SBD_CUDA(cudaMemcpyAsync(st, c->stats, sizeof st, cudaMemcpyDeviceToHost, s));
            SBD_CUDA(cudaMemcpyAsync(&hs, c->chst, sizeof hs, cudaMemcpyDeviceToHost, s));
            SBD_CUDA(cudaStreamSynchronize(s));
            if (hs.buf) { std::swap(c->px0, c->px1); std::swap(c->py0, c->py1); }  // next warm start reads px0/py0
            const double obj = 0.5 * st[1] + tau * st[0];                         // :443  (st[1] = rss, Parseval)
            if (objective) objective[outer] = obj;
            if (mses && x_true) mses[outer] = st[5] / P;                          // :447
            if (distance) distance[outer - 1] = std::sqrt(st[2]) / std::sqrt(st[3] + st[4]);      // :450
            bool stop = false;
            if (outer > 1) stop = std::fabs(obj - prev_obj) / prev_obj < tolA;    // :457, :470
            prev_obj = obj;
            if (stop) break;
        }
        if (n_outer) *n_outer = std::min(outer, maxiter);
        SBD_CUDA(cudaMemcpyAsync(x, d_x, bytes, cudaMemcpyDeviceToHost, s));
        SBD_CUDA(cudaStreamSynchronize(s));
    } catch (const Error& e) {
        rc = fail(c, e);
    }
    return rc;
}

// ---------------------------------------------------------------- comm
int sbd_comm_unique_id(char id[SBD_NCCL_ID_BYTES]) {
    if (!id) return SBD_E_INVALID;
    if (!g_nccl.load()) { g_create_error = "sbd_comm_unique_id: libnccl.so.2 not found"; return SBD_E_COMM; }
    nccl_uid u;
    if (g_nccl.GetUniqueId(&u) != 0) { g_create_error = "ncclGetUniqueId failed"; return SBD_E_COMM; }
    memcpy(id, u.internal, SBD_NCCL_ID_BYTES);
    return SBD_OK;
}

int sbd_comm_init(sbd_ctx* c, int nranks, int rank, const char id[SBD_NCCL_ID_BYTES]) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(id && nranks >= 1 && rank >= 0 && rank < nranks, SBD_E_INVALID, "sbd_comm_init: bad argument");
    SBD_REQUIRE(g_nccl.load(), SBD_E_COMM, "sbd_comm_init: libnccl.so.2 not found");
    SBD_CUDA(cudaSetDevice(c->device));
    nccl_uid u;
    memcpy(u.internal, id, SBD_NCCL_ID_BYTES);
    nccl_comm comm = nullptr;
    const int rc = g_nccl.CommInitRank(&comm, nranks, u, rank);
    if (rc != 0)
        throw Error{SBD_E_COMM, std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error")};
    c->comm = comm; c->nranks = nranks; c->rank = rank;
    SBD_CATCH(c)
}

int sbd_comm_destroy(sbd_ctx* c) {
    if (!c) return SBD_E_INVALID;
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    c->comm = nullptr; c->nranks = 1; c->rank = 0;
    return SBD_OK;
}

}  // extern "C"

// ===========================================================================
// SAPG driver
// ===========================================================================
namespace {

// device trace arrays: slices of one block that lives in the context and only ever grows
struct DevTraces {
    Traces t;
    double* delta = nullptr;
    double* errpsf = nullptr;
    double* cur = nullptr;
    double* take(size_t n) { double* p = cur; cur += n; return p; }
};

// spectral analysis of the current X: tv, X^ (in S1) and the Parseval sums
void analyse(sbd_ctx* c, int nch) {
    { PhaseTimer pt(c, 4); tvnorm(c, c->X, c->stats, NSTAT, nch); }
    { PhaseTimer pt(c, 5);
      rows_fwd(c, c->X, c->S1, nch);
      cols<COL_FWD_REDUCE>(c, c->S1, c->S1, nch); }
}

void gather_stats(sbd_ctx* c, int nch, const double** stats_out) {
    if (c->comm) {
        PhaseTimer pt(c, 7);
        const int rc = g_nccl.AllGather(c->stats, c->allstats, (size_t)nch * NSTAT, NCCL_FLOAT64, c->comm, c->stream);
        if (rc != 0) throw Error{SBD_E_COMM, "ncclAllGather failed"};
        *stats_out = c->allstats;
    } else {
        *stats_out = c->stats;
    }
}

void copy_trace(double* dst, const double* src, size_t n, cudaStream_t s) {
    if (dst && n) SBD_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToHost, s));
}

void sapg_run_impl(sbd_ctx* c, const double* d_y, const double* d_X0, const double* d_xtrue,
                   const sbd_params* prm, const double* d_noise, sbd_traces* out) {
    require_fft(c);
    SBD_REQUIRE(prm && out, SBD_E_INVALID, "sbd_sapg_run: params/traces NULL");
    const int nch = prm->n_chains;
    SBD_REQUIRE(nch >= 1 && nch <= c->max_batch, SBD_E_INVALID, "sbd_sapg_run: n_chains must be in [1, max_batch]");
    SBD_REQUIRE(prm->samples >= 1 && prm->warmup >= 0, SBD_E_INVALID, "sbd_sapg_run: samples >= 1, warmup >= 0");
    SBD_REQUIRE(prm->chambolle_maxiter >= 1, SBD_E_INVALID, "sbd_sapg_run: chambolle_maxiter >= 1");
    c->stat_levels = 0;
    c->diag_levels = 0;
    c->quant_levels = 0;
    SBD_REQUIRE(c->post_levels == 0 || prm->burnIn >= 1, SBD_E_INVALID,
                "sbd_sapg_run: posterior statistics (sbd_set_posterior) need burnIn >= 1");
    SBD_REQUIRE(c->post_diag == 0 || c->post_levels > 0, SBD_E_INVALID,
                "sbd_sapg_run: posterior diagnostics (sbd_set_posterior_diagnostics) need the posterior statistics on "
                "(sbd_set_posterior with levels >= 1)");
    SBD_REQUIRE(c->post_ci == 0.0 || c->post_levels > 0, SBD_E_INVALID,
                "sbd_sapg_run: posterior quantiles (sbd_set_posterior_quantiles) need the posterior statistics on "
                "(sbd_set_posterior with levels >= 1)");
    SBD_REQUIRE(c->post_ci == 0.0 ||
                (long long)nch * std::max(prm->samples - prm->burnIn, 0) < (1LL << 31), SBD_E_INVALID,
                "sbd_sapg_run: posterior quantiles need n_chains * (samples - burnIn) < 2^31 (int32 marker positions)");
    const int ntot = std::max(prm->total_chains, nch);
    if (c->comm) SBD_REQUIRE(ntot == nch * c->nranks, SBD_E_INVALID, "sbd_sapg_run: total_chains must be n_chains * nranks");
    else SBD_REQUIRE(ntot == nch, SBD_E_COMM, "sbd_sapg_run: total_chains > n_chains needs sbd_comm_init");
    // geometry (= summation order of the partial sums) from the total chain count: bit-identical for any sharding
    struct GeomReset { sbd_ctx* c; int old; ~GeomReset() { c->geom_total = old; c->geom_batch = -1; } } geom_reset{c, c->geom_total};
    if (c->geom_total < ntot) { c->geom_total = ntot; c->geom_batch = -1; }
    ensure_ws(c, nch);
    cudaStream_t s = c->stream;
    for (int i = 0; i < SBD_N_PHASES; ++i) { c->phase_ms[i] = 0.0; c->phase_calls[i] = 0; }
    const bool want_profile = c->profile;
    c->profile = false;             // phases are timed over the main loop only

    const int samples = prm->samples, warmup = prm->warmup, burnIn = prm->burnIn;
    const int npsi = (c->model == SBD_LAPLACE) ? 1 : 2;
    SapgConst k;
    memset(&k, 0, sizeof k);
    k.model = c->model; k.t = c->t; k.npsi = npsi; k.phi = c->phi;
    k.gam = prm->gam; k.lamb = prm->lamb; k.sq2gam = std::sqrt(2.0 * prm->gam); k.prox_lambda = prm->prox_lambda;
    k.min_th = prm->min_th; k.max_th = prm->max_th; k.c_theta = prm->c_theta;
    for (int p = 0; p < 2; ++p) {
        k.psi_min[p] = prm->psi_min[p]; k.psi_max[p] = prm->psi_max[p]; k.c_psi[p] = prm->c_psi[p];
        k.psi_fixed[p] = prm->psi_fixed[p]; k.fix_psi[p] = prm->fix_psi[p];
    }
    k.sigma2_min = std::min(prm->sigma2_min, prm->sigma2_max);      // Guassian.m:51-52
    k.sigma2_max = std::max(prm->sigma2_min, prm->sigma2_max);
    k.c_sigma2 = prm->c_sigma2; k.sigma2_fixed = prm->sigma2_fixed; k.fix_sigma = prm->fix_sigma;
    k.dimX = (double)c->npix; k.n_local = nch; k.n_total = ntot;
    k.burnIn = burnIn; k.samples = samples; k.warmup = warmup; k.has_xtrue = d_xtrue != nullptr;

    // device traces (no allocation in the steady state: the block is kept in the context)
    DevTraces dt;
    {
        const size_t wu = (size_t)std::max(warmup, 1), S = (size_t)samples;
        const size_t need = wu + 11 * S + (S + 1) + S;
        if (need > c->trace_d_cap) { dfree(c->trace_d); c->trace_d = dalloc<double>(need); c->trace_d_cap = need; }
        if (S > c->trace_i_cap) { dfree(c->trace_i); c->trace_i = dalloc<int>(S); c->trace_i_cap = S; }
        SBD_CUDA(cudaMemsetAsync(c->trace_d, 0, need * sizeof(double), s));
        SBD_CUDA(cudaMemsetAsync(c->trace_i, 0, S * sizeof(int), s));
        dt.cur = c->trace_d;
        dt.t.logPiWU = dt.take(wu);
        dt.t.thetas = dt.take(S); dt.t.sigmas = dt.take(S); dt.t.psi0 = dt.take(S); dt.t.psi1 = dt.take(S);
        dt.t.g_theta = dt.take(S); dt.t.g_psi0 = dt.take(S); dt.t.g_psi1 = dt.take(S); dt.t.g_sigma = dt.take(S);
        dt.t.logPi = dt.take(S); dt.t.gX = dt.take(S); dt.t.sqerr = dt.take(S);
        dt.delta = dt.take(S + 1); dt.errpsf = dt.take(S);
        dt.t.chamb_k = c->trace_i;
        std::vector<double> hd(samples + 1, 0.0);
        for (int i = 1; i <= samples; ++i)                          // delta(i), Guassian.m:55
            hd[i] = prm->d_scale * (std::pow((double)i, -prm->d_exp) / k.dimX);
        SBD_CUDA(cudaMemcpyAsync(dt.delta, hd.data(), sizeof(double) * hd.size(), cudaMemcpyHostToDevice, s));
        SBD_CUDA(cudaStreamSynchronize(s));
        dt.t.delta = dt.delta;
    }
    if (ntot > c->allstats_cap) { dfree(c->allstats); c->allstats = dalloc<double>((size_t)ntot * NSTAT); c->allstats_cap = ntot; }
    // posterior statistics: the running mean becomes required, M2 sits next to it; blocks of size >= 2 in post_blk
    const int L = c->post_levels;
    double* post = nullptr;
    if (prm->post_mean || L > 0) {
        if (c->post_batch < nch) { dfree(c->post); c->post = dalloc<double>((size_t)nch * c->npix); c->post_batch = nch; }
        post = c->post;
        SBD_CUDA(cudaMemsetAsync(post, 0, sizeof(double) * nch * c->npix, s));
    }
    PostGeom pg;
    memset(&pg, 0, sizeof pg);
    size_t blk_half = 0, out_elems = 0;
    unsigned post_tiles = 0;
    if (L > 0) {
        if (c->post_m2_batch < nch) {
            dfree(c->post_m2); c->post_m2 = dalloc<double>((size_t)nch * c->npix); c->post_m2_batch = nch;
        }
        SBD_CUDA(cudaMemsetAsync(c->post_m2, 0, sizeof(double) * nch * c->npix, s));
        pg.rows = c->nx; pg.cols = c->ny; pg.levels = L; pg.tiles_x = (c->nx + POST_TILE - 1) / POST_TILE;
        for (int j = 0; j < L; ++j) {
            const int sz = 1 << j;
            pg.bx[j] = (c->nx + sz - 1) / sz; pg.by[j] = (c->ny + sz - 1) / sz;
            if (j >= 1) { pg.off[j] = blk_half; blk_half += (size_t)nch * post_blocks(c, j); }
            out_elems += 3 * post_blocks(c, j);
        }
        post_tiles = (unsigned)(pg.tiles_x * ((c->ny + POST_TILE - 1) / POST_TILE));
        if (2 * blk_half > c->post_blk_cap) { dfree(c->post_blk); c->post_blk = dalloc<double>(2 * blk_half); c->post_blk_cap = 2 * blk_half; }
        if (out_elems > c->post_out_cap) { dfree(c->post_out); c->post_out = dalloc<double>(out_elems); c->post_out_cap = out_elems; }
        if (blk_half) SBD_CUDA(cudaMemsetAsync(c->post_blk, 0, sizeof(double) * 2 * blk_half, s));
    }
    // batch means and split halves (DiagAcc): the pixel scale in diag_pix, the levels >= 1 in diag_blk, both laid out
    // bsum, mb, m2b [nch][elements], hm, hm2 [2*nch][elements]
    const bool diag = c->post_diag != 0;
    DiagAcc dpix, dblk;
    memset(&dpix, 0, sizeof dpix);
    memset(&dblk, 0, sizeof dblk);
    if (diag) {
        const int n = std::max(samples - burnIn, 0);
        int b = c->post_diag;
        if (b < 0) {                            // floor(sqrt(n))
            b = (int)std::sqrt((double)n);
            while ((long long)b * b > n) --b;
            while ((long long)(b + 1) * (b + 1) <= n) ++b;
        }
        dpix.b = b; dpix.nbatch = b > 0 ? n / b : 0; dpix.h = n / 2; dpix.n = n;
        dblk.b = dpix.b; dblk.nbatch = dpix.nbatch; dblk.h = dpix.h; dblk.n = n;
        const size_t img = (size_t)nch * c->npix;
        if (c->diag_pix_batch < nch) {
            dfree(c->diag_pix); c->diag_pix_batch = 0;          // stays consistent if the allocation throws
            c->diag_pix = dalloc<double>(7 * img); c->diag_pix_batch = nch;
        }
        dpix.bsum = c->diag_pix; dpix.mb = dpix.bsum + img; dpix.m2b = dpix.mb + img;
        dpix.hm = dpix.m2b + img; dpix.hm2 = dpix.hm + 2 * img;
        SBD_CUDA(cudaMemsetAsync(c->diag_pix, 0, sizeof(double) * 7 * img, s));
        if (7 * blk_half > c->diag_blk_cap) {
            dfree(c->diag_blk); c->diag_blk_cap = 0;
            c->diag_blk = dalloc<double>(7 * blk_half); c->diag_blk_cap = 7 * blk_half;
        }
        dblk.bsum = c->diag_blk; dblk.mb = dblk.bsum + blk_half; dblk.m2b = dblk.mb + blk_half;
        dblk.hm = dblk.m2b + blk_half; dblk.hm2 = dblk.hm + 2 * blk_half;
        if (blk_half) SBD_CUDA(cudaMemsetAsync(c->diag_blk, 0, sizeof(double) * 7 * blk_half, s));
        if (2 * out_elems > c->diag_out_cap) {
            dfree(c->diag_out); c->diag_out_cap = 0;
            c->diag_out = dalloc<double>(2 * out_elems); c->diag_out_cap = 2 * out_elems;
        }
    }
    // credible intervals and median (QuantAcc): P^2 state over the E elements of all levels, the pixel scale read
    // from X, the levels >= 1 from the block means k_post_blocks<., true> stores in quant_blk (post_blk layout)
    const bool quant = c->post_ci != 0.0;
    QuantAcc qa;
    memset(&qa, 0, sizeof qa);
    double qp[3] = {0.0, 0.0, 0.0};         // lower, median, upper = f[2], f[4], f[6]
    if (quant) {
        const double al = c->post_ci;
        const double f[9] = {0.0, al / 4, al / 2, 0.25 + al / 4, 0.5, 0.75 - al / 4, 1 - al / 2, 1 - al / 4, 1.0};
        for (int i = 0; i < 9; ++i) qa.f[i] = f[i];
        qp[0] = f[2]; qp[1] = f[4]; qp[2] = f[6];
        qa.levels = L;
        for (int j = 0; j < L; ++j) {
            qa.start[j] = qa.E; qa.nb[j] = post_blocks(c, j); qa.E += qa.nb[j];
        }
        if (qa.E > c->quant_cap) {
            dfree(c->quant_q); dfree(c->quant_n); c->quant_cap = 0;     // stays consistent if an allocation throws
            c->quant_q = dalloc<double>(9 * qa.E); c->quant_n = dalloc<int>(7 * qa.E); c->quant_cap = qa.E;
        }
        if (blk_half > c->quant_blk_cap) {
            dfree(c->quant_blk); c->quant_blk_cap = 0;
            c->quant_blk = dalloc<double>(blk_half); c->quant_blk_cap = blk_half;
        }
        if (out_elems > c->quant_out_cap) {
            dfree(c->quant_out); c->quant_out_cap = 0;
            c->quant_out = dalloc<double>(out_elems); c->quant_out_cap = out_elems;
        }
        qa.q = c->quant_q; qa.np = c->quant_n;
        qa.src[0] = c->X;
        for (int j = 1; j < L; ++j) qa.src[j] = c->quant_blk + pg.off[j];
    }

    cudaEvent_t ev0, ev1;
    SBD_CUDA(cudaEventCreate(&ev0)); SBD_CUDA(cudaEventCreate(&ev1));
    SBD_CUDA(cudaEventRecord(ev0, s));

    // ---- setup: parameters(1), Y^, X = X0 on every chain
    double psi0v[2] = {prm->psi_init[0], prm->psi_init[1]};
    set_params_device(c, prm->th_init, prm->sigma2_init, psi0v, prm->prox_lambda, prm->chambolle_maxiter,
                      prm->chambolle_tol, prm->chambolle_tau);
    k_psf_taps<<<1, 256, 0, s>>>(c->model, c->t, c->phi, c->ctl, nullptr, c->taps);
    LAUNCH_CHECK(c);
    psf_refresh_coef(c, c->nk);
    SBD_CUDA(cudaMemcpyAsync(c->ximg, d_y, sizeof(double) * c->npix, cudaMemcpyDeviceToDevice, s));
    rows_fwd(c, c->ximg, c->yhat, 1);
    cols<COL_FWD>(c, c->yhat, c->yhat, 1);
    k_bcast_image<<<(unsigned)((c->npix + 255) / 256), 256, 0, s>>>(d_X0 ? d_X0 : d_y, c->X, c->npix, nch);
    LAUNCH_CHECK(c);
    if (d_xtrue) {
        k_sqdiff<<<dim3(256, nch), 256, 0, s>>>(c->X, d_xtrue, c->npix, c->part_sq, c->cnt_sq, c->stats);
        LAUNCH_CHECK(c);
        double st[NSTAT];
        SBD_CUDA(cudaMemcpyAsync(st, c->stats, sizeof st, cudaMemcpyDeviceToHost, s));
        SBD_CUDA(cudaStreamSynchronize(s));
        out->err_warm0 = 10.0 * std::log10(st[4] / k.dimX);        // laplace.m:28 via utils/MSE.m:3
    }

    const double* gstats = nullptr;
    bool mark_langevin = false;         // set for the last iteration: X is final once its Langevin kernel has run
    auto prox = [&](int mode) {
        PhaseTimer pt(c, 3);
        const bool rec = mode == 2;         // main loop: sweeps of chain 0 -> `chambolle_iters`
        const bool done = chambolle(c, c->X, c->P, nch, prm->chambolle_maxiter, true, false, false,       // zero start: chambolle_prox_TV_stop.m:68-69
                                    rec ? dt.t.chamb_k : nullptr, samples);
        if (rec && !done) { k_chamb_record<<<1, 1, 0, c->stream>>>(c->chst, c->ctl, dt.t.chamb_k, samples); LAUNCH_CHECK(c); }
    };
    // gradF with the CURRENT parameters from the spectrum of the current sample (S1): what the next Langevin update uses
    auto gradient = [&]() {
        PhaseTimer pt(c, 0);
        cols<COL_MUL_INV>(c, c->S1, c->S2, nch);
        rows_inv(c, c->S2, c->Gf, nch);
    };
    auto scalar = [&](int mode) {
        PhaseTimer pt(c, 6);
        k_sapg_scalar<<<1, 256, 0, s>>>(mode, k, c->ctl, gstats, c->chst, dt.t, c->taps);
        LAUNCH_CHECK(c);
        if (mode == 2) psf_refresh_coef(c, c->nk);
    };
    // One MYULA iteration, starting at its Langevin update (the gradient it needs was formed by the previous unit):
    //     X <- Langevin(X, prox, gradF)                                     Guassian.m:160-161
    //     prox(X, theta_old)                                                :162        } independent of each other:
    //     statistics of X, [all-gather,] scalar update, gradF(new params)   :165-208    } two streams
    // The prox only READS X and its own buffers and works from a snapshot of lambda*theta (k_chamb_reset), so it runs
    // on prox_stream next to the analysis of the same sample, the parameter update and the next gradient - the
    // memory-bound FFT passes fill the issue-bound Chambolle sweeps.  Same kernels, same order per buffer: results
    // are bit-identical to the serial order (SBD_OVERLAP=0 / sbd_set_option("overlap", 0); profiling runs serially).
    auto unit = [&](int mode, bool grad_after) {
        { PhaseTimer pt(c, 1);
          const unsigned gx = (unsigned)(((c->npix + 1) / 2 + 255) / 256);
          if (diag)
              k_langevin<LGV_DIAG><<<dim3(gx, nch), 256, 0, s>>>(c->X, c->P, c->Gf, d_noise, post, c->post_m2, dpix, c->ctl,
                                                                 k.gam, k.lamb, k.sq2gam, c->npix, nch, prm->seed,
                                                                 prm->chain_offset, burnIn);
          else if (L > 0)
              k_langevin<LGV_M2><<<dim3(gx, nch), 256, 0, s>>>(c->X, c->P, c->Gf, d_noise, post, c->post_m2, dpix, c->ctl,
                                                               k.gam, k.lamb, k.sq2gam, c->npix, nch, prm->seed,
                                                               prm->chain_offset, burnIn);
          else
              k_langevin<LGV_MEAN><<<dim3(gx, nch), 256, 0, s>>>(c->X, c->P, c->Gf, d_noise, post, nullptr, dpix, c->ctl,
                                                                 k.gam, k.lamb, k.sq2gam, c->npix, nch, prm->seed,
                                                                 prm->chain_offset, burnIn);
          LAUNCH_CHECK(c);
          if (mark_langevin) SBD_CUDA(cudaEventRecord(c->ev_langevin, s)); }
        const bool ov = c->opt_overlap != 0 && !c->profile;
        if (ov) {
            SBD_CUDA(cudaEventRecord(c->ev_fork, s));
            SBD_CUDA(cudaStreamWaitEvent(c->prox_stream, c->ev_fork, 0));
            {
                StreamScope sc(c, c->prox_stream);
                c->arm_ev_reset = true;
                try { prox(mode); } catch (...) { c->arm_ev_reset = false; throw; }
                c->arm_ev_reset = false;
                SBD_CUDA(cudaEventRecord(c->ev_join, c->stream));
            }
        } else {
            prox(mode);
        }
        if (L >= 2 && mode == 2) {      // block moments of the new sample; reads X, like the prox next to it
            PhaseTimer pt(c, 1);
            auto kb = diag ? (quant ? k_post_blocks<true, true> : k_post_blocks<true, false>)
                           : (quant ? k_post_blocks<false, true> : k_post_blocks<false, false>);
            kb<<<dim3(post_tiles, nch), 256, 0, s>>>(c->X, c->post_blk, c->post_blk + blk_half, dblk, c->quant_blk, pg,
                                                     c->ctl, burnIn);
            LAUNCH_CHECK(c);
        }
        if (quant && mode == 2) {       // P^2 markers of every element; reads X and the block means just stored
            PhaseTimer pt(c, 1);
            k_post_quantile<<<(unsigned)((qa.E + 255) / 256), 256, 0, s>>>(qa, c->ctl, burnIn, nch);
            LAUNCH_CHECK(c);
        }
        analyse(c, nch);
        if (d_xtrue) {
            k_sqdiff<<<dim3(256, nch), 256, 0, s>>>(c->X, d_xtrue, c->npix, c->part_sq, c->cnt_sq, c->stats);
            LAUNCH_CHECK(c);
        }
        gather_stats(c, nch, &gstats);
        if (ov) SBD_CUDA(cudaStreamWaitEvent(s, c->ev_reset, 0));    // the prox has its snapshot of lambda*theta
        scalar(mode);
        if (grad_after) gradient();
        if (ov) SBD_CUDA(cudaStreamWaitEvent(s, c->ev_join, 0));
    };

    // n iterations.  With use_graph the fixed launch sequence of one iteration (all scalars are device-resident, both
    // streams) is captured once and replayed: at small image sizes the iteration is launch-bound and the graph
    // removes most of the per-launch CPU cost.
    // `last_of_run`: the last iteration is launched eagerly, records ev_langevin right after its Langevin kernel (so
    // that the copy of the last samples can overlap its prox / spectral analysis) and forms no gradient after it.
    auto run_loop = [&](int n, int mode, bool last_of_run) {
        if (n <= 0) return;
        // use_graph: 1 on, 0 off, -1 automatic = on for small problems, where the iteration is launch-bound
        const bool want_graph = prm->use_graph > 0 || (prm->use_graph < 0 && (long long)c->npix * nch <= (1LL << 21));
        const bool graph = want_graph && !c->profile && n >= 5;
        if (!graph) {
            for (int i = 0; i < n; ++i) {
                const bool last = last_of_run && i == n - 1;
                mark_langevin = last && out->X_last != nullptr;
                unit(mode, !last);
            }
            mark_langevin = false;
            return;
        }
        if (last_of_run) n -= 1;                                    // the last one runs eagerly below
        unit(mode, true);                                           // first iteration eagerly (sets kernel attributes)
        cudaGraph_t g = nullptr;
        cudaGraphExec_t ge = nullptr;
        const long long l0 = c->launches;
        SBD_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
        try {
            unit(mode, true);
        } catch (...) {
            cudaStreamEndCapture(s, &g);
            if (g) cudaGraphDestroy(g);
            throw;
        }
        SBD_CUDA(cudaStreamEndCapture(s, &g));
        const long long per_iter = c->launches - l0;
        c->launches = l0;
        SBD_CUDA(cudaGraphInstantiate(&ge, g, 0));
        for (int i = 1; i < n; ++i) SBD_CUDA(cudaGraphLaunch(ge, s));
        c->launches += per_iter * (n - 1);
        if (last_of_run) { mark_langevin = out->X_last != nullptr; unit(mode, false); mark_langevin = false; }
        SBD_CUDA(cudaStreamSynchronize(s));
        cudaGraphExecDestroy(ge);
        cudaGraphDestroy(g);
    };

    // ---- warm-up (Guassian.m:67-93)
    analyse(c, nch);
    prox(1);                                                        // :76
    gradient();                                                     // gradF(X_wu; initial parameters) for the first update
    run_loop(warmup - 1, 1, false);                                 // :78  for ii = 2:warmupSteps
    if (out->X_warm)
        SBD_CUDA(cudaMemcpyAsync(out->X_warm, c->X, sizeof(double) * nch * c->npix, cudaMemcpyDeviceToHost, s));

    // ---- main loop (Guassian.m:137-248).  The state after warm-up already holds
    // prox(X, theta(1)) (:140) and the statistics of X for logPiTraceX(1) (:137).
    gather_stats(c, nch, &gstats);      // (also lines the ranks up before the timed main loop)
    scalar(0);
    c->profile = want_profile;
    cudaEvent_t evm;
    SBD_CUDA(cudaEventCreate(&evm));
    SBD_CUDA(cudaEventRecord(evm, s));
    const long long launches0 = c->launches;
    const bool overlap_xlast = out->X_last != nullptr && samples >= 2;
    // the timed region holds the whole work of samples-1 iterations: the gradient of the first one is formed here
    // (again - the warm-up left one behind, outside the clock), the last one forms none after itself
    if (samples >= 2) gradient();
    run_loop(samples - 1, 2, true);                                 // :158  for ii = 2:total_iter
    SBD_CUDA(cudaEventRecord(ev1, s));
    if (overlap_xlast) {
        // X is final after the last Langevin kernel; what follows in that iteration only reads it.  One copy per
        // chain on the copy stream, behind the event: it overlaps the last prox and spectral analysis.
        SBD_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_langevin, 0));
        for (int ch = 0; ch < nch; ++ch)
            SBD_CUDA(cudaMemcpyAsync(out->X_last + (size_t)ch * c->npix, c->X + (size_t)ch * c->npix,
                                     sizeof(double) * c->npix, cudaMemcpyDeviceToHost, c->copy_stream));
    }
    out->launches_main = c->launches - launches0;
    c->profile = false;

    // ---- err_psf on the device, then bring the trajectories home
    const bool dbg_host = getenv("SBD_TRACE_HOST") != nullptr;
    auto now_ms = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double H0 = now_ms();
    if (dbg_host) { cudaStreamSynchronize(s); fprintf(stderr, "[sbd] impl: loops drained after %.1f ms more\n", now_ms() - H0); }
    const double H1 = now_ms();
    double* d_errpsf = dt.errpsf;
    k_err_psf<<<samples, 256, 0, s>>>(c->model, c->t, c->phi, dt.t.psi0, dt.t.psi1, prm->err_psf_lag,
                                      prm->psi_true[0], prm->psi_true[1], samples, d_errpsf);
    LAUNCH_CHECK(c);

    std::vector<double> th(samples), sg(samples), p0(samples), p1(samples), sq(samples);
    SBD_CUDA(cudaMemcpyAsync(th.data(), dt.t.thetas, sizeof(double) * samples, cudaMemcpyDeviceToHost, s));
    SBD_CUDA(cudaMemcpyAsync(sg.data(), dt.t.sigmas, sizeof(double) * samples, cudaMemcpyDeviceToHost, s));
    SBD_CUDA(cudaMemcpyAsync(p0.data(), dt.t.psi0, sizeof(double) * samples, cudaMemcpyDeviceToHost, s));
    SBD_CUDA(cudaMemcpyAsync(p1.data(), dt.t.psi1, sizeof(double) * samples, cudaMemcpyDeviceToHost, s));
    SBD_CUDA(cudaMemcpyAsync(sq.data(), dt.t.sqerr, sizeof(double) * samples, cudaMemcpyDeviceToHost, s));
    copy_trace(out->logPiTrace_WU, dt.t.logPiWU, warmup, s);
    copy_trace(out->grad_theta, dt.t.g_theta, samples, s);
    copy_trace(out->grad_psi0, dt.t.g_psi0, samples, s);
    copy_trace(out->grad_psi1, dt.t.g_psi1, samples, s);
    copy_trace(out->grad_sigma, dt.t.g_sigma, samples, s);
    copy_trace(out->logPiTraceX, dt.t.logPi, samples, s);
    copy_trace(out->gXTrace, dt.t.gX, samples, s);
    copy_trace(out->err_psf, d_errpsf, samples, s);
    if (out->chambolle_iters)
        SBD_CUDA(cudaMemcpyAsync(out->chambolle_iters, dt.t.chamb_k, sizeof(int) * samples, cudaMemcpyDeviceToHost, s));
    if (out->X_last && !overlap_xlast)
        SBD_CUDA(cudaMemcpyAsync(out->X_last, c->X, sizeof(double) * nch * c->npix, cudaMemcpyDeviceToHost, s));
    if (out->X_mean && prm->post_mean) {
        k_chain_mean<<<(unsigned)((c->npix + 255) / 256), 256, 0, s>>>(post, c->Gf, c->npix, nch);
        LAUNCH_CHECK(c);
        SBD_CUDA(cudaMemcpyAsync(out->X_mean, c->Gf, sizeof(double) * c->npix, cudaMemcpyDeviceToHost, s));
    }
    {   // posterior statistics over this context's chains, per level (sbd_posterior_stats copies them out)
        size_t off = 0;
        for (int j = 0; j < L; ++j) {
            const size_t nb = post_blocks(c, j);
            const double* m = j == 0 ? post : c->post_blk + pg.off[j];
            const double* m2 = j == 0 ? c->post_m2 : c->post_blk + blk_half + pg.off[j];
            k_post_finalize<<<(unsigned)((nb + 255) / 256), 256, 0, s>>>(m, m2, nb, nch, c->post_out + off,
                                                                        c->post_out + off + nb, c->post_out + off + 2 * nb);
            LAUNCH_CHECK(c);
            off += 3 * nb;
        }
    }
    if (diag) {  // batch means over the nch chains, halves over the 2*nch half-chains (sbd_posterior_diagnostics)
        size_t off = 0;
        for (int j = 0; j < L; ++j) {
            const size_t nb = post_blocks(c, j);
            const DiagAcc& a = j == 0 ? dpix : dblk;
            const size_t o = j == 0 ? 0 : pg.off[j];
            double* r = c->diag_out + off;
            k_post_finalize<<<(unsigned)((nb + 255) / 256), 256, 0, s>>>(a.mb + o, a.m2b + o, nb, nch, r, r + nb, r + 2 * nb);
            LAUNCH_CHECK(c);
            k_post_finalize<<<(unsigned)((nb + 255) / 256), 256, 0, s>>>(a.hm + 2 * o, a.hm2 + 2 * o, nb, 2 * nch, r + 3 * nb,
                                                                        r + 4 * nb, r + 5 * nb);
            LAUNCH_CHECK(c);
            off += 6 * nb;
        }
    }
    const long long qcount = (long long)nch * std::max(samples - burnIn, 0);
    if (quant) {  // lower / median / upper per level (sbd_posterior_quantiles)
        size_t off = 0;
        for (int j = 0; j < L; ++j) {
            const size_t nb = qa.nb[j];
            double* r = c->quant_out + off;
            k_post_quantile_finalize<<<(unsigned)((nb + 255) / 256), 256, 0, s>>>(
                qa.q, qa.E, qa.start[j], nb, (int)qcount, qp[0], qp[1], qp[2], r, r + nb, r + 2 * nb);
            LAUNCH_CHECK(c);
            off += 3 * nb;
        }
    }
    SBD_CUDA(cudaStreamSynchronize(s));
    if (overlap_xlast) SBD_CUDA(cudaStreamSynchronize(c->copy_stream));
    if (dbg_host) fprintf(stderr, "[sbd] impl: read-back %.1f ms\n", now_ms() - H1);
    float ms = 0.f;
    SBD_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    out->seconds = ms * 1e-3;
    SBD_CUDA(cudaEventElapsedTime(&ms, evm, ev1));
    out->seconds_main = ms * 1e-3;
    cudaEventDestroy(ev0); cudaEventDestroy(ev1); cudaEventDestroy(evm);
    c->profile = want_profile;
    resolve_phase_events(c);
    out->last_samp = samples;                                       // Guassian.m:252 (no early break, Q10)
    if (L > 0) { c->stat_levels = L; c->stat_n = std::max(samples - burnIn, 0); c->stat_chains = nch; }
    if (diag) { c->diag_levels = L; c->diag_b = dpix.b; c->diag_nbatch = dpix.nbatch; c->diag_h = dpix.h; }
    if (quant) { c->quant_levels = L; c->quant_alpha = c->post_ci; c->quant_count = qcount; }

    // ---- host post-processing of the scalar trajectories (Guassian.m:218-247,258-284)
    if (out->thetas) memcpy(out->thetas, th.data(), sizeof(double) * samples);
    if (out->sigmas) memcpy(out->sigmas, sg.data(), sizeof(double) * samples);
    if (out->psi0) memcpy(out->psi0, p0.data(), sizeof(double) * samples);
    if (out->psi1) memcpy(out->psi1, p1.data(), sizeof(double) * samples);
    if (out->err_sample)
        for (int i = 0; i < samples; ++i)
            out->err_sample[i] = d_xtrue ? 10.0 * std::log10(sq[i] / k.dimX) : 0.0;    // utils/MSE.m:3
    const double nan = std::numeric_limits<double>::quiet_NaN();
    const std::vector<double>* trj[4] = {&th, &p0, &p1, &sg};
    double* tolv[4] = {out->tol_theta, out->tol_psi0, out->tol_psi1, out->tol_sigma};
    double* meanv[4] = {out->mean_theta, out->mean_psi0, out->mean_psi1, out->mean_sigma};
    for (int q = 0; q < 4; ++q) {
        const std::vector<double>& v = *trj[q];
        double run = 0.0;           // sum(v(burnIn:ii))
        double prev_mean = nan;     // mean(v(burnIn:ii-1)); empty range -> NaN (Q11)
        if (tolv[q]) tolv[q][0] = 0.0;
        for (int ii = 1; ii <= samples; ++ii) {
            double mean = nan;
            if (burnIn >= 1 && ii >= burnIn) {
                run += v[ii - 1];
                mean = run / (double)(ii - burnIn + 1);
            }
            if (ii >= 2 && tolv[q]) tolv[q][ii - 1] = std::fabs(mean - prev_mean) / prev_mean;   // :218-231
            if (ii > burnIn && ii >= 2 && meanv[q] && burnIn >= 1) meanv[q][ii - burnIn - 1] = mean;  // :236-244
            prev_mean = mean;
        }
        out->EB[q] = (burnIn >= 1 && samples >= burnIn) ? run / (double)(samples - burnIn + 1) : nan;   // :258 (Q12)
    }
}

}  // namespace

extern "C" {

int sbd_sapg_run_dev(sbd_ctx* c, const double* d_y, const double* d_X0, const sbd_params* prm, sbd_traces* out) {
    if (!c) return SBD_E_INVALID;
    SBD_TRY(c)
    SBD_REQUIRE(d_y, SBD_E_INVALID, "sbd_sapg_run_dev: y is NULL");
    SBD_CUDA(cudaSetDevice(c->device));
    sapg_run_impl(c, d_y, d_X0, nullptr, prm, nullptr, out);
    SBD_CATCH(c)
}

int sbd_sapg_run(sbd_ctx* c, const double* y, const double* X0, const double* x_true,
                 const sbd_params* prm, const double* noise, sbd_traces* out) {
    if (!c) return SBD_E_INVALID;
    double *d_x0 = nullptr, *d_xt = nullptr, *d_nz = nullptr;
    int rc = SBD_OK;
    const bool dbg = getenv("SBD_TRACE_HOST") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double T0 = now();
    double T1 = T0, T2 = T0;
    try {
        SBD_REQUIRE(y && prm && out, SBD_E_INVALID, "sbd_sapg_run: y/params/traces NULL");
        SBD_CUDA(cudaSetDevice(c->device));
        const size_t bytes = sizeof(double) * c->npix;
        // staging images live in the context: a cudaFree per call was measured to cost up to 0.6 s here
        // (it tears down whatever the driver deferred, e.g. the graphs of the run)
        if (!c->in_y) c->in_y = dalloc<double>(c->npix);
        SBD_CUDA(cudaMemcpyAsync(c->in_y, y, bytes, cudaMemcpyHostToDevice, c->stream));
        if (X0) {
            if (!c->in_x0) c->in_x0 = dalloc<double>(c->npix);
            d_x0 = c->in_x0;
            SBD_CUDA(cudaMemcpyAsync(d_x0, X0, bytes, cudaMemcpyHostToDevice, c->stream));
        }
        if (x_true) {
            if (!c->in_xt) c->in_xt = dalloc<double>(c->npix);
            d_xt = c->in_xt;
            SBD_CUDA(cudaMemcpyAsync(d_xt, x_true, bytes, cudaMemcpyHostToDevice, c->stream));
        }
        if (noise) {
            const size_t draws = (size_t)std::max(prm->warmup - 1, 0) + (size_t)std::max(prm->samples - 1, 0);
            const size_t n = draws * (size_t)prm->n_chains * c->npix;
            d_nz = dalloc<double>(n);
            SBD_CUDA(cudaMemcpyAsync(d_nz, noise, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
        }
        T1 = now();
        sapg_run_impl(c, c->in_y, d_x0, d_xt, prm, d_nz, out);
        T2 = now();
    } catch (const Error& e) {
        rc = fail(c, e);
    }
    cudaStreamSynchronize(c->stream);
    const double T3 = now();
    if (d_nz) cudaFree(d_nz);
    if (dbg) fprintf(stderr, "[sbd] sapg_run host ms: inputs %.1f  impl %.1f  sync %.1f  free %.1f\n", T1 - T0, T2 - T1, T3 - T2, now() - T3);
    return rc;
}

}  // extern "C"
