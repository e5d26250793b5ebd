// sapg.cuh - MYULA Langevin update, SAPG scalar updates, monitoring kernels.
//
// Reference lines restated here:
//   Langevin step     SAPG/SAPG_algorithm_Guassian.m:80-81,160-161 (moffat :80-82,159-161; laplace :81-83,154-156)
//   theta update      Guassian.m:165-167   (moffat :167,176-177; laplace :161,169-170)
//   PSF-param update  Guassian.m:170-185   (moffat :164-165,180-193; laplace :159,173-178)
//   sigma^2 update    Guassian.m:188-194   (moffat :166,196-201; laplace :160,181-186)
//   traces            Guassian.m:197-208   (moffat :203-209; laplace :188-195)
//   err_psf           Guassian.m:144-146,203-204 with utils/l2.m:1-3 (squared spectral norm, Q8)
#pragma once
#include "common.cuh"
#include "philox.cuh"
#include "psf.cuh"

namespace sbd {

// ---- batch-means and split-half accumulators (DESIGN.md "Posterior statistics") ---------------------------------
// Per chain and element (a pixel, or a block mean at s >= 2), for the sample v with window index k = ii - burnIn
// (1 .. n), next to the window's Welford pair (m, M2):
//   batch means  k <= B*b: bsum += v; at k = q*b: Y = bsum / b, Welford (mb, M2b) of Y with count q, bsum = 0.
//                The n - B*b samples after the last batch are not batched.
//   split halves half 1 is (m, M2) at k = h, copied there; half 2 is a Welford pair of k = n-h+1 .. n with count
//                k - (n-h).  For odd n the middle sample belongs to neither.
// Layout: bsum, mb, m2b like (m, M2), [chains][elements]; hm, hm2 [2*chains][elements] with half-chain 2c+half-1, so
// that k_post_finalize over 2C "chains" forms the half-chain statistics in the order (c, half 1), (c, half 2).
struct DiagAcc {
    double *bsum, *mb, *m2b, *hm, *hm2;
    int b, nbatch, h, n;                    // batch length b, batches B, half length h, window length n (per run)
};

// NE consecutive elements: one scalar, or two in one 16-byte access
template <int NE>
__device__ __forceinline__ void ld_n(const double* p, double (&v)[NE]) {
    if constexpr (NE == 2) { const double2 t = *reinterpret_cast<const double2*>(p); v[0] = t.x; v[1] = t.y; }
    else v[0] = *p;
}
template <int NE>
__device__ __forceinline__ void st_n(double* p, const double (&v)[NE]) {
    if constexpr (NE == 2) *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
    else *p = v[0];
}

// Sample v of NE consecutive elements at idx in the chain arrays and hidx in half-chain 2c (2c+1 is `stride` further);
// (mn, m2) is the window's Welford pair after v.  Every branch depends only on k and the run constants.
template <int NE>
__device__ __forceinline__ void diag_step(const DiagAcc& a, size_t idx, size_t hidx, size_t stride, int k,
                                          const double (&v)[NE], const double (&mn)[NE], const double (&m2)[NE]) {
    if (k <= a.nbatch * a.b) {
        double s[NE];
        ld_n(a.bsum + idx, s);
#pragma unroll
        for (int e = 0; e < NE; ++e) s[e] += v[e];
        if (k % a.b == 0) {
            const double inv = 1.0 / (double)(k / a.b);
            double m[NE], q[NE];
            ld_n(a.mb + idx, m); ld_n(a.m2b + idx, q);
#pragma unroll
            for (int e = 0; e < NE; ++e) {
                const double y = s[e] / (double)a.b, d = y - m[e];
                m[e] += d * inv;
                q[e] += d * (y - m[e]);
                s[e] = 0.0;
            }
            st_n(a.mb + idx, m); st_n(a.m2b + idx, q);
        }
        st_n(a.bsum + idx, s);
    }
    if (k == a.h) { st_n(a.hm + hidx, mn); st_n(a.hm2 + hidx, m2); }
    const int k2 = k - (a.n - a.h);
    if (k2 >= 1) {
        const double inv = 1.0 / (double)k2;
        double m[NE], q[NE];
        ld_n(a.hm + hidx + stride, m); ld_n(a.hm2 + hidx + stride, q);
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const double d = v[e] - m[e];
            m[e] += d * inv;
            q[e] += d * (v[e] - m[e]);
        }
        st_n(a.hm + hidx + stride, m); st_n(a.hm2 + hidx + stride, q);
    }
}

// what k_langevin accumulates over the window ii = burnIn+1 .. samples besides the running mean
enum { LGV_MEAN = 0, LGV_M2 = 1, LGV_DIAG = 2 };

// X <- | X + gam*(P - X)/lamb - gam*Gf + sqrt(2 gam) Z |   (two elements per thread)
// grid = (ceil(ceil(npix/2)/blockDim), n_chains)
// An odd npix puts the element pairs of every other chain off the 16-byte grid: scalar accesses there, and the last
// element of an image (a pair of its own) takes z0 of its pair (oracle/philox.py).
// LGV_M2: also accumulate the per-chain sum of squared deviations (Welford) next to the running mean; post_m2 is then
// non-null whenever post_mean is.  The mean update is the same expression either way, so X_mean does not change.
// LGV_DIAG: M2 and the batch-means / split-half accumulators of `dg` (diag_step); unused by the other modes.
template <int MODE>
__global__ void k_langevin(double* __restrict__ X, const double* __restrict__ P,
                           const double* __restrict__ Gf, const double* __restrict__ noise,
                           double* __restrict__ post_mean, double* __restrict__ post_m2, const DiagAcc dg,
                           const Control* __restrict__ ctl,
                           double gam, double lamb, double sq2gam, size_t npix, int n_chains,
                           uint64_t seed, int chain_offset, int burnIn) {
    constexpr bool M2 = MODE != LGV_MEAN, DIAG = MODE == LGV_DIAG;
    const size_t pair = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (2 * pair >= npix) return;
    const int ch = blockIdx.y;
    const size_t off = (size_t)ch * npix + 2 * pair;
    const unsigned int draw = ctl->draw;
    if (npix & 1) {
        const bool two = 2 * pair + 1 < npix;
        double2 z;
        if (noise) {
            const double* nz = noise + ((size_t)draw * n_chains + ch) * npix + 2 * pair;
            z = make_double2(__ldg(nz), two ? __ldg(nz + 1) : 0.0);
        } else {
            z = philox_normal2(seed, (uint32_t)(chain_offset + ch), draw, pair);
        }
        const int ne = two ? 2 : 1;
        const bool acc = post_mean && ctl->phase == 1 && ctl->ii > burnIn;
        for (int e = 0; e < ne; ++e) {
            const double x = X[off + e], p = __ldg(P + off + e), gf = __ldg(Gf + off + e), ze = e ? z.y : z.x;
            const double r = fabs(((x + (gam * (p - x)) / lamb) - gam * gf) + sq2gam * ze);
            X[off + e] = r;
            if (acc) {
                const double inv = 1.0 / (double)(ctl->ii - burnIn);
                const double m = post_mean[off + e], d = r - m, mn = m + d * inv;
                post_mean[off + e] = mn;
                if (M2) {
                    const double q = post_m2[off + e] + d * (r - mn);
                    post_m2[off + e] = q;
                    if (DIAG) {
                        const double vr[1] = {r}, vm[1] = {mn}, vq[1] = {q};
                        diag_step<1>(dg, off + e, 2 * (size_t)ch * npix + 2 * pair + e, npix, ctl->ii - burnIn,
                                     vr, vm, vq);
                    }
                }
            }
        }
        return;
    }
    double2 z;
    if (noise) {
        z = __ldg(reinterpret_cast<const double2*>(noise + ((size_t)draw * n_chains + ch) * npix + 2 * pair));
    } else {
        z = philox_normal2(seed, (uint32_t)(chain_offset + ch), draw, pair);
    }
    const double2 x = *reinterpret_cast<const double2*>(X + off);
    const double2 p = __ldg(reinterpret_cast<const double2*>(P + off));
    const double2 gf = __ldg(reinterpret_cast<const double2*>(Gf + off));
    double2 r;
    // evaluated left to right like the MATLAB expression
    r.x = fabs(((x.x + (gam * (p.x - x.x)) / lamb) - gam * gf.x) + sq2gam * z.x);
    r.y = fabs(((x.y + (gam * (p.y - x.y)) / lamb) - gam * gf.y) + sq2gam * z.y);
    *reinterpret_cast<double2*>(X + off) = r;
    if (post_mean && ctl->phase == 1 && ctl->ii > burnIn) {
        // running mean over ii = burnIn+1 .. (posterior mean the reference left stubbed,
        // Guassian.m:233-235,246)
        const double inv = 1.0 / (double)(ctl->ii - burnIn);
        double2 m = *reinterpret_cast<double2*>(post_mean + off);
        const double2 d = make_double2(r.x - m.x, r.y - m.y);
        m.x += d.x * inv;
        m.y += d.y * inv;
        *reinterpret_cast<double2*>(post_mean + off) = m;
        if (M2) {   // M2 += d * (r - m_new)   (Welford; block sizes > 1: k_post_blocks)
            double2 q = *reinterpret_cast<double2*>(post_m2 + off);
            q.x += d.x * (r.x - m.x);
            q.y += d.y * (r.y - m.y);
            *reinterpret_cast<double2*>(post_m2 + off) = q;
            if (DIAG) {
                const double vr[2] = {r.x, r.y}, vm[2] = {m.x, m.y}, vq[2] = {q.x, q.y};
                diag_step<2>(dg, off, 2 * (size_t)ch * npix + 2 * pair, npix, ctl->ii - burnIn, vr, vm, vq);
            }
        }
    }
}

// sum (X - x_true)^2 per chain -> stats[ch*NSTAT + 4]     (laplace.m:189 via utils/MSE.m)
__global__ void k_sqdiff(const double* __restrict__ X, const double* __restrict__ xt, size_t npix,
                         double* __restrict__ partials, unsigned int* __restrict__ counters,
                         double* __restrict__ stats) {
    __shared__ double sm[32];
    const int ch = blockIdx.y;
    double acc[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (size_t)gridDim.x * blockDim.x) {
        const double d = X[(size_t)ch * npix + i] - __ldg(xt + i);
        acc[0] += d * d;
    }
    block_sum<1>(acc, sm);
    double* part = partials + (size_t)ch * gridDim.x;
    if (threadIdx.x == 0) part[blockIdx.x] = acc[0];
    if (last_block_ticket(counters + ch, gridDim.x)) {
        if (threadIdx.x < 32) {
            const double tot = warp_sum_partials(part, (int)gridDim.x, 1);
            if (threadIdx.x == 0) stats[(size_t)ch * NSTAT + 4] = tot;
        }
    }
}

__device__ __forceinline__ double clipd(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// mode 0: start of the main loop (logPiTraceX(1), Guassian.m:137); mode 1: warm-up
// iteration (:85); mode 2: SAPG iteration (:165-208).  One block of 256 threads:
// thread 0 does the scalar algebra, then the block rebuilds the PSF taps for the
// new parameters.  `stats` holds [n_total][NSTAT] per-chain sums in global chain
// order (after the all-gather), so every rank computes bit-identical updates.
__global__ void k_sapg_scalar(int mode, const SapgConst c, Control* __restrict__ ctl,
                              const double* __restrict__ stats, const ChambState* __restrict__ chst,
                              Traces tr, double* __restrict__ taps) {
    __shared__ double sm[3 * MAXT * MAXT + 3];
    if (threadIdx.x == 0) {
        const double th = ctl->theta, s2 = ctl->sigma2;
        double sGt = 0, sG0 = 0, sG1 = 0, sGs = 0, sLp = 0, sGx = 0, sSq = 0;
        for (int ch = 0; ch < c.n_total; ++ch) {
            const double* st = stats + (size_t)ch * NSTAT;
            const double tv = st[0], rss = st[1];
            const double f = rss / (2.0 * s2);                          // op.f, run_Gaussian_demo.m:171
            sGt += c.dimX / th - tv;                                    // Guassian.m:165
            sG0 += st[2] / s2;                                          // op.grad_w1, demo:173
            sG1 += st[3] / s2;                                          // op.grad_w2, demo:174
            sGs += rss / (2.0 * (s2 * s2)) - c.dimX / (2.0 * s2);       // op.gradF_sigma, demo:175
            sLp += -f - th * tv;                                        // op.logPi, demo:195
            sGx += tv;
            sSq += st[4];
        }
        const double n = (double)c.n_total;                             // mean(g_b), moffat.m:170-173
        const double G_t = sGt / n, G_0 = sG0 / n, G_1 = sG1 / n, G_s = sGs / n;
        const double logpi = sLp / n, gx = sGx / n, sq = sSq / n;
        if (mode == 0) {
            tr.logPi[0] = logpi;
            tr.thetas[0] = th; tr.sigmas[0] = s2; tr.psi0[0] = ctl->psi[0]; tr.psi1[0] = ctl->psi[1];
            tr.sqerr[0] = sq;
            tr.chamb_k[0] = chst[0].k;
            ctl->prox_count = 1;                                        // slot of the first main-loop prox (k_chamb_record)
            ctl->ii = 2;
            ctl->phase = 1;
            ctl->post_n = 0;
        } else if (mode == 1) {
            const int ii = ctl->ii;
            tr.logPiWU[ii - 1] = logpi;
            ctl->ii = ii + 1;
            ctl->draw += 1u;
        } else {
            const int ii = ctl->ii, k = ii - 1;
            const double dl = tr.delta[ii];
            const double thn = clipd(th + c.c_theta * dl * G_t, c.min_th, c.max_th);        // :166-167
            double psn[2];
            const double G[2] = {G_0, G_1};
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                const double v = c.fix_psi[p] ? c.psi_fixed[p] : ctl->psi[p] - c.c_psi[p] * dl * G[p];  // :171-175
                psn[p] = (p < c.npsi) ? clipd(v, c.psi_min[p], c.psi_max[p]) : ctl->psi[p];           // :176
            }
            const double sv = c.fix_sigma ? c.sigma2_fixed : s2 + c.c_sigma2 * dl * G_s;    // :189-193
            const double s2n = clipd(sv, c.sigma2_min, c.sigma2_max);                        // :194
            tr.thetas[k] = thn; tr.sigmas[k] = s2n; tr.psi0[k] = psn[0]; tr.psi1[k] = psn[1];
            tr.g_theta[k] = G_t; tr.g_psi0[k] = G_0; tr.g_psi1[k] = G_1; tr.g_sigma[k] = G_s;  // :197-200
            tr.logPi[k] = logpi;                                                            // :207
            tr.gX[k - 1] = gx;                                                              // :208 (Q22)
            tr.sqerr[k] = sq;                                                               // (chamb_k[k]: k_chamb_record)
            ctl->theta = thn; ctl->sigma2 = s2n; ctl->psi[0] = psn[0]; ctl->psi[1] = psn[1];
            ctl->prox_lambda_theta = c.prox_lambda * thn;
            ctl->inv_scale = 1.0 / (s2n * c.dimX);
            ctl->ii = ii + 1;
            ctl->draw += 1u;
        }
    }
    __syncthreads();
    if (mode == 2) {
        __threadfence_block();
        psf_taps_block(c.model, c.t, c.phi, ctl->psi[0], ctl->psi[1], taps, sm);
    }
}

// err_psf(k) = l2(psf(psi0[k], psi1[k - lag]), psf_true) = sigma_max(diff)^2
// (Guassian.m:203-204 with Q9 lag; moffat.m:204-205; laplace.m:190-191; utils/l2.m)
// One block per trajectory slot.
__global__ void k_err_psf(int model, int t, double phi, const double* __restrict__ psi0,
                          const double* __restrict__ psi1, int lag, double true0, double true1,
                          int n, double* __restrict__ out) {
    __shared__ double sm[3 * MAXT * MAXT + 3];
    __shared__ double tp[6 * MAXT * MAXT];
    __shared__ double D[MAXT * MAXT];
    __shared__ double M[MAXT * MAXT];
    const int k = blockIdx.x;
    if (k >= n) return;
    const int kl = (k - lag < 0) ? 0 : k - lag;
    psf_taps_block(model, t, phi, psi0[k], psi1[kl], tp, sm);
    __syncthreads();
    psf_taps_block(model, t, phi, true0, true1, tp + 3 * MAXT * MAXT, sm);
    __syncthreads();
    const int tt = t * t;
    if (threadIdx.x < tt) D[threadIdx.x] = tp[threadIdx.x] - tp[3 * MAXT * MAXT + threadIdx.x];
    __syncthreads();
    if (threadIdx.x < tt) {                         // M = D' * D  (symmetric t x t)
        const int a = threadIdx.x % t, b = threadIdx.x / t;
        double s = 0.0;
        for (int i = 0; i < t; ++i) s += D[a * t + i] * D[b * t + i];
        M[a * t + b] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {                         // cyclic Jacobi eigenvalue iteration
        for (int sweep = 0; sweep < 30; ++sweep) {
            double offd = 0.0;
            for (int p = 0; p < t; ++p)
                for (int q = p + 1; q < t; ++q) offd += M[p * t + q] * M[p * t + q];
            if (offd < 1e-300) break;
            for (int p = 0; p < t; ++p)
                for (int q = p + 1; q < t; ++q) {
                    const double apq = M[p * t + q];
                    if (apq == 0.0) continue;
                    const double app = M[p * t + p], aqq = M[q * t + q];
                    const double tau = (aqq - app) / (2.0 * apq);
                    const double tn = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                    const double cs = 1.0 / sqrt(1.0 + tn * tn), sn = tn * cs;
                    for (int r = 0; r < t; ++r) {
                        const double arp = M[r * t + p], arq = M[r * t + q];
                        M[r * t + p] = cs * arp - sn * arq;
                        M[r * t + q] = sn * arp + cs * arq;
                    }
                    for (int r = 0; r < t; ++r) {
                        const double apr = M[p * t + r], aqr = M[q * t + r];
                        M[p * t + r] = cs * apr - sn * aqr;
                        M[q * t + r] = sn * apr + cs * aqr;
                    }
                }
        }
        double mx = 0.0;
        for (int p = 0; p < t; ++p) mx = fmax(mx, M[p * t + p]);
        out[k] = mx;                                // largest eigenvalue of D'D = norm(D)^2
    }
}

// average the per-chain posterior means
__global__ void k_chain_mean(const double* __restrict__ in, double* __restrict__ out, size_t npix, int n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    double s = 0.0;
    for (int c = 0; c < n; ++c) s += in[(size_t)c * npix + i];
    out[i] = s / (double)n;
}

// ---- posterior moments at block sizes s = 2^j (DESIGN.md "Posterior statistics") --------------------------------
// Per chain and block, Welford accumulators over the main-loop samples ii = burnIn+1 .. samples of the block mean
// v = (sum of the block) / (pixels it contains):  d = v - m;  m += d / n_ii;  M2 += d (v - m),  n_ii = ii - burnIn.
// j = 0 is the pixel scale (k_langevin<LGV_M2>); k_post_blocks does j = 1 .. levels-1.
constexpr int POST_MAXL = 7;                // block sizes 1 .. 64
constexpr int POST_TILE = 64;               // pixels per side of the tile one thread block reduces
struct PostGeom {
    int rows, cols, levels, tiles_x;        // tiles_x = ceil(rows / POST_TILE)
    int bx[POST_MAXL], by[POST_MAXL];       // blocks along rows / cols at level j: ceil(rows / 2^j), ceil(cols / 2^j)
    size_t off[POST_MAXL];                  // level j >= 1: offset of its [n_chains][bx*by] accumulators
};

// DIAG: also the batch-means / split-half accumulators of dg (diag_step); their half-chain arrays of level j start at
// 2 * off[j].  QUANT: also store the block mean v into qv (layout of bm) for k_post_quantile.
template <bool DIAG, bool QUANT>
__device__ __forceinline__ void post_welford(double* __restrict__ bm, double* __restrict__ bm2, const DiagAcc& dg,
                                             double* __restrict__ qv, const PostGeom& g, int j, int ch, int tx, int ty,
                                             int a, int b, double sum, double inv, int k) {
    const int n = POST_TILE >> j, I = tx * n + a, J = ty * n + b;
    if (I >= g.bx[j] || J >= g.by[j]) return;
    const int s = 1 << j;
    const int cnt = (min((I + 1) * s, g.rows) - I * s) * (min((J + 1) * s, g.cols) - J * s);  // partial edge blocks
    const double v = sum / (double)cnt;
    const size_t nb = (size_t)g.bx[j] * g.by[j], e = (size_t)J * g.bx[j] + I;
    const size_t idx = g.off[j] + (size_t)ch * nb + e;
    if (QUANT) qv[idx] = v;
    const double m = bm[idx], d = v - m, mn = m + d * inv;
    bm[idx] = mn;
    if (DIAG) {
        const double q = bm2[idx] + d * (v - mn);
        bm2[idx] = q;
        const double vv[1] = {v}, vm[1] = {mn}, vq[1] = {q};
        diag_step<1>(dg, idx, 2 * g.off[j] + 2 * (size_t)ch * nb + e, nb, k, vv, vm, vq);
    } else {
        bm2[idx] += d * (v - mn);
    }
}

// One 64 x 64 tile of one chain's new sample per block, grid = (tiles, n_chains).  Level 1 sums 2 x 2 pixels read
// straight from X, every further level sums 2 x 2 sums of the level below in shared memory, always as
// (top-left + bottom-left) + (top-right + bottom-right) with zeros outside the image: the order depends only on
// rows, cols and the level.  Runs only in the main loop after burn-in (Control, so a captured graph stays valid).
template <bool DIAG, bool QUANT>
__global__ void __launch_bounds__(256) k_post_blocks(const double* __restrict__ X, double* __restrict__ bm,
                                                     double* __restrict__ bm2, const DiagAcc dg,
                                                     double* __restrict__ qv, const PostGeom g,
                                                     const Control* __restrict__ ctl, int burnIn) {
    __shared__ double sm[32 * 32 + 16 * 16 + 8 * 8 + 4 * 4 + 2 * 2 + 1];
    if (!(ctl->phase == 1 && ctl->ii > burnIn)) return;
    const int k = ctl->ii - burnIn;
    const double inv = 1.0 / (double)k;
    const int ch = blockIdx.y, tx = blockIdx.x % g.tiles_x, ty = blockIdx.x / g.tiles_x;
    const int rows = g.rows, cols = g.cols;
    const double* x = X + (size_t)ch * rows * cols;
    for (int e = threadIdx.x; e < 32 * 32; e += blockDim.x) {
        const int a = e & 31, b = e >> 5;
        const int i = tx * POST_TILE + 2 * a, j = ty * POST_TILE + 2 * b;
        const bool i0 = i < rows, i1 = i + 1 < rows, j0 = j < cols, j1 = j + 1 < cols;
        const double* p = x + (size_t)j * rows + i;
        const double v00 = (i0 && j0) ? p[0] : 0.0, v10 = (i1 && j0) ? p[1] : 0.0;
        const double v01 = (i0 && j1) ? p[rows] : 0.0, v11 = (i1 && j1) ? p[rows + 1] : 0.0;
        const double sum = (v00 + v10) + (v01 + v11);
        sm[e] = sum;
        post_welford<DIAG, QUANT>(bm, bm2, dg, qv, g, 1, ch, tx, ty, a, b, sum, inv, k);
    }
    const double* prev = sm;
    double* cur = sm + 32 * 32;
#pragma unroll      // constant level indices: the PostGeom arrays stay in the parameter bank (no local copy)
    for (int lv = 2; lv < POST_MAXL; ++lv) {
        if (lv >= g.levels) break;
        __syncthreads();
        const int n = POST_TILE >> lv, n2 = 2 * n;
        for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
            const int a = e % n, b = e / n;
            const double* q = prev + 2 * b * n2 + 2 * a;
            const double sum = (q[0] + q[1]) + (q[n2] + q[n2 + 1]);
            cur[e] = sum;
            post_welford<DIAG, QUANT>(bm, bm2, dg, qv, g, lv, ch, tx, ty, a, b, sum, inv, k);
        }
        prev = cur;
        cur += n * n;
    }
}

// Over the chains of this context, per element of one level (local chain order, as k_chain_mean):
// mean = (sum_c m_c) / C,  within = sum_c M2_c,  between = sum_c (m_c - mean)^2
__global__ void k_post_finalize(const double* __restrict__ m, const double* __restrict__ m2, size_t nb, int n,
                                double* __restrict__ mean, double* __restrict__ within, double* __restrict__ between) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    double s = 0.0;
    for (int c = 0; c < n; ++c) s += m[(size_t)c * nb + i];
    const double mu = s / (double)n;
    double w = 0.0, b = 0.0;
    for (int c = 0; c < n; ++c) {
        w += m2[(size_t)c * nb + i];
        const double d = m[(size_t)c * nb + i] - mu;
        b += d * d;
    }
    mean[i] = mu; within[i] = w; between[i] = b;
}

// ---- posterior quantiles: extended P^2 (DESIGN.md "Credible intervals and the median") --------------------------
// One estimator per element of every level (not per chain): at each main-loop step after burn-in the values of the C
// chains are fed in local chain order, so after k window steps it has seen N = C*k values.  9 markers, heights q_i and
// integer positions n_i with desired positions 1 + (N-1) f_i.  N <= 9: q holds the values sorted.  Every expression is
// that of tests/posterior_quantile_oracle.py, evaluated with __d*_rn (no FMA contraction), so both agree bitwise.
// State SoA over the E elements of all levels: q [9][E], np [7][E] (n_1 .. n_7; n_0 = 1 and n_8 = N are implied).
struct QuantAcc {
    double* q;
    int* np;
    double f[9];                            // marker probabilities, formed on the host
    size_t E;                               // elements of all levels
    int levels;
    size_t start[POST_MAXL];                // first element of level j
    size_t nb[POST_MAXL];                   // elements of level j = chain stride of its values
    const double* src[POST_MAXL];           // values of level j: X (j = 0), block means of k_post_blocks (j >= 1)
};

// one thread per element of all levels; grid = ceil(E / 256).  Runs only in the main loop after burn-in (Control).
__global__ void __launch_bounds__(256) k_post_quantile(const QuantAcc a, const Control* __restrict__ ctl, int burnIn,
                                                       int n_chains) {
    if (!(ctl->phase == 1 && ctl->ii > burnIn)) return;
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.E) return;
    const double* src = a.src[0];
    size_t nb = a.nb[0], le = e;
#pragma unroll      // constant level indices: the QuantAcc arrays stay in the parameter bank
    for (int j = 1; j < POST_MAXL; ++j)
        if (j < a.levels && e >= a.start[j]) { src = a.src[j]; nb = a.nb[j]; le = e - a.start[j]; }
    int N = (ctl->ii - burnIn - 1) * n_chains;      // values seen before this step (C*n < 2^31: checked on the host)
    double q[9];
    int n[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) q[i] = a.q[(size_t)i * a.E + e];
#pragma unroll
    for (int i = 1; i < 8; ++i) n[i] = a.np[(size_t)(i - 1) * a.E + e];
    n[0] = 1;
    for (int c = 0; c < n_chains; ++c, ++N) {
        const double x = __ldg(src + (size_t)c * nb + le);
        if (N < 9) {                                // insertion: q[0..N] sorted, x after the values <= x
#pragma unroll
            for (int i = 8; i >= 0; --i) {
                if (i <= N) {
                    const bool keep = i < N && q[i] <= x;
                    const bool shift = i >= 1 && q[i >= 1 ? i - 1 : 0] > x;
                    q[i] = keep ? q[i] : (shift ? q[i >= 1 ? i - 1 : 0] : x);
                }
            }
            if (N == 8) {
#pragma unroll
                for (int i = 1; i < 8; ++i) n[i] = i + 1;
            }
            continue;
        }
        int k = 0;
        if (x < q[0]) { q[0] = x; k = 0; }
        else if (x >= q[8]) { q[8] = x; k = 7; }
        else {
#pragma unroll
            for (int i = 1; i < 8; ++i) if (q[i] <= x) k = i;
        }
#pragma unroll
        for (int i = 1; i < 8; ++i) n[i] += i > k;
        n[8] = N + 1;                               // the count after x
        const double Nm1 = (double)N;               // (N+1) - 1
#pragma unroll
        for (int i = 1; i < 8; ++i) {
            const double d = __dsub_rn(__dadd_rn(1.0, __dmul_rn(Nm1, a.f[i])), (double)n[i]);
            const int dr = n[i + 1] - n[i], dl = n[i] - n[i - 1];
            if ((d >= 1.0 && dr > 1) || (d <= -1.0 && dl > 1)) {
                // parabolic prediction over one common denominator: one division per moving marker instead of three
                // (the markers of a warp move in different iterations; profiles/r06_posterior_quantiles.md)
                const int s = d >= 1.0 ? 1 : -1;
                const double sd = (double)s, ndr = (double)dr, ndl = (double)dl;
                const double dq1 = __dsub_rn(q[i + 1], q[i]), dq0 = __dsub_rn(q[i], q[i - 1]);
                const double num = __dadd_rn(__dmul_rn(__dmul_rn(__dadd_rn(ndl, sd), ndl), dq1),
                                             __dmul_rn(__dmul_rn(__dsub_rn(ndr, sd), ndr), dq0));
                const double den = __dmul_rn(__dmul_rn(ndr, ndl), __dadd_rn(ndr, ndl));
                const double qp = __dadd_rn(q[i], __ddiv_rn(__dmul_rn(sd, num), den));
                if (q[i - 1] < qp && qp < q[i + 1]) q[i] = qp;
                else q[i] = __dadd_rn(q[i], __dmul_rn(sd, s > 0 ? __ddiv_rn(dq1, ndr) : __ddiv_rn(dq0, ndl)));
                n[i] += s;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) a.q[(size_t)i * a.E + e] = q[i];
#pragma unroll
    for (int i = 1; i < 8; ++i) a.np[(size_t)(i - 1) * a.E + e] = n[i];
}

// lower / median / upper (probabilities p[0..2]) of the nb elements of one level starting at element e0 after N
// values: N >= 9 the markers q_2, q_4, q_6; 1 <= N < 9 the linear interpolation of the sorted values
// v[h] + (h - floor h)(v[h+1] - v[h]), h = (N-1) p; N = 0 NaN
__global__ void k_post_quantile_finalize(const double* __restrict__ q, size_t E, size_t e0, size_t nb, int N,
                                         double p0, double p1, double p2, double* __restrict__ lower,
                                         double* __restrict__ median, double* __restrict__ upper) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    const double* v = q + e0 + i;
    const double p[3] = {p0, p1, p2};
    double r[3];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        if (N >= 9) {
            r[t] = v[(size_t)(2 + 2 * t) * E];
        } else if (N == 0) {
            r[t] = __longlong_as_double(0x7ff8000000000000LL);
        } else {
            const double h = __dmul_rn((double)(N - 1), p[t]), fl = floor(h), fr = __dsub_rn(h, fl);
            const int lo = (int)fl;
            const double vl = v[(size_t)lo * E];
            r[t] = fr == 0.0 ? vl : __dadd_rn(vl, __dmul_rn(fr, __dsub_rn(v[(size_t)(lo + 1) * E], vl)));
        }
    }
    lower[i] = r[0]; median[i] = r[1]; upper[i] = r[2];
}

// sum of x over one image -> out[0]   (mean(mean(Ax)), run_Gaussian_demo.m:148)
__global__ void k_sum(const double* __restrict__ x, size_t npix, double* __restrict__ partials,
                      unsigned int* __restrict__ counter, double* __restrict__ out) {
    __shared__ double sm[32];
    double acc[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (size_t)gridDim.x * blockDim.x) acc[0] += x[i];
    block_sum<1>(acc, sm);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc[0];
    if (last_block_ticket(counter, gridDim.x)) {
        if (threadIdx.x < 32) {
            const double tot = warp_sum_partials(partials, (int)gridDim.x, 1);
            if (threadIdx.x == 0) out[0] = tot;
        }
    }
}

__global__ void k_fill(double* __restrict__ x, size_t n, double v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = v;
}

__global__ void k_scale(double* __restrict__ x, size_t n, double a) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = x[i] * a;         // the reference divides (x = x/val); a = 1/val is passed as such
}

__global__ void k_div(double* __restrict__ x, size_t n, double d) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = x[i] / d;
}

// y = ax + sigma * z, z from `noise` or Philox (stream = 0xFFFF0000 + which)
__global__ void k_add_noise(const double* __restrict__ ax, const double* __restrict__ noise, double sigma,
                            double* __restrict__ y, size_t npix, uint64_t seed, uint32_t stream) {
    const size_t pair = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (2 * pair >= npix) return;
    if (npix & 1) {                 // the last element of an odd image takes z0 of its pair
        const bool two = 2 * pair + 1 < npix;
        const double2 z = noise ? make_double2(noise[2 * pair], two ? noise[2 * pair + 1] : 0.0)
                                : philox_normal2(seed, stream, 0u, pair);
        y[2 * pair] = ax[2 * pair] + sigma * z.x;
        if (two) y[2 * pair + 1] = ax[2 * pair + 1] + sigma * z.y;
        return;
    }
    double2 z;
    if (noise) z = *reinterpret_cast<const double2*>(noise + 2 * pair);
    else z = philox_normal2(seed, stream, 0u, pair);
    const double2 a = *reinterpret_cast<const double2*>(ax + 2 * pair);
    *reinterpret_cast<double2*>(y + 2 * pair) = make_double2(a.x + sigma * z.x, a.y + sigma * z.y);
}

__global__ void k_philox_image(double* __restrict__ x, size_t npix, uint64_t seed, uint32_t stream) {
    const size_t pair = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (2 * pair >= npix) return;
    const double2 z = philox_normal2(seed, stream, 0u, pair);
    if (npix & 1) {                 // odd image: the last element takes z0 of its pair
        x[2 * pair] = z.x;
        if (2 * pair + 1 < npix) x[2 * pair + 1] = z.y;
        return;
    }
    *reinterpret_cast<double2*>(x + 2 * pair) = z;
}

// ---- SALSA (ADMM) elementwise pieces, SALSA/SALSA_v2.m:428-450 ----------------------------
// v = PTx - bu                                                                (:428 argument)
__global__ void k_salsa_pre(const double* __restrict__ x, const double* __restrict__ bu, double* __restrict__ v, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = x[i] - bu[i];
}
// r = ATy + mu*(u + bu)                                                       (:433)
__global__ void k_salsa_r(const double* __restrict__ aty, const double* __restrict__ u, const double* __restrict__ bu,
                          double mu, double* __restrict__ r, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) r[i] = aty[i] + mu * (u[i] + bu[i]);
}
// bu = bu + (u - x) (:439) and the sums for `distance` (:450) and `mses` (:447):
// out[0] = sum (x-u)^2, out[1] = sum x^2, out[2] = sum u^2, out[3] = sum (x-true)^2
__global__ void k_salsa_post(const double* __restrict__ x, const double* __restrict__ u, double* __restrict__ bu,
                             const double* __restrict__ xtrue, size_t n, double* __restrict__ partials,
                             unsigned int* __restrict__ counter, double* __restrict__ out) {
    __shared__ double sm[4 * 32];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const double xv = x[i], uv = u[i];
        bu[i] = bu[i] + (uv - xv);
        const double d = xv - uv;
        acc[0] += d * d; acc[1] += xv * xv; acc[2] += uv * uv;
        if (xtrue) { const double e = xv - xtrue[i]; acc[3] += e * e; }
    }
    block_sum<4>(acc, sm);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) partials[q * gridDim.x + blockIdx.x] = acc[q];
    }
    if (last_block_ticket(counter, gridDim.x)) {
        if (threadIdx.x < 32) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double tot = warp_sum_partials(partials + q * gridDim.x, (int)gridDim.x, 1);
                if (threadIdx.x == 0) out[q] = tot;
            }
        }
    }
}

__global__ void k_bcast_image(const double* __restrict__ src, double* __restrict__ dst, size_t npix, int n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const double v = src[i];
    for (int c = 0; c < n; ++c) dst[(size_t)c * npix + i] = v;
}

}  // namespace sbd
