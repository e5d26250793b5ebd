// fft_any.cuh - the 2-D real FFT passes for image sizes that are not powers of two: every side in [2, 4096] with no
// prime factor above 7 (fft_plan.h decides which sizes come here).  Same spectral epilogues as fft.cuh / fft2.cuh, on
// a runtime plan.
//
// 1-D engine: mixed-radix Stockham (radices 8, 4, 2, 3, 5, 7; plan in fft_plan.h), in place in ONE shared-memory line
// of n double2.  A stage reads all its operands into registers (a thread owns at most 16 / R butterflies, <= 16
// complex values), waits at a barrier and writes its results.  Twiddles: W_n^m from the exact per-length table
// (tw_nx / tw_ny, long-double on the host), one load per twiddle - no products of table entries, no recurrence.
//
// Layout: column-contiguous half spectrum spec[img][k][q] (k = 0..nx/2, q = 0..ny-1) as in fft2.cuh.
// Rows pass: one block per pair of real lines (z = a + i b), split into the two half spectra with Z[k] <-> Z[n-k]; an
//   odd ny leaves the last line alone, paired with zero.  The Nyquist bin exists only for even nx.
// Column pass: one block per (image, bin k), the column (ny*16 bytes, contiguous) in shared memory.  The PSF spectra
//   K^[k,q] = sum_j c_j(k) W_ny^(q j) are evaluated on the fly (Horner form, any psf_size) from the column coefficients
//   of k_psf_colcoef; Y^ is stored as is (not pre-rotated).
// The geometry (threads per line) depends on the size only, so every sum has the same order for any batch and sharding.
#pragma once
#include "fft.cuh"
#include "fft_plan.h"

namespace sbd {

// ---- small DFTs ---------------------------------------------------------------------------------------------------
// cos / sin (2 pi m / R) for the odd radices
template <int R>
__device__ __forceinline__ constexpr double any_cos(int m) {
    m %= R;
    if (R == 3) return m == 0 ? 1.0 : -0.5;
    if (R == 5) {
        constexpr double c1 = 0.30901699437494742410, c2 = -0.80901699437494742410;
        return m == 0 ? 1.0 : (m == 1 || m == 4) ? c1 : c2;
    }
    constexpr double c1 = 0.62348980185873353053, c2 = -0.22252093395631440429, c3 = -0.90096886790241912624;
    return m == 0 ? 1.0 : (m == 1 || m == 6) ? c1 : (m == 2 || m == 5) ? c2 : c3;
}
template <int R>
__device__ __forceinline__ constexpr double any_sin(int m) {
    m %= R;
    if (R == 3) return m == 0 ? 0.0 : (m == 1 ? 0.86602540378443864676 : -0.86602540378443864676);
    if (R == 5) {
        constexpr double s1 = 0.95105651629515357212, s2 = 0.58778525229247312917;
        return m == 0 ? 0.0 : m == 1 ? s1 : m == 2 ? s2 : m == 3 ? -s2 : -s1;
    }
    constexpr double s1 = 0.78183148246802980871, s2 = 0.97492791218182360702, s3 = 0.43388373911755812048;
    return m == 0 ? 0.0 : m == 1 ? s1 : m == 2 ? s2 : m == 3 ? s3 : m == 4 ? -s3 : m == 5 ? -s2 : -s1;
}

// X[k] = a_k - i b_k, X[R-k] = a_k + i b_k (forward) with a_k = x0 + sum_j (x_j + x_(R-j)) cos(2 pi j k / R),
// b_k = sum_j (x_j - x_(R-j)) sin(2 pi j k / R); the inverse swaps the signs of i b_k
template <int R, bool INV>
__device__ __forceinline__ void dft_odd(double2* v) {
    constexpr int H = (R - 1) / 2;
    double2 s[H], d[H];
#pragma unroll
    for (int j = 1; j <= H; ++j) { s[j - 1] = cadd(v[j], v[R - j]); d[j - 1] = csub(v[j], v[R - j]); }
    double2 out0 = v[0];
#pragma unroll
    for (int j = 0; j < H; ++j) out0 = cadd(out0, s[j]);
#pragma unroll
    for (int k = 1; k <= H; ++k) {
        double2 a = v[0], b = make_double2(0.0, 0.0);
#pragma unroll
        for (int j = 1; j <= H; ++j) {
            const double c = any_cos<R>(j * k), sn = any_sin<R>(j * k);
            a.x = fma(s[j - 1].x, c, a.x); a.y = fma(s[j - 1].y, c, a.y);
            b.x = fma(d[j - 1].x, sn, b.x); b.y = fma(d[j - 1].y, sn, b.y);
        }
        const double2 ib = mul_mi<INV>(b);          // -i b forward, +i b inverse
        v[k] = cadd(a, ib);
        v[R - k] = csub(a, ib);
    }
    v[0] = out0;
}

template <int R, bool INV>
__device__ __forceinline__ void any_dft(double2* v) {
    if constexpr (R == 2) {
        const double2 a = v[0];
        v[0] = cadd(a, v[1]); v[1] = csub(a, v[1]);
    } else if constexpr (R == 4 || R == 8) {
        Dft<R, INV>::run(v);
    } else {
        dft_odd<R, INV>(v);
    }
}

// One in-place Stockham stage of radix R over the line s (n points; ns = product of the earlier radices).
// Butterfly j (< n/R) reads s[j + r n/R], multiplies operand r by W_n^(r k n/(ns R)), k = j mod ns, and writes
// s[(j - k) R + k + r ns].  Load and store are separate calls with the barrier between them in any_fft: the register
// array v is then one for every radix (a barrier inside each radix's code is merged by the compiler, which keeps the
// arrays of all radices live at once - 166 registers for two radices instead of 100).
template <int R, bool INV>
__device__ __forceinline__ void any_stage_load(double2 (&v)[16], const double2* __restrict__ s, int n, int ns, int T,
                                               const double2* __restrict__ tw) {
    constexpr int MB = 16 / R;
    const int nb = n / R, step = n / (ns * R);
#pragma unroll
    for (int m = 0; m < MB; ++m) {
        const int j = threadIdx.x + m * T;
        if (j < nb) {
#pragma unroll
            for (int r = 0; r < R; ++r) v[m * R + r] = s[j + r * nb];
            if (ns > 1) {
                const int k = j % ns;
#pragma unroll
                for (int r = 1; r < R; ++r) v[m * R + r] = cmul(v[m * R + r], twid<INV>(tw, r * k * step));
            }
            any_dft<R, INV>(&v[m * R]);
        }
    }
}
template <int R>
__device__ __forceinline__ void any_stage_store(const double2 (&v)[16], double2* __restrict__ s, int n, int ns, int T) {
    constexpr int MB = 16 / R;
    const int nb = n / R;
#pragma unroll
    for (int m = 0; m < MB; ++m) {
        const int j = threadIdx.x + m * T;
        if (j < nb) {
            const int k = j % ns, base = (j - k) * R + k;
#pragma unroll
            for (int r = 0; r < R; ++r) s[base + r * ns] = v[m * R + r];
        }
    }
}

// Whole transform of the line s (natural order in and out).  The caller has filled s and passed a barrier; every
// thread of the block calls it.
template <bool INV>
__device__ __forceinline__ void any_fft(double2* __restrict__ s, const AnyPlan& p, const double2* __restrict__ tw) {
    int ns = 1;
    for (int st = 0; st < p.nst; ++st) {
        const int R = p.r[st];
        double2 v[16];
        switch (R) {
            case 2: any_stage_load<2, INV>(v, s, p.n, ns, p.T, tw); break;
            case 3: any_stage_load<3, INV>(v, s, p.n, ns, p.T, tw); break;
            case 4: any_stage_load<4, INV>(v, s, p.n, ns, p.T, tw); break;
            case 5: any_stage_load<5, INV>(v, s, p.n, ns, p.T, tw); break;
            case 7: any_stage_load<7, INV>(v, s, p.n, ns, p.T, tw); break;
            default: any_stage_load<8, INV>(v, s, p.n, ns, p.T, tw); break;
        }
        __syncthreads();
        switch (R) {
            case 2: any_stage_store<2>(v, s, p.n, ns, p.T); break;
            case 3: any_stage_store<3>(v, s, p.n, ns, p.T); break;
            case 4: any_stage_store<4>(v, s, p.n, ns, p.T); break;
            case 5: any_stage_store<5>(v, s, p.n, ns, p.T); break;
            case 7: any_stage_store<7>(v, s, p.n, ns, p.T); break;
            default: any_stage_store<8>(v, s, p.n, ns, p.T); break;
        }
        __syncthreads();
        ns *= R;
    }
}

// ---------------------------------------------------------------------------
// rows pass, forward.  grid = (ceil(ny/2), batch), block = p.T, dynamic smem = nx*16 bytes
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(512) k_rows_any_fwd(const double* __restrict__ x, double2* __restrict__ spec, const AnyPlan p,
                                                      int ny, size_t img_stride, size_t spec_stride, const double2* __restrict__ tw) {
    extern __shared__ double2 abuf[];
    const int N = p.n, img = blockIdx.y, q0 = 2 * blockIdx.x;
    const bool two = q0 + 1 < ny;
    const double* xa = x + (size_t)img * img_stride + (size_t)q0 * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) abuf[i] = make_double2(__ldg(xa + i), two ? __ldg(xa + N + i) : 0.0);
    __syncthreads();
    any_fft<false>(abuf, p, tw);
    // A[k] = (Z[k] + conj Z[N-k]) / 2 (line q0), B[k] = (Z[k] - conj Z[N-k]) / (2i) (line q0 + 1)
    double2* so = spec + (size_t)img * spec_stride + q0;
    for (int k = threadIdx.x; k <= N / 2; k += blockDim.x) {
        const double2 zk = abuf[k], zm = abuf[k == 0 ? 0 : N - k];
        so[(size_t)k * ny] = make_double2(0.5 * (zk.x + zm.x), 0.5 * (zk.y - zm.y));
        if (two) so[(size_t)k * ny + 1] = make_double2(0.5 * (zk.y + zm.y), 0.5 * (zm.x - zk.x));
    }
}

// rows pass, inverse (unnormalised; 1/(nx ny) is folded into the column pass).  Same geometry.
__global__ void __launch_bounds__(512) k_rows_any_inv(const double2* __restrict__ spec, double* __restrict__ out, const AnyPlan p,
                                                      int ny, size_t img_stride, size_t spec_stride, const double2* __restrict__ tw) {
    extern __shared__ double2 abuf[];
    const int N = p.n, img = blockIdx.y, q0 = 2 * blockIdx.x;
    const bool two = q0 + 1 < ny;
    const double2* si = spec + (size_t)img * spec_stride + q0;
    for (int k = threadIdx.x; k <= N / 2; k += blockDim.x) {
        const double2 A = __ldg(si + (size_t)k * ny);
        const double2 B = two ? __ldg(si + (size_t)k * ny + 1) : make_double2(0.0, 0.0);
        if (k == 0 || 2 * k == N) {
            abuf[k] = make_double2(A.x, B.x);                   // C2R: imaginary parts of the real bins dropped
        } else {
            abuf[k] = make_double2(A.x - B.y, A.y + B.x);       // Z[k] = A + i B
            abuf[N - k] = make_double2(A.x + B.y, B.x - A.y);   // Z[N-k] = conj(A) + i conj(B)
        }
    }
    __syncthreads();
    any_fft<true>(abuf, p, tw);
    double* xo = out + (size_t)img * img_stride + (size_t)q0 * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const double2 z = abuf[i];
        xo[i] = z.x;
        if (two) xo[N + i] = z.y;
    }
}

// ---------------------------------------------------------------------------
// column pass.  grid = (batch, nk), block = p.T, dynamic smem = ny*16 bytes.  Modes as in fft.cuh (ColMode); a.tw is
// the table of length ny, a.coef the column coefficients of k_psf_colcoef.
// ---------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(512) k_cols_any(const ColArgs a, const AnyPlan p) {
    extern __shared__ double2 abuf[];
    __shared__ double2 coefS[3][MAXT];
    __shared__ double redS[3 * 32];
    const int N = p.n, img = blockIdx.x, k = blockIdx.y;
    const size_t col = (size_t)img * a.spec_stride + (size_t)k * N;
    const double2* in = a.in + col;
    double2* out = a.out + col;
    const double2* yh = a.yhat + (size_t)k * N;
    for (int e = threadIdx.x; e < 3 * a.t; e += blockDim.x) {
        const int m = e / a.t, j = e - m * a.t;
        coefS[m][j] = __ldg(a.coef + ((size_t)m * a.nk + k) * MAXT + j);
    }
    const int msel = (a.opsel == SBD_OP_A || a.opsel == SBD_OP_AT) ? 0 : (a.opsel == SBD_OP_D0 ? 1 : 2);
    const double sc = a.ctl->inv_scale;
    __syncthreads();
    auto kern = [&](int m, int q) { return psf_horner(coefS[m], a.t, __ldg(a.tw + q)); };     // K^[k, q] of kernel m
    for (int q = threadIdx.x; q < N; q += blockDim.x) {
        double2 v = __ldg(in + q);
        if (MODE == COL_MUL_INV) {                  // G^ = conj(H)(H X^ - Y^) / (sigma2 nx ny)
            const double2 H = kern(0, q);
            const double2 R = csub(cmul(H, v), __ldg(yh + q));
            const double2 G = cmulc(R, H);
            v = make_double2(G.x * sc, G.y * sc);
        }
        abuf[q] = v;
    }
    __syncthreads();
    any_fft<MODE == COL_MUL_INV>(abuf, p, a.tw);
    double acc[3] = {0.0, 0.0, 0.0};
    if (MODE == COL_MUL_INV || MODE == COL_FWD) {
        for (int q = threadIdx.x; q < N; q += blockDim.x) out[q] = abuf[q];
    } else if (MODE == COL_FWD_REDUCE) {
        // rss = sum |H X^ - Y^|^2, c_d = sum Re conj(D_d X^)(H X^ - Y^)     (Hermitian weight applied once at the end)
        for (int q = threadIdx.x; q < N; q += blockDim.x) {
            const double2 x = abuf[q];
            out[q] = x;
            const double2 R = csub(cmul(kern(0, q), x), __ldg(yh + q));
            const double2 T0 = cmul(kern(1, q), x);
            acc[0] += R.x * R.x + R.y * R.y;
            acc[1] += T0.x * R.x + T0.y * R.y;
            if (a.npsi > 1) {
                const double2 T1 = cmul(kern(2, q), x);
                acc[2] += T1.x * R.x + T1.y * R.y;
            }
        }
        const double wt = (k == 0 || 2 * k == a.nxfull) ? 1.0 : 2.0;
        acc[0] *= wt; acc[1] *= wt; acc[2] *= wt;
    } else {
        // COL_OP / COL_FILTER: spectral multiply in shared memory, then the inverse transform
        for (int q = threadIdx.x; q < N; q += blockDim.x) {
            const double2 z = abuf[q];
            if (MODE == COL_FILTER) {
                // x = invLS(r): X^ = R^ / (|H|^2 + mu) (run_Gaussian_demo.m:224); rss = |Y^ - H X^|^2
                const double2 H = kern(0, q);
                const double F = 1.0 / ((H.x * H.x + H.y * H.y) + a.mu);
                const double2 X = make_double2(z.x * F, z.y * F);
                const double2 R = csub(__ldg(yh + q), cmul(H, X));
                acc[0] += R.x * R.x + R.y * R.y;
                abuf[q] = make_double2(X.x * a.opscale, X.y * a.opscale);
            } else {
                double2 K = kern(msel, q);
                if (a.opsel == SBD_OP_AT) K.y = -K.y;
                const double2 y = cmul(K, z);
                abuf[q] = make_double2(y.x * a.opscale, y.y * a.opscale);
            }
        }
        if (MODE == COL_FILTER) acc[0] *= (k == 0 || 2 * k == a.nxfull) ? 1.0 : 2.0;
        __syncthreads();
        any_fft<true>(abuf, p, a.tw);
        for (int q = threadIdx.x; q < N; q += blockDim.x) out[q] = abuf[q];
    }

    if (MODE == COL_FWD_REDUCE || MODE == COL_FILTER) {
        block_sum<3>(acc, redS);
        const unsigned int ncolumns = gridDim.y;
        double* part = a.partials + (size_t)img * ncolumns * 4;
        if (threadIdx.x == 0) {
            part[k * 4 + 0] = acc[0];
            part[k * 4 + 1] = acc[1];
            part[k * 4 + 2] = acc[2];
        }
        if (last_block_ticket(a.counters + img, ncolumns)) {
            if (threadIdx.x < 32) {
                const double invP = 1.0 / ((double)a.nxfull * (double)N);
                const double s0 = warp_sum_partials(part + 0, (int)ncolumns, 4);
                const double s1 = warp_sum_partials(part + 1, (int)ncolumns, 4);
                const double s2 = warp_sum_partials(part + 2, (int)ncolumns, 4);
                if (threadIdx.x == 0) {
                    double* st = a.stats + (size_t)img * NSTAT;
                    st[1] = s0 * invP; st[2] = s1 * invP; st[3] = s2 * invP;
                }
            }
        }
    }
}

}  // namespace sbd
