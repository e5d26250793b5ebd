// psf.cuh - parametric PSF taps, their parameter derivatives and the
// on-the-fly spectrum  H[k,q] = sum_{i,j<t} h[i,j] e^{-2 pi i k i/nx} e^{-2 pi i q j/ny}
// which is what utils/resize.m:1-12 (pad at the top-left corner + fft2) yields.
//
// Reference formulas restated here:
//   utils/Gaussian_psf.m:2-19, utils/Sum_gauss_psf.m:1-28, utils/diff_fftgaus_w1.m:2-26, w2.m:2-26
//   utils/moffat_psf.m:2-23,   utils/sum_mof_psf.m:1-40,   utils/diff_moffat_alpha.m:1-22, beta.m:1-23
//   utils/laplace_psf.m:1-15,  utils/sum_lap_psf.m:1-28,   utils/diff_laplace_b.m:1-19
#pragma once
#include "common.cuh"
#include <type_traits>

namespace sbd {

// One block (>= t*t threads, blockDim <= 256).  taps layout: [m][j*t + i],
// m = 0 PSF, 1 d/dpsi0, 2 d/dpsi1;  i = row (fast axis), j = column.
// `sm` : 3*MAXT*MAXT + 3 doubles of shared memory.
__device__ __forceinline__ void psf_taps_block(int model, int t, double phi, double p0, double p1,
                                               double* __restrict__ taps, double* sm) {
    const int e = threadIdx.x, tt = t * t;
    double f = 0.0, d0 = 0.0, d1 = 0.0;
    if (e < tt) {
        const int i = e % t, j = e / t;
        const double half = 0.5 * (double)(t - 1);
        const double xi = (double)i - half;         // row coordinate   (v in Gaussian_psf.m:9)
        const double xj = (double)j - half;         // column coordinate (u)
        const double twopi = 6.283185307179586476925286766559;
        if (model == SBD_GAUSSIAN) {
            const double w1 = p0, w2 = p1;
            double sn, cs;
            sincos(phi, &sn, &cs);
            const double U = xj * cs - xi * sn;     // Gaussian_psf.m:11
            const double V = xj * sn + xi * cs;     // :12
            const double c = w1 * w1 * (U * U) + w2 * w2 * (V * V);    // :14
            const double ex = exp(-c / 2.0);
            f = ((w1 * w2) / twopi) * ex;                               // :16
            d0 = (w2 / twopi) * (1.0 - w1 * w1 * (U * U)) * ex;         // Sum_gauss_psf.m:22
            d1 = (w1 / twopi) * (1.0 - w2 * w2 * (V * V)) * ex;         // Sum_gauss_psf.m:20
        } else if (model == SBD_MOFFAT) {
            const double a = p0, b = p1, b2 = b + 2.0;
            const double xy = xi * xi + xj * xj;                        // moffat_psf.m:15
            const double a2 = a * a;
            const double base = xy * a2 / b + 1.0;
            const double pw = pow(base, -b2 / 2.0);
            f = a2 * pw / twopi;                                        // moffat_psf.m:16
            // diff_moffat_alpha.m:17 - the stray 2 in the denominator is the reference's (Q7)
            d0 = (2.0 - ((b2 * xy * a2) / (2.0 * (b + xy * a2)))) * pw * (a / twopi);
            // diff_moffat_beta.m:17-18
            d1 = (-log(base) + (b2 * xy * a2) / (b * (b + xy * a2))) * pw * (a2 / (2.0 * twopi));
        } else {
            const double b = p0;
            const double s = fabs(xi) + fabs(xj);
            const double ex = exp(-b * s);
            f = (b * b / 4.0) * ex;                                     // laplace_psf.m:8
            d0 = ((2.0 * b - b * b * s) / 4.0) * ex;                    // diff_laplace_b.m:10-12
            d1 = 0.0;
        }
        sm[e] = f; sm[MAXT * MAXT + e] = d0; sm[2 * MAXT * MAXT + e] = d1;
    }
    __syncthreads();
    if (threadIdx.x < 3) {                           // sequential sums (fixed order)
        double s = 0.0;
        const double* p = sm + threadIdx.x * MAXT * MAXT;
        for (int q = 0; q < tt; ++q) s += p[q];
        sm[3 * MAXT * MAXT + threadIdx.x] = s;
    }
    __syncthreads();
    if (e < tt) {
        const double S = sm[3 * MAXT * MAXT], S0 = sm[3 * MAXT * MAXT + 1], S1 = sm[3 * MAXT * MAXT + 2];
        taps[e] = f / S;                                                // Gaussian_psf.m:18
        taps[tt + e] = (d0 * S - f * S0) / (S * S);                     // diff_fftgaus_w1.m:24
        taps[2 * tt + e] = (d1 * S - f * S1) / (S * S);
    }
}

__global__ void k_psf_taps(int model, int t, double phi, const Control* __restrict__ ctl,
                           const double* __restrict__ psi_override, double* __restrict__ taps) {
    __shared__ double sm[3 * MAXT * MAXT + 3];
    const double p0 = psi_override ? psi_override[0] : ctl->psi[0];
    const double p1 = psi_override ? psi_override[1] : ctl->psi[1];
    psf_taps_block(model, t, phi, p0, p1, taps, sm);
}

// coef[m][k][j] = sum_i taps[m][j*t+i] * W_nx^{k i},  k < nk, j < t.
// One thread per (m,k,j).  tw_nx[n] = exp(-2 pi i n / nx).
__global__ void k_psf_colcoef(int t, int nx, int nk, const double* __restrict__ taps,
                              const double2* __restrict__ tw_nx, double2* __restrict__ coef) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int total = 3 * nk * t;
    if (idx >= total) return;
    const int j = idx % t, k = (idx / t) % nk, m = idx / (t * nk);
    const double* h = taps + (size_t)m * t * t + (size_t)j * t;
    double re = 0.0, im = 0.0;
    for (int i = 0; i < t; ++i) {
        const double2 w = tw_nx[(int)(((long long)k * i) % nx)];
        re = fma(h[i], w.x, re);
        im = fma(h[i], w.y, im);
    }
    coef[((size_t)m * nk + k) * MAXT + j] = make_double2(re, im);
}

// Horner evaluation of sum_j a[j] w^j
__device__ __forceinline__ double2 psf_horner(const double2* __restrict__ a, int t, double2 w) {
    double2 acc = a[t - 1];
    for (int j = t - 2; j >= 0; --j) acc = cfma(acc, w, a[j]);
    return acc;
}

// Point-symmetric 7-tap form (psf_size = 7, the size of every reference demo).  The taps of the three
// models satisfy h[i][j] = h[6-i][6-j] (also the rotated Gaussian, phi != 0), so the column coefficients
// c_j(k) = sum_i h[i][j] wk^i obey c_(6-j) = wk^6 conj(c_j).  With d_j = wk^-3 c_j (d_(6-j) = conj d_j) and
// w = e^(i th), |w| = 1:
//     sum_j c_j w^j = (wk w)^3 * S,    S = e0 + sum_{m=1..3} (e_m cos(m th) + f_m sin(m th))   REAL
//     e0 = Re d_3,  e_m = Re(d_(3+m) + d_(3-m)),  f_m = -Im(d_(3+m) - d_(3-m)),  (cos, sin)(m th) = w^m
// i.e. 6 real multiply-adds per kernel, and the complex factor (wk w)^3 is shared by the three kernels
// of the likelihood pass (the Horner form costs 24 per kernel).  b[m] = (e_m, f_m); b[0] = (e0, 0).
struct PsfW3 { double c1, s1, c2, s2; double2 w3; };
__device__ __forceinline__ PsfW3 psf_w3(double2 w) {
    const double2 w2 = cmul(w, w);
    PsfW3 p;
    p.w3 = cmul(w2, w);
    p.c1 = w.x; p.s1 = w.y; p.c2 = w2.x; p.s2 = w2.y;
    return p;
}
__device__ __forceinline__ double psf_sym3(const double2* __restrict__ b, const PsfW3& p) {
    double s = b[0].x;
    s = fma(b[1].x, p.c1, s); s = fma(b[1].y, p.s1, s);
    s = fma(b[2].x, p.c2, s); s = fma(b[2].y, p.s2, s);
    s = fma(b[3].x, p.w3.x, s); s = fma(b[3].y, p.w3.y, s);
    return s;
}
// the (e_m, f_m) pair from the column coefficients c[0..6] and wk3c = conj(wk^3)
__device__ __forceinline__ double2 psf_sym3_coef(const double2* __restrict__ c, double2 wk3c, int m) {
    if (m == 0) return make_double2(cmul(wk3c, c[3]).x, 0.0);
    const double2 hi = cmul(wk3c, c[3 + m]), lo = cmul(wk3c, c[3 - m]);
    return make_double2(hi.x + lo.x, -(hi.y - lo.y));
}

// ---------------------------------------------------------------------------
// The real factor S along the R outputs of one radix-R butterfly.
// A thread of the column pass owns, per butterfly, the bins q_r = jb + r*N/R, r = 0..R-1 (the outputs of the last
// forward stage, or the operands of the first inverse stage), i.e. w_(q_r) = w_jb * W_R^r with W_R = e^(-2 pi i / R).
// With A_j = (e_j - i f_j) * w_jb^j = (x_j, y_j):
//     S_r = e0 + sum_{j=1..3} Re[A_j W_R^(j r)] = e0 + sum_j (x_j cos(2 pi j r / R) + y_j sin(2 pi j r / R)),
// whose angles are compile-time constants: no per-element w^2, w^3, no table look-ups.  Half-turn symmetry
// (j r -> j (r + R/2) flips the sign of the odd j) and the quarter-turn symmetry of the j = 2 term give
//     S_r = P_r + Q_r,  S_(r+R/2) = P_r - Q_r,  P_r = e0 + T2_r,  P_(r+R/4) = e0 - T2_r,  Q_r = T1_r + T3_r,
// about 60 fp64 operations for the 16 values of a radix-16 butterfly instead of 16 * (6 + the per-element powers
// of w).  The values are produced four at a time (r, r+R/4, r+R/2, r+3R/4) so that no array of R values is live.
// ---------------------------------------------------------------------------
template <int N16>
__device__ __forceinline__ double rot_re(double x, double y) {      // x cos(2 pi n/16) + y sin(2 pi n/16)
    constexpr int n = ((N16 % 16) + 16) % 16;
    constexpr double H = 0.70710678118654752440, C1 = 0.92387953251128675613, S1 = 0.38268343236508977173;
    if constexpr (n == 0) return x;
    else if constexpr (n == 4) return y;
    else if constexpr (n == 8) return -x;
    else if constexpr (n == 12) return -y;
    else if constexpr (n == 2) return (x + y) * H;
    else if constexpr (n == 6) return (y - x) * H;
    else if constexpr (n == 10) return -((x + y) * H);
    else if constexpr (n == 14) return (x - y) * H;
    else {
        constexpr double c = (n == 1 || n == 15) ? C1 : (n == 3 || n == 13) ? S1 : (n == 5 || n == 11) ? -S1 : -C1;
        constexpr double sn = (n == 1 || n == 7) ? S1 : (n == 3 || n == 5) ? C1 : (n == 9 || n == 15) ? -S1 : -C1;
        return fma(x, c, y * sn);
    }
}
struct PsfSeqW { double2 w1, w2, w3; };      // w_jb, w_jb^2, w_jb^3
__device__ __forceinline__ PsfSeqW psf_seq_w(double2 w) {
    PsfSeqW p; p.w1 = w; p.w2 = cmul(w, w); p.w3 = cmul(p.w2, w);
    return p;
}
struct PsfSeqK { double e0, x[3], y[3]; };   // one kernel along one butterfly: e0 and A_j = (x_j, y_j)
// b = coefS[c][m] (b[0] = (e0, 0), b[j] = (e_j, f_j))
__device__ __forceinline__ PsfSeqK psf_seq_prep(const double2* __restrict__ b, const PsfSeqW& w) {
    PsfSeqK k;
    k.e0 = b[0].x;
    // (e - i f)(a + i b) = (e a + f b) + i (e b - f a)
    k.x[0] = fma(b[1].x, w.w1.x, b[1].y * w.w1.y); k.y[0] = fma(b[1].x, w.w1.y, -b[1].y * w.w1.x);
    k.x[1] = fma(b[2].x, w.w2.x, b[2].y * w.w2.y); k.y[1] = fma(b[2].x, w.w2.y, -b[2].y * w.w2.x);
    k.x[2] = fma(b[3].x, w.w3.x, b[3].y * w.w3.y); k.y[2] = fma(b[3].x, w.w3.y, -b[3].y * w.w3.x);
    return k;
}
// the four values S[i] at r + i*R/4, i = 0..3 (r < R/4): they share T2 and the two Q sums
template <int R, int r>
__device__ __forceinline__ void psf_seq_eval4(const PsfSeqK& k, double (&S)[4]) {
    static_assert(R == 4 || R == 8 || R == 16, "radix");
    static_assert(r >= 0 && r < R / 4, "r");
    constexpr int u = 16 / R, r1 = r + R / 4;
    const double T2 = rot_re<2 * r * u>(k.x[1], k.y[1]);
    const double P0 = k.e0 + T2, P1 = k.e0 - T2;
    const double Q0 = rot_re<1 * r * u>(k.x[0], k.y[0]) + rot_re<3 * r * u>(k.x[2], k.y[2]);
    const double Q1 = rot_re<1 * r1 * u>(k.x[0], k.y[0]) + rot_re<3 * r1 * u>(k.x[2], k.y[2]);
    S[0] = P0 + Q0; S[1] = P1 + Q1; S[2] = P0 - Q0; S[3] = P1 - Q1;
}
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f) {
    if constexpr (B < E) {
        f(std::integral_constant<int, B>{});
        static_for<B + 1, E>(f);
    }
}

// Full rows x cols spectrum for sbd_psf_spectrum (API / parity path only).
// coef was built with nk = nx.  Output column-major: element (k,q) at q*nx+k.
__global__ void k_psf_spectrum(int t, int nx, int ny, int m, const double2* __restrict__ coef,
                               const double2* __restrict__ tw_ny, double* __restrict__ re,
                               double* __restrict__ im) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)nx * ny) return;
    const int k = (int)(idx % nx), q = (int)(idx / nx);
    const double2* a = coef + ((size_t)m * nx + k) * MAXT;
    double sr = 0.0, si = 0.0;
    for (int j = 0; j < t; ++j) {
        const double2 w = tw_ny[(int)(((long long)q * j) % ny)];
        const double2 p = cmul(a[j], w);
        sr += p.x; si += p.y;
    }
    re[idx] = sr; im[idx] = si;
}

}  // namespace sbd
