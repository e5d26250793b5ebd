// fft_plan.h - which image sizes the FFT operators take, and the radix plan of the mixed-radix path (fft_any.cuh).
// Plain C++ (no CUDA): sbd_create classifies a size with it before it looks for a device, and the CPU tests compile it
// on its own.
//
//   pow2   : rows and cols powers of two in [16, 4096]                                  -> fft.cuh / fft2.cuh
//   smooth : every other size with both sides in [2, 4096] and no prime factor above 7  -> fft_any.cuh
//   else   : the FFT operators return SBD_E_UNSUPPORTED with the message of fft_size_error
#pragma once
#include <algorithm>
#include <string>

namespace sbd {

constexpr int ANY_MAXN = 4096;
constexpr int ANY_MAXST = 8;        // 3^7 = 2187 is the longest plan (7 stages)

// Stockham plan of one length: radices in stage order and the threads per line.  A thread owns at most 16 / R
// butterflies of a radix-R stage (<= 16 complex values), so T >= (n / R) / (16 / R) for every stage.
struct AnyPlan {
    int n, nst, T;
    int r[ANY_MAXST];
};

inline bool any_plan(int n, AnyPlan* p) {
    if (n < 2 || n > ANY_MAXN) return false;
    AnyPlan q = {};
    q.n = n;
    int m = n, twos = 0;
    while (m % 2 == 0) { m /= 2; ++twos; }
    while (twos >= 3) { q.r[q.nst++] = 8; twos -= 3; }
    if (twos) q.r[q.nst++] = 1 << twos;
    for (int f : {3, 5, 7})
        while (m % f == 0) { m /= f; q.r[q.nst++] = f; }
    if (m != 1) return false;
    int T = 32;
    for (int s = 0; s < q.nst; ++s) {
        const int R = q.r[s], mb = 16 / R, nb = n / R;
        T = std::max(T, (nb + mb - 1) / mb);
    }
    q.T = (T + 31) / 32 * 32;
    *p = q;
    return true;
}

// "481 = 13·37"
inline std::string factorization(int n) {
    std::string f;
    int m = n;
    for (int d = 2; d * d <= m; ++d)
        while (m % d == 0) { f += (f.empty() ? "" : "\xC2\xB7") + std::to_string(d); m /= d; }
    if (m > 1) f += (f.empty() ? "" : "\xC2\xB7") + std::to_string(m);
    return std::to_string(n) + " = " + f;
}

// "" when the FFT operators support rows x cols, otherwise the reason, naming the side at fault
inline std::string fft_size_error(int rows, int cols) {
    const char* names[2] = {"rows", "cols"};
    const int sides[2] = {rows, cols};
    for (int i = 0; i < 2; ++i) {
        AnyPlan p;
        if (sides[i] > ANY_MAXN)
            return std::string(names[i]) + " = " + factorization(sides[i]) + ": FFT lengths must be at most 4096";
        if (!any_plan(sides[i], &p))
            return std::string(names[i]) + " = " + factorization(sides[i]) + ": FFT lengths need prime factors \xE2\x89\xA4 7";
    }
    return "";
}

}  // namespace sbd
