// mt19937.cuh -- arithmetic of NumPy's legacy Gaussian draw, shared by the kernels of mt19937.cu
// and by its host hooks (so the CPU tests exercise the very code the device runs).
//
// RandomState(seed).normal(loc=0, scale, size=N) (numpy/random/src/legacy/legacy-distributions.c,
// legacy_gauss; the reference draws Theta with it, rla/embeddings.py:269,458) reads the MT19937 word
// stream w[0], w[1], ... in ATTEMPTS of four words:
//   x1 = 2 d(w0, w1) - 1,  x2 = 2 d(w2, w3) - 1,  d(a, b) = ((a >> 5) 2^26 + (b >> 6)) / 2^53   (exact)
//   r2 = fl(fl(x1 x1) + fl(x2 x2))   (no FMA), rejected when r2 >= 1 or r2 == 0
// and the p-th accepted attempt gives outputs 2p = 0 + scale (f x2), 2p + 1 = 0 + scale (f x1) with
// f = sqrt(-2 log(r2) / r2), log being the C library's.
//
// Every floating-point step below is an IEEE operation in round-to-nearest written as such
// (mul_rn / add_rn / ...): a contracted FMA in x1 x1 + x2 x2 would change which attempts are
// accepted and shift the whole stream.  mt19937.cu is also compiled with --fmad=false.
//
// The one step that is not IEEE-defined is log.  ext_log computes log(r2) as an unevaluated sum
// hi + lo with a relative error below 2^-66 (error <= 2^-13 ulp of the result, far inside the
// 2^-8 ulp the argument needs), and hi = fl(hi + lo) is its correctly rounded value unless the
// exact log lies next to a rounding midpoint.  near_midpoint() flags the pairs whose hi + lo lies
// within w ulp of a midpoint.  ASSUMPTION: the C library's log is within 0.519 ulp of the exact
// value (glibc >= 2.28 documents this bound for its log; its own test suite checks it).  Then for
// an unflagged pair with w = 2^-5 the exact value is at least 2^-5 - 2^-13 > 0.019 ulp away from
// any midpoint, every value within 0.519 ulp of it rounds to the same double, and libm's log
// returns hi.  Flagged pairs (about 2w of them) get libm's log from the host (mt19937.cu).
#pragma once
#include <math.h>
#include <stdint.h>

namespace rla {
namespace mt {

constexpr int N = 624;         // words of state
constexpr int M = 397;
constexpr int DEG = 19937;     // degree of the characteristic polynomial

__host__ __device__ __forceinline__ uint32_t twist(uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
    return c ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

__host__ __device__ __forceinline__ uint32_t temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// IEEE double operations, round to nearest, never contracted
__host__ __device__ __forceinline__ double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double add_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ double sub_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ __forceinline__ double div_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
__host__ __device__ __forceinline__ double sqrt_rn(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return sqrt(a);
#endif
}
__host__ __device__ __forceinline__ double fma_rn(double a, double b, double c) {
#ifdef __CUDA_ARCH__
    return __fma_rn(a, b, c);
#else
    return fma(a, b, c);
#endif
}

struct Attempt {
    double x1, x2, r2;
    bool accept;
};

// one attempt from its four (tempered) words
__host__ __device__ __forceinline__ Attempt attempt(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    const double d1 = div_rn(add_rn(mul_rn((double)(w0 >> 5), 67108864.0), (double)(w1 >> 6)), 9007199254740992.0);
    const double d2 = div_rn(add_rn(mul_rn((double)(w2 >> 5), 67108864.0), (double)(w3 >> 6)), 9007199254740992.0);
    Attempt a;
    a.x1 = sub_rn(mul_rn(2.0, d1), 1.0);
    a.x2 = sub_rn(mul_rn(2.0, d2), 1.0);
    a.r2 = add_rn(mul_rn(a.x1, a.x1), mul_rn(a.x2, a.x2));
    a.accept = a.r2 < 1.0 && a.r2 != 0.0;
    return a;
}

// ---- double-double arithmetic (Dekker / Knuth error-free transformations)
struct DD {
    double hi, lo;
};
__host__ __device__ __forceinline__ DD two_sum(double a, double b) {
    const double s = add_rn(a, b);
    const double bb = sub_rn(s, a);
    return DD{s, add_rn(sub_rn(a, sub_rn(s, bb)), sub_rn(b, bb))};
}
__host__ __device__ __forceinline__ DD quick_two_sum(double a, double b) {   // |a| >= |b|
    const double s = add_rn(a, b);
    return DD{s, sub_rn(b, sub_rn(s, a))};
}
__host__ __device__ __forceinline__ DD dd_add(DD a, DD b) {
    DD s = two_sum(a.hi, b.hi);
    const DD t = two_sum(a.lo, b.lo);
    s = quick_two_sum(s.hi, add_rn(s.lo, t.hi));
    return quick_two_sum(s.hi, add_rn(s.lo, t.lo));
}
__host__ __device__ __forceinline__ DD dd_mul(DD a, DD b) {
    const double p = mul_rn(a.hi, b.hi);
    const double e = fma_rn(a.hi, b.hi, -p);
    return quick_two_sum(p, add_rn(e, add_rn(mul_rn(a.hi, b.lo), mul_rn(a.lo, b.hi))));
}
__host__ __device__ __forceinline__ DD dd_mul_d(DD a, double b) {
    const double p = mul_rn(a.hi, b);
    const double e = fma_rn(a.hi, b, -p);
    return quick_two_sum(p, add_rn(e, mul_rn(a.lo, b)));
}

// log(x) for 0 < x < 1 (the r2 of an accepted attempt) as hi + lo, hi = fl(hi + lo).
// x = 2^e m with m in [sqrt(1/2), sqrt(2)); log m = 2 atanh(s), s = (m - 1) / (m + 1), |s| < 0.1716.
// m - 1 is exact (Sterbenz), so near x = 1 this is log1p(x - 1) with full relative accuracy.
// 2 atanh(s) = 2 s (1 + s^2/3 + s^4/5 + s^6 A), A = sum_{j>=3} s^(2j-6) / (2j+1) in plain double
// (its rounding error, weighted by s^6 < 2^-15, and the truncation after j = 13, below (0.0295)^14,
// stay under 2^-66 relative); the rest in double-double (about 2^-100).  x >= 2^-104 for every r2,
// so there are no subnormals.
__host__ __device__ __forceinline__ DD ext_log(double x) {
    int e;
    double m = frexp(x, &e);                                   // x = m 2^e, m in [0.5, 1)
    if (m < 0.70710678118654757) {
        m = mul_rn(m, 2.0);
        e -= 1;
    }
    const double num = sub_rn(m, 1.0);
    const DD den = two_sum(m, 1.0);
    const double sh = div_rn(num, den.hi);
    const double r = sub_rn(fma_rn(-sh, den.hi, num), mul_rn(sh, den.lo));
    const DD s = quick_two_sum(sh, div_rn(r, den.hi));
    const DD s2 = dd_mul(s, s);
    double a = 1.0 / 27.0;
    a = fma_rn(a, s2.hi, 1.0 / 25.0);
    a = fma_rn(a, s2.hi, 1.0 / 23.0);
    a = fma_rn(a, s2.hi, 1.0 / 21.0);
    a = fma_rn(a, s2.hi, 1.0 / 19.0);
    a = fma_rn(a, s2.hi, 1.0 / 17.0);
    a = fma_rn(a, s2.hi, 1.0 / 15.0);
    a = fma_rn(a, s2.hi, 1.0 / 13.0);
    a = fma_rn(a, s2.hi, 1.0 / 11.0);
    a = fma_rn(a, s2.hi, 1.0 / 9.0);
    a = fma_rn(a, s2.hi, 1.0 / 7.0);
    DD b = dd_add(DD{0.2, -1.1102230246251566e-17}, dd_mul_d(s2, a));               // 1/5 + s^2 A
    b = dd_add(DD{0.3333333333333333, 1.850371707708594e-17}, dd_mul(s2, b));       // 1/3 + ...
    b = dd_add(DD{1.0, 0.0}, dd_mul(s2, b));                                          // 1 + ...
    DD lm = dd_mul(s, b);
    lm.hi = mul_rn(lm.hi, 2.0);
    lm.lo = mul_rn(lm.lo, 2.0);
    if (e == 0) return lm;
    return dd_add(dd_mul_d(DD{0.6931471805599453, 2.3190468138462996e-17}, (double)e), lm);
}

// true when hi + lo lies within w ulp of a rounding midpoint of hi (the ulp on lo's side)
__host__ __device__ __forceinline__ bool near_midpoint(DD v, double w) {
    const double nb = nextafter(v.hi, v.lo > 0.0 ? HUGE_VAL : -HUGE_VAL);   // (double, double): the device overload
    const double gap = fabs(sub_rn(nb, v.hi));
    return fabs(v.lo) >= mul_rn(0.5 - w, gap);
}

// f = sqrt(-2 log(r2) / r2) and the output 0 + scale (f x), as legacy_gauss / legacy_normal
__host__ __device__ __forceinline__ double gauss_f(double log_r2, double r2) {
    return sqrt_rn(div_rn(mul_rn(-2.0, log_r2), r2));
}
__host__ __device__ __forceinline__ double gauss_out(double scale, double f, double x) {
    return add_rn(0.0, mul_rn(scale, mul_rn(f, x)));
}

}  // namespace mt
}  // namespace rla
