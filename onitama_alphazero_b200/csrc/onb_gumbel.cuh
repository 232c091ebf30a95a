// onb_gumbel.cuh -- the arithmetic of the Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f), shared by the kernels
// (onb_mcts.cu) and the CPU oracle (tests/gumbel_oracle.cpp includes this file and compiles it with g++ -ffp-contract=off).
//
// onb_log / onb_exp are built from IEEE basic operations only (+ - * /, a double -> int truncation, exponent and significand bit
// manipulation) with no FMA contraction: __dadd_rn / __dmul_rn / __ddiv_rn on the device, plain operators on the host. They
// therefore give the same bits on the CPU and on the GPU, which CUDA's and libm's log / exp do not. They restate fdlibm's
// __ieee754_log and __ieee754_exp (Sun Microsystems, freely distributable), accurate to about 1 ulp.
#pragma once
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define ONB_GHD __host__ __device__ __forceinline__
#else
#define ONB_GHD inline
#endif

namespace onb_gumbel {

#if defined(__CUDA_ARCH__)
ONB_GHD double g_add(double a, double b) { return __dadd_rn(a, b); }
ONB_GHD double g_sub(double a, double b) { return __dsub_rn(a, b); }
ONB_GHD double g_mul(double a, double b) { return __dmul_rn(a, b); }
ONB_GHD double g_div(double a, double b) { return __ddiv_rn(a, b); }
ONB_GHD uint64_t g_bits(double x) { return (uint64_t)__double_as_longlong(x); }
ONB_GHD double g_from(uint64_t b) { return __longlong_as_double((long long)b); }
#else
ONB_GHD double g_add(double a, double b) { return a + b; }
ONB_GHD double g_sub(double a, double b) { return a - b; }
ONB_GHD double g_mul(double a, double b) { return a * b; }
ONB_GHD double g_div(double a, double b) { return a / b; }
ONB_GHD uint64_t g_bits(double x) { uint64_t b; memcpy(&b, &x, 8); return b; }
ONB_GHD double g_from(uint64_t b) { double x; memcpy(&x, &b, 8); return x; }
#endif
ONB_GHD uint32_t g_hi(double x) { return (uint32_t)(g_bits(x) >> 32); }
ONB_GHD uint32_t g_lo(double x) { return (uint32_t)g_bits(x); }
ONB_GHD double g_with_hi(double x, uint32_t hi) { return g_from(((uint64_t)hi << 32) | g_lo(x)); }
ONB_GHD double g_inf() { return g_from(0x7FF0000000000000ull); }

// natural logarithm; x = 0 -> -inf, x < 0 -> NaN
ONB_GHD double onb_log(double x) {
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, two54 = 1.80143985094819840000e+16;
    const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                 Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                 Lg7 = 1.479819860511658591e-01;
    int32_t hx = (int32_t)g_hi(x);
    const uint32_t lx = g_lo(x);
    int32_t k = 0;
    if (hx < 0x00100000) {  // x < 2^-1022
        if (((hx & 0x7fffffff) | (int32_t)lx) == 0) return -g_inf();
        if (hx < 0) return g_from(0x7FF8000000000000ull);
        k -= 54;
        x = g_mul(x, two54);  // subnormal: scale up
        hx = (int32_t)g_hi(x);
    }
    if (hx >= 0x7ff00000) return g_add(x, x);
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    const int32_t i0 = (hx + 0x95f64) & 0x100000;
    x = g_with_hi(x, (uint32_t)(hx | (i0 ^ 0x3ff00000)));  // normalise x or x / 2 into [sqrt(2)/2, sqrt(2))
    k += (i0 >> 20);
    const double f = g_sub(x, 1.0);
    const double dk = (double)k;
    if ((0x000fffff & (2 + hx)) < 3) {  // |f| < 2^-20
        if (f == 0.0) return k == 0 ? 0.0 : g_add(g_mul(dk, ln2_hi), g_mul(dk, ln2_lo));
        const double R = g_mul(g_mul(f, f), g_sub(0.5, g_mul(0.33333333333333333, f)));
        if (k == 0) return g_sub(f, R);
        return g_sub(g_mul(dk, ln2_hi), g_sub(g_sub(R, g_mul(dk, ln2_lo)), f));
    }
    const double s = g_div(f, g_add(2.0, f));
    const double z = g_mul(s, s);
    int32_t i = hx - 0x6147a;
    const double w = g_mul(z, z);
    const int32_t j = 0x6b851 - hx;
    const double t1 = g_mul(w, g_add(Lg2, g_mul(w, g_add(Lg4, g_mul(w, Lg6)))));
    const double t2 = g_mul(z, g_add(Lg1, g_mul(w, g_add(Lg3, g_mul(w, g_add(Lg5, g_mul(w, Lg7)))))));
    i |= j;
    const double R = g_add(t2, t1);
    if (i > 0) {
        const double hfsq = g_mul(g_mul(0.5, f), f);
        if (k == 0) return g_sub(f, g_sub(hfsq, g_mul(s, g_add(hfsq, R))));
        return g_sub(g_mul(dk, ln2_hi), g_sub(g_sub(hfsq, g_add(g_mul(s, g_add(hfsq, R)), g_mul(dk, ln2_lo))), f));
    }
    if (k == 0) return g_sub(f, g_mul(s, g_sub(f, R)));
    return g_sub(g_mul(dk, ln2_hi), g_sub(g_sub(g_mul(s, g_sub(f, R)), g_mul(dk, ln2_lo)), f));
}

// e^x; -inf -> 0, +inf -> inf
ONB_GHD double onb_exp(double x) {
    const double o_threshold = 7.09782712893383973096e+02, u_threshold = -7.45133219101941108420e+02;
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, invln2 = 1.44269504088896338700e+00;
    const double twom1000 = 9.33263618503218878990e-302;
    const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
                 P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
    uint32_t hx = g_hi(x);
    const int32_t xsb = (int32_t)((hx >> 31) & 1u);
    hx &= 0x7fffffffu;
    if (hx >= 0x40862E42u) {  // |x| >= 709.78...
        if (hx >= 0x7ff00000u) {
            if (((hx & 0xfffffu) | g_lo(x)) != 0) return g_add(x, x);  // NaN
            return xsb == 0 ? x : 0.0;
        }
        if (x > o_threshold) return g_inf();
        if (x < u_threshold) return 0.0;
    }
    double hi = 0.0, lo = 0.0;
    int32_t k = 0;
    if (hx > 0x3fd62e42u) {  // |x| > 0.5 ln2
        if (hx < 0x3FF0A2B2u) {  // and |x| < 1.5 ln2
            hi = xsb ? g_add(x, ln2_hi) : g_sub(x, ln2_hi);
            lo = xsb ? -ln2_lo : ln2_lo;
            k = 1 - xsb - xsb;
        } else {
            k = (int32_t)g_add(g_mul(invln2, x), xsb ? -0.5 : 0.5);  // truncation towards zero
            const double t = (double)k;
            hi = g_sub(x, g_mul(t, ln2_hi));  // t * ln2_hi is exact here
            lo = g_mul(t, ln2_lo);
        }
        x = g_sub(hi, lo);
    } else if (hx < 0x3e300000u) {  // |x| < 2^-28
        return g_add(1.0, x);
    }
    const double t = g_mul(x, x);
    const double c = g_sub(x, g_mul(t, g_add(P1, g_mul(t, g_add(P2, g_mul(t, g_add(P3, g_mul(t, g_add(P4, g_mul(t, P5))))))))));
    if (k == 0) return g_sub(1.0, g_sub(g_div(g_mul(x, c), g_sub(c, 2.0)), x));
    const double y = g_sub(1.0, g_sub(g_sub(lo, g_div(g_mul(x, c), g_sub(2.0, c))), hi));
    if (k >= -1021) return g_with_hi(y, g_hi(y) + ((uint32_t)k << 20));
    return g_mul(g_with_hi(y, g_hi(y) + ((uint32_t)(k + 1000) << 20)), twom1000);
}

// Gumbel draw from one counter-RNG word r (draw 0x10000 + child index): scale * (-log(-log(u))), u = (r + 0.5) 2^-32 in (0, 1)
constexpr uint32_t kGumbelDraw = 0x10000u;
ONB_GHD double gumbel_of(uint32_t r, double scale) {
    const double u = g_mul(g_add((double)r, 0.5), 2.3283064365386962890625e-10);
    return g_mul(scale, -onb_log(-onb_log(u)));
}
// prior logit: log P, -inf for P = 0
ONB_GHD double logit_of(double p) { return p > 0.0 ? onb_log(p) : -g_inf(); }
// the score floor of the root selection: max(-1e9, s)
ONB_GHD double score_floor(double s) { return s > -1e9 ? s : -1e9; }

// Sequential halving: the visit count a considered action has at each of the n descents of a search with m considered actions
// (mctx's get_sequence_of_considered_visits). out[0 .. n).
inline void seq_halving(uint32_t m, uint32_t n, uint32_t* out) {
    if (m <= 1) {
        for (uint32_t i = 0; i < n; ++i) out[i] = i;
        return;
    }
    uint32_t log2max = 0;
    while ((1u << log2max) < m) ++log2max;
    uint32_t visits[64] = {0};
    uint32_t c = m, len = 0;
    while (len < n) {
        uint32_t e = n / (log2max * c);
        if (e < 1) e = 1;
        for (uint32_t r = 0; r < e && len < n; ++r) {
            for (uint32_t a = 0; a < c && len < n; ++a) out[len++] = visits[a];
            for (uint32_t a = 0; a < c; ++a) visits[a] += 1;
        }
        c = c / 2 > 2 ? c / 2 : 2;
    }
}

}  // namespace onb_gumbel
