// glibc_log.cuh — glibc's double-precision log(), reproduced operation by operation.
//
// Why: the reference's hyperscore is `(Σb+1)(Σy+1).ln() + lnfact(nb) + lnfact(ny)` with Rust's f64::ln (scoring.rs:179-201), and f64::ln
// is the platform libm's log(). Candidates are ranked by a stable sort on that f64 (scoring.rs:495), so two candidates whose products differ
// by one ulp are ordered by the last bit of log(). CUDA's log() is a different (<= 1 ulp) function; to keep ranks — and the reported
// hyperscore / poisson — bit-identical to the CPU path, the kernels evaluate the same algorithm glibc >= 2.28 uses (Szabolcs Nagy's log from
// ARM optimized-routines: sysdeps/ieee754/dbl-64/e_log.c; musl ships the same code) with the same tables (glibc_log_data.cuh, generated from
// libm.so.6 by tools/gen_glibc_log_table.py) and the same rounding sequence:
//
//   variant 0  "fma":   what x86-64 glibc's ifunc picks on every CPU with FMA + AVX2 (`__log_fma`): e_log.c compiled with -mfma -mavx2, where
//                       gcc contracts a*b+c into fused multiply-adds. The fusion pattern below is transcribed from the disassembly of
//                       Ubuntu GLIBC 2.39's __log_fma (libm.so.6 + 0x79d50) and noted next to each operation.
//   variant 1  "nofma": e_log.c as written (no contraction, r from the chi/clo table): `__log_sse2` / `__log_avx`, aarch64 without
//                       -ffp-contract, musl.
//
// The host side (sage_b200.cu: probe_host_log) evaluates both variants on the CPU, compares them with the host libm's log() on a few
// thousand inputs and selects the one that matches bit for bit, so the device follows whatever libm the caller's Rust binary would use.
// tests/test_glibc_log.py checks the host evaluation against libm on 10^7 inputs (CPU) and the device evaluation against libm (GPU).
#pragma once
#include <stdint.h>
#include <string.h>

#include "glibc_log_data.cuh"

#if defined(__CUDACC__)
#define SB_HD __host__ __device__ __forceinline__
#else
#define SB_HD inline
#endif

namespace sb { namespace glog {

#if defined(__CUDA_ARCH__)
SB_HD double g_fma(double a, double b, double c) { return __fma_rn(a, b, c); }
SB_HD double g_add(double a, double b) { return __dadd_rn(a, b); }
SB_HD double g_sub(double a, double b) { return __dsub_rn(a, b); }
SB_HD double g_mul(double a, double b) { return __dmul_rn(a, b); }
SB_HD uint64_t g_bits(double x) { return (uint64_t)__double_as_longlong(x); }
SB_HD double g_dbl(uint64_t u) { return __longlong_as_double((long long)u); }
SB_HD double g_tab(int i) { return TAB[i]; }
SB_HD double g_tab2(int i) { return TAB2[i]; }
#else
}}  // close namespaces around the host-only includes
#include <cmath>
namespace sb { namespace glog {
// volatile temporaries: the host compiler must not contract or re-associate these either
SB_HD double g_fma(double a, double b, double c) { return std::fma(a, b, c); }
SB_HD double g_add(double a, double b) { volatile double r = a + b; return r; }
SB_HD double g_sub(double a, double b) { volatile double r = a - b; return r; }
SB_HD double g_mul(double a, double b) { volatile double r = a * b; return r; }
SB_HD uint64_t g_bits(double x) { uint64_t u; memcpy(&u, &x, 8); return u; }
SB_HD double g_dbl(uint64_t u) { double x; memcpy(&x, &u, 8); return x; }
SB_HD double g_tab(int i) { return H_TAB[i]; }
SB_HD double g_tab2(int i) { return H_TAB2[i]; }
#endif

// log(x) exactly as glibc computes it. FMA == true: variant 0, false: variant 1.
template <bool FMA>
SB_HD double glibc_log(double x) {
    uint64_t ix = g_bits(x);
    const uint32_t top = (uint32_t)(ix >> 48);
    constexpr uint64_t LO = 0x3fee000000000000ull;   // asuint64(1.0 - 0x1p-4)
    constexpr uint64_t HI = 0x3ff1090000000000ull;   // asuint64(1.0 + 0x1.09p-4)
    if (ix - LO < HI - LO) {
        // x close to 1: log(1+r) = r - r^2/2 + r^3 * poly1(r), with r - r^2/2 evaluated in two pieces
        if (ix == 0x3ff0000000000000ull) return 0.0;
        const double r = g_sub(x, 1.0);
        const double r2 = g_mul(r, r);
        const double r3 = g_mul(r, r2);
        double y, hi, lo;
        if (FMA) {
            const double t1 = g_fma(r, B2, B1);            // B1 + r*B2
            const double t2 = g_fma(r, B5, B4);            // B4 + r*B5
            const double t3 = g_fma(r, B8, B7);            // B7 + r*B8
            const double u1 = g_fma(r2, B3, t1);           // + r2*B3
            const double u2 = g_fma(r2, B6, t2);           // + r2*B6
            const double u3 = g_fma(r2, B9, t3);           // + r2*B9
            const double v3 = g_fma(r3, B10, u3);          // + r3*B10
            const double v2 = g_fma(v3, r3, u2);
            const double v1 = g_fma(v2, r3, u1);           // B1 + r*B2 + r2*B3 + r3*(...)
            const double a = g_fma(r, 0x1p27, r);          // r + w, w = r * 2^27 (fused)
            const double rhi = g_fma(-0x1p27, r, a);       // r + w - w (fused: -(2^27 * r) + a)
            const double rlo = g_sub(r, rhi);
            const double rr = g_mul(rhi, rhi);
            hi = g_fma(rr, B0, r);                         // hi = r + rhi*rhi*B0
            const double d = g_sub(r, hi);
            const double s = g_add(r, rhi);
            lo = g_fma(rr, B0, d);                         // lo = r - hi + rhi*rhi*B0
            lo = g_fma(g_mul(B0, rlo), s, lo);             // lo += B0*rlo*(rhi + r)
            y = g_fma(v1, r3, lo);                         // y = r3*poly + lo
        } else {
            // y = r3 * (B[1] + r*B[2] + r2*B[3] + r3*(B[4] + r*B[5] + r2*B[6] + r3*(B[7] + r*B[8] + r2*B[9] + r3*B[10])))
            const double p3 = g_add(g_add(g_add(B7, g_mul(r, B8)), g_mul(r2, B9)), g_mul(r3, B10));
            const double p2 = g_add(g_add(g_add(B4, g_mul(r, B5)), g_mul(r2, B6)), g_mul(r3, p3));
            const double p1 = g_add(g_add(g_add(B1, g_mul(r, B2)), g_mul(r2, B3)), g_mul(r3, p2));
            y = g_mul(r3, p1);
            double w = g_mul(r, 0x1p27);
            const double rhi = g_sub(g_add(r, w), w);
            const double rlo = g_sub(r, rhi);
            w = g_mul(g_mul(rhi, rhi), B0);
            hi = g_add(r, w);
            lo = g_add(g_sub(r, hi), w);
            lo = g_add(lo, g_mul(g_mul(B0, rlo), g_add(rhi, r)));
            y = g_add(y, lo);
        }
        return g_add(y, hi);
    }
    if (top - 0x0010u >= 0x7ff0u - 0x0010u) {
        // x < 0x1p-1022 or inf or nan
        if (ix * 2 == 0) return g_dbl(0xfff0000000000000ull);                // log(+-0) = -inf
        if (ix == 0x7ff0000000000000ull) return x;                            // log(inf) = inf
        if ((top & 0x8000u) || (top & 0x7ff0u) == 0x7ff0u) return g_dbl(0x7ff8000000000000ull) ;  // x < 0 or nan -> nan (payload/sign not reproduced)
        ix = g_bits(g_mul(x, 0x1p52));                                        // subnormal: normalise
        ix -= 52ull << 52;
    }
    // x = 2^k z, z in [OFF, 2*OFF): log(x) = log1p(z/c - 1) + log(c) + k*Ln2
    constexpr uint64_t OFF = 0x3fe6000000000000ull;
    const uint64_t tmp = ix - OFF;
    const int i = (int)((tmp >> (52 - 7)) & 127);
    const int k = (int)((int64_t)tmp >> 52);
    const uint64_t iz = ix - (tmp & (0xfffull << 52));
    const double invc = g_tab(2 * i), logc = g_tab(2 * i + 1);
    const double z = g_dbl(iz);
    const double kd = (double)k;
    if (FMA) {
        const double r = g_fma(z, invc, -1.0);
        const double w = g_fma(kd, LN2HI, logc);           // kd*Ln2hi + logc (fused)
        const double hi = g_add(r, w);
        const double lo = g_fma(kd, LN2LO, g_add(g_sub(w, hi), r));   // w - hi + r + kd*Ln2lo (last product fused)
        const double r2 = g_mul(r, r);
        const double p1 = g_fma(r, A2, A1);                // A1 + r*A2
        const double p2 = g_fma(r, A4, A3);                // A3 + r*A4
        const double q = g_fma(r2, A0, lo);                // lo + r2*A0
        const double p = g_fma(p2, r2, p1);                // A1 + r*A2 + r2*(A3 + r*A4)
        const double y = g_fma(g_mul(r, r2), p, q);        // lo + r2*A0 + r*r2*p
        return g_add(y, hi);
    } else {
        const double r = g_mul(g_sub(g_sub(z, g_tab2(2 * i)), g_tab2(2 * i + 1)), invc);
        const double w = g_add(g_mul(kd, LN2HI), logc);
        const double hi = g_add(w, r);
        const double lo = g_add(g_add(g_sub(w, hi), r), g_mul(kd, LN2LO));
        const double r2 = g_mul(r, r);
        // y = lo + r2*A[0] + r*r2*(A[1] + r*A[2] + r2*(A[3] + r*A[4])) + hi
        const double inner = g_add(g_add(A1, g_mul(r, A2)), g_mul(r2, g_add(A3, g_mul(r, A4))));
        const double y = g_add(g_add(lo, g_mul(r2, A0)), g_mul(g_mul(r, r2), inner));
        return g_add(y, hi);
    }
}

// ---------------------------------------------------------------------------------------------------------------------------------------
// log1pf(x) exactly as glibc computes it (sysdeps/ieee754/flt-32/s_log1pf.c, the fdlibm algorithm; x86-64 glibc ships ONE build of it, plain
// SSE arithmetic without contraction — checked against the disassembly of Ubuntu GLIBC 2.39's __log1pf). Rust's f32::ln_1p, which the reference's
// OpenMS hyperscore uses (scoring.rs:190-197), is this function. tests/test_glibc_log.py compares the host evaluation below with libm's
// log1pf on EVERY float (2^32 inputs), and the device evaluation on a sample.
#if defined(__CUDA_ARCH__)
SB_HD float gf_add(float a, float b) { return __fadd_rn(a, b); }
SB_HD float gf_sub(float a, float b) { return __fsub_rn(a, b); }
SB_HD float gf_mul(float a, float b) { return __fmul_rn(a, b); }
SB_HD float gf_div(float a, float b) { return __fdiv_rn(a, b); }
SB_HD int32_t gf_bits(float x) { return __float_as_int(x); }
SB_HD float gf_flt(int32_t u) { return __int_as_float(u); }
#else
SB_HD float gf_add(float a, float b) { volatile float r = a + b; return r; }
SB_HD float gf_sub(float a, float b) { volatile float r = a - b; return r; }
SB_HD float gf_mul(float a, float b) { volatile float r = a * b; return r; }
SB_HD float gf_div(float a, float b) { volatile float r = a / b; return r; }
SB_HD int32_t gf_bits(float x) { int32_t u; memcpy(&u, &x, 4); return u; }
SB_HD float gf_flt(int32_t u) { float x; memcpy(&x, &u, 4); return x; }
#endif

SB_HD float glibc_log1pf(float x) {
    const float ln2_hi = gf_flt(0x3f317180), ln2_lo = gf_flt(0x3717f7d1);
    const float Lp1 = gf_flt(0x3f2aaaab), Lp2 = gf_flt(0x3ecccccd), Lp3 = gf_flt(0x3e924925), Lp4 = gf_flt(0x3e638e29), Lp5 = gf_flt(0x3e3a3325),
                Lp6 = gf_flt(0x3e1cd04f), Lp7 = gf_flt(0x3e178897);
    const int32_t hx = gf_bits(x), ax = hx & 0x7fffffff;
    int32_t k = 1, hu = 0;
    float f = 0.0f, c = 0.0f, u;
    if (hx < 0x3ed413d7) {                       // x < 0.41422
        if (ax >= 0x3f800000) {                  // x <= -1.0, or a negative NaN
            if (x == -1.0f) return gf_flt((int32_t)0xff800000);   // log1p(-1) = -inf
            // (x - x) / (x - x) on x86-64 SSE: a NaN x comes back quieted, sign and payload kept; else the default NaN 0xffc00000
            return gf_flt(ax > 0x7f800000 ? (hx | 0x00400000) : (int32_t)0xffc00000);
        }
        if (ax < 0x31000000) {                   // |x| < 2^-29
            if (ax < 0x24800000) return x;       // |x| < 2^-54
            return gf_sub(x, gf_mul(gf_mul(x, x), 0.5f));
        }
        if (hx > 0 || hx <= (int32_t)0xbe95f61f) { k = 0; f = x; hu = 1; }   // -0.2929 < x < 0.41422
    }
    // x + x: +inf, or a NaN x quieted as the host leaves it (the device's own add would give its canonical 0x7fffffff)
    if (hx >= 0x7f800000) return gf_flt(ax > 0x7f800000 ? (hx | 0x00400000) : hx);
    if (k != 0) {
        if (hx < 0x5a000000) {
            u = gf_add(1.0f, x);
            hu = gf_bits(u);
            k = (hu >> 23) - 127;
            c = k > 0 ? gf_sub(1.0f, gf_sub(u, x)) : gf_sub(x, gf_sub(u, 1.0f));   // correction term
            c = gf_div(c, u);
        } else {
            u = x;
            hu = gf_bits(u);
            k = (hu >> 23) - 127;
            c = 0.0f;
        }
        hu &= 0x007fffff;
        if (hu < 0x3504f7) {
            u = gf_flt(hu | 0x3f800000);         // normalize u
        } else {
            k += 1;
            u = gf_flt(hu | 0x3f000000);         // normalize u / 2
            hu = (0x00800000 - hu) >> 2;
        }
        f = gf_sub(u, 1.0f);
    }
    const float hfsq = gf_mul(gf_mul(0.5f, f), f);
    const float kf = (float)k;
    if (hu == 0) {                               // |f| < 2^-20
        if (f == 0.0f) {
            if (k == 0) return 0.0f;
            c = gf_add(c, gf_mul(kf, ln2_lo));
            return gf_add(gf_mul(kf, ln2_hi), c);
        }
        const float R = gf_mul(hfsq, gf_sub(1.0f, gf_mul(Lp1, f)));   // (float)0.66666666666666666 == Lp1
        if (k == 0) return gf_sub(f, R);
        return gf_sub(gf_mul(kf, ln2_hi), gf_sub(gf_sub(R, gf_add(gf_mul(kf, ln2_lo), c)), f));
    }
    const float s = gf_div(f, gf_add(2.0f, f));
    const float z = gf_mul(s, s);
    float R = gf_mul(z, Lp7);
    R = gf_mul(z, gf_add(Lp6, R));
    R = gf_mul(z, gf_add(Lp5, R));
    R = gf_mul(z, gf_add(Lp4, R));
    R = gf_mul(z, gf_add(Lp3, R));
    R = gf_mul(z, gf_add(Lp2, R));
    R = gf_mul(z, gf_add(Lp1, R));
    if (k == 0) return gf_sub(f, gf_sub(hfsq, gf_mul(s, gf_add(hfsq, R))));
    return gf_sub(gf_mul(kf, ln2_hi), gf_sub(gf_sub(hfsq, gf_add(gf_mul(s, gf_add(hfsq, R)), gf_add(gf_mul(kf, ln2_lo), c))), f));
}

SB_HD double glibc_log_v(double x, int variant) { return variant == 1 ? glibc_log<false>(x) : glibc_log<true>(x); }

}}  // namespace sb::glog
