// Goldilocks base field Fp, p = 2^64 - 2^32 + 1 (reference README.md:4; `cheetah::Fp`, call sites
// src/signature.rs:278-298).  Elements are canonical u64 values (the reference's raw limbs are
// canonical, not Montgomery -- SURVEY.md App. A).
//
// Device code is written on 32-bit halves: every 32x32->64 product is one IMAD.WIDE on the
// integer-multiply pipe.  The special-form reduction (2^64 = 2^32-1, 2^96 = -1 mod p) folds x2 (2^32-1)
// in ONE multiply-add (IMAD.WIDE with carry-out) and applies the two wrap corrections together: 13.75
// against 13.10 M/s with an add/subtract fold (profiles/r2_variants.md, v15).
// Sums of 64x64 products are kept in a lazy accumulator
// made of an "even" part E (words at bit 0,32,64,96,128: lo*lo and hi*hi products, one carry chain)
// and an "odd" part O (words at bit 32,64,96: the two cross products).  A 64x64 product therefore
// costs 4 IMAD.WIDE + 3 carry adds, and a whole dot product is reduced once.
//
// The same header compiles on the host (g++) with portable fallbacks for the PTX blocks; that
// build is used ONLY by tests/hostsim to unit-test the formulas without a GPU.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SB_DEV __device__ __forceinline__
#define SB_DEV_NOINLINE __device__ __noinline__
#else
#define SB_DEV static inline __attribute__((always_inline))
#define SB_DEV_NOINLINE static __attribute__((noinline))
#endif

namespace sb {

// TEST-ONLY (tests/hostsim): count the 32x32->64 multiplies an algorithm executes, for the cost figures in DESIGN.md
#if !defined(__CUDA_ARCH__) && defined(SB_COUNT_WIDE)
static unsigned long long g_wide_count = 0;
#define SB_WIDE(n) (g_wide_count += (n))
#else
#define SB_WIDE(n) ((void)0)
#endif

typedef uint64_t fp_t;
static constexpr uint64_t FP_P = 0xffffffff00000001ULL;
static constexpr uint64_t FP_EPS = 0xffffffffULL;  // 2^64 mod p

// a - b for a canonical and b <= p: one borrow chain, then "borrowed 2^64 == EPS too much" is undone
// with the borrow mask (5 instructions, no compare/select).
SB_DEV fp_t fp_sub(fp_t a, fp_t b) {
#if defined(__CUDA_ARCH__)
    uint32_t a0 = (uint32_t)a, a1 = (uint32_t)(a >> 32), b0 = (uint32_t)b, b1 = (uint32_t)(b >> 32), d0, d1;
    asm("{\n\t"
        ".reg .u32 m;\n\t"
        "sub.cc.u32 %0, %2, %4;\n\t"
        "subc.cc.u32 %1, %3, %5;\n\t"
        "subc.u32 m, 0, 0;\n\t"
        "sub.cc.u32 %0, %0, m;\n\t"
        "subc.u32 %1, %1, 0;\n\t"
        "}"
        : "=&r"(d0), "=&r"(d1)
        : "r"(a0), "r"(a1), "r"(b0), "r"(b1));
    return ((uint64_t)d1 << 32) | d0;
#else
    uint64_t d = a - b;
    return (a < b) ? d - FP_EPS : d;  // d + p == d - (2^32 - 1) (mod 2^64)
#endif
}
// a + b = a - (p - b); p - b is in [1, p] and fp_sub accepts a subtrahend equal to p
SB_DEV fp_t fp_add(fp_t a, fp_t b) { return fp_sub(a, FP_P - b); }
SB_DEV fp_t fp_neg(fp_t a) { return a ? FP_P - a : 0; }
SB_DEV fp_t fp_dbl(fp_t a) { return fp_add(a, a); }

// x = x0 + x1*2^32 + x2*2^64 (x2 < 2^32)  ->  x mod p as ANY 64-bit representative ("nc": may be >= p):
//   x = (x1:x0) + x2*(2^32-1)
// Every consumer that only multiplies (wide_mac, fp_mul_nc, ...) or uses the value as the MINUEND of fp_sub accepts
// this form; the canonicalisation below costs 4 more instructions and is only paid where a value is compared,
// stored, negated (p - x) or subtracted.
SB_DEV fp_t fp_reduce96_nc(uint32_t x0, uint32_t x1, uint32_t x2) {
#if defined(__CUDA_ARCH__)
    uint32_t t0, t1;
    asm("{\n\t"
        ".reg .u32 c;\n\t"
        "mad.lo.cc.u32 %0, %4, 0xffffffff, %2;\n\t"   // (x1:x0) + x2 * (2^32 - 1)
        "madc.hi.cc.u32 %1, %4, 0xffffffff, %3;\n\t"
        "addc.u32 c, 0, 0;\n\t"                       // wrapped 2^64 == EPS: + c EPS = - (0 : c) + (c : 0)
        "sub.cc.u32 %0, %0, c;\n\t"
        "subc.u32 %1, %1, 0;\n\t"
        "add.u32 %1, %1, c;\n\t"
        "}"
        : "=&r"(t0), "=&r"(t1)
        : "r"(x0), "r"(x1), "r"(x2));
    return ((uint64_t)t1 << 32) | t0;
#else
    uint64_t t = ((uint64_t)x1 << 32) | x0;
    uint64_t m = ((uint64_t)x2 << 32) - x2;
    uint64_t r = t + m;
    if (r < m) r += FP_EPS;  // r <= 2^64 - 2^33 after the wrap: cannot overflow again
    return r;
#endif
}
// ... -> canonical x mod p
// any 64-bit representative -> the canonical one (select form: no 64-bit compare / subtract)
SB_DEV fp_t fp_canon_sel(fp_t r) {
#if defined(__CUDA_ARCH__)
    uint32_t t0 = (uint32_t)r, t1 = (uint32_t)(r >> 32);
    bool ge = (t1 == 0xffffffffu) & (t0 != 0);  // t >= p  <=>  high word all ones and low word >= 1
    t1 = ge ? 0u : t1;
    t0 -= ge ? 1u : 0u;
    return ((uint64_t)t1 << 32) | t0;
#else
    if (r >= FP_P) r -= FP_P;
    return r;
#endif
}
SB_DEV fp_t fp_reduce96(uint32_t x0, uint32_t x1, uint32_t x2) { return fp_canon_sel(fp_reduce96_nc(x0, x1, x2)); }

// x = x0 + x1*2^32 + x2*2^64 + x3*2^96 + x4*2^128  ->  x mod p
// using 2^64 = 2^32-1, 2^96 = -1, 2^128 = -2^32 (mod p):
//   x = (x0 + x1*2^32) - (x3 + x4*2^32) + x2*(2^32-1)
// x4 must be small (< 2^31): it only ever holds the carries of a dot product.
template <bool CANON>
SB_DEV fp_t fp_reduce160_t(uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t x4) {
#if defined(__CUDA_ARCH__)
    // V = (x1:x0) + x2 (2^32 - 1) - (x4:x3) lies in (-2^40, 2^65 - 2^33): the subtraction may borrow (m = -1), the fold
    // may carry (c = 1); the net multiple k = c + m of 2^64 = EPS (mod p) is applied once -- (t + k EPS) cannot wrap
    // again (k = 1: t <= 2^64 - 2^33; k = -1: t >= 2^64 - 2^40).  Subtracting first lets the fold's carry-out land
    // directly in k (one addc instead of an addc, an add and a predicated copy), and k EPS = (k : 0) - (k >> 31 : k) is
    // applied as a subtraction, which needs no negated copy of k.  t and k are those of the fold-first order.
    uint32_t t0, t1;
    asm("{\n\t"
        ".reg .u32 m, k;\n\t"
        "sub.cc.u32 %0, %2, %5;\n\t"
        "subc.cc.u32 %1, %3, %6;\n\t"
        "subc.u32 m, 0, 0;\n\t"
        "mad.lo.cc.u32 %0, %4, 0xffffffff, %0;\n\t"
        "madc.hi.cc.u32 %1, %4, 0xffffffff, %1;\n\t"
        "addc.u32 k, m, 0;\n\t"
        "shr.s32 m, k, 31;\n\t"           // + k EPS = - (k >> 31 : k) + (k : 0)
        "sub.cc.u32 %0, %0, k;\n\t"
        "subc.u32 %1, %1, m;\n\t"
        "add.u32 %1, %1, k;\n\t"
        "}"
        : "=&r"(t0), "=&r"(t1)
        : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(x4));
    fp_t r = ((uint64_t)t1 << 32) | t0;
    return CANON ? fp_canon_sel(r) : r;
#else
    uint64_t lo = ((uint64_t)x1 << 32) | x0;
    uint64_t sub = ((uint64_t)x4 << 32) | x3;
    uint64_t t = lo - sub;
    if (lo < sub) t -= FP_EPS;  // t >= 2^64 - sub >> EPS: no second borrow
    return CANON ? fp_reduce96((uint32_t)t, (uint32_t)(t >> 32), x2) : fp_reduce96_nc((uint32_t)t, (uint32_t)(t >> 32), x2);
#endif
}
SB_DEV fp_t fp_reduce160(uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t x4) {
    return fp_reduce160_t<true>(x0, x1, x2, x3, x4);
}

// Lazy accumulator of a sum of 64x64-bit products: value = E + O * 2^32
struct wide_acc {
    uint32_t e0, e1, e2, e3, e4;  // bits 0, 32, 64, 96, 128
    uint32_t o1, o2, o3;          // bits 32, 64, 96
};
SB_DEV void wide_zero(wide_acc& w) { w = wide_acc{0, 0, 0, 0, 0, 0, 0, 0}; }

// w += a * b, a and b any 64-bit values; up to 2^30 products may be accumulated
SB_DEV void wide_mac(wide_acc& w, uint64_t a, uint64_t b) {
    uint32_t a0 = (uint32_t)a, a1 = (uint32_t)(a >> 32), b0 = (uint32_t)b, b1 = (uint32_t)(b >> 32);
#if defined(__CUDA_ARCH__)
    asm("mad.lo.cc.u32 %0, %8, %10, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %11, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %11, %3;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        "mad.lo.cc.u32 %5, %8, %11, %5;\n\t"
        "madc.hi.cc.u32 %6, %8, %11, %6;\n\t"
        "addc.u32 %7, %7, 0;\n\t"
        "mad.lo.cc.u32 %5, %9, %10, %5;\n\t"
        "madc.hi.cc.u32 %6, %9, %10, %6;\n\t"
        "addc.u32 %7, %7, 0;"
        : "+r"(w.e0), "+r"(w.e1), "+r"(w.e2), "+r"(w.e3), "+r"(w.e4), "+r"(w.o1), "+r"(w.o2), "+r"(w.o3)
        : "r"(a0), "r"(a1), "r"(b0), "r"(b1));
#else
    SB_WIDE(4);
    typedef unsigned __int128 u128;
    u128 e_lo = ((u128)w.e2 << 64) | ((uint64_t)w.e1 << 32) | w.e0;   // e0..e2 (96 bits) + carries into e3,e4
    u128 E = e_lo + ((u128)w.e3 << 96);
    uint64_t e4 = w.e4;
    u128 p00 = (u128)((uint64_t)a0 * b0), p11 = (u128)((uint64_t)a1 * b1) << 64;
    u128 s = E + p00;
    if (s < E) e4++;
    u128 s2 = s + p11;
    if (s2 < s) e4++;
    w.e0 = (uint32_t)s2; w.e1 = (uint32_t)(s2 >> 32); w.e2 = (uint32_t)(s2 >> 64); w.e3 = (uint32_t)(s2 >> 96);
    w.e4 = (uint32_t)e4;
    u128 O = ((u128)w.o3 << 64) | ((uint64_t)w.o2 << 32) | w.o1;
    O += (uint64_t)a0 * b1;
    O += (uint64_t)a1 * b0;
    w.o1 = (uint32_t)O; w.o2 = (uint32_t)(O >> 32); w.o3 = (uint32_t)(O >> 64);
#endif
}
// w += a * a (3 products; the cross product is added twice)
SB_DEV void wide_mac_sqr(wide_acc& w, uint64_t a) {
    uint32_t a0 = (uint32_t)a, a1 = (uint32_t)(a >> 32);
#if defined(__CUDA_ARCH__)
    asm("{\n\t"
        ".reg .u32 x0, x1;\n\t"
        "mad.lo.cc.u32 %0, %8, %8, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %8, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %9, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %9, %3;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        "mul.lo.u32 x0, %8, %9;\n\t"
        "mul.hi.u32 x1, %8, %9;\n\t"
        "add.cc.u32 %5, %5, x0;\n\t"
        "addc.cc.u32 %6, %6, x1;\n\t"
        "addc.u32 %7, %7, 0;\n\t"
        "add.cc.u32 %5, %5, x0;\n\t"
        "addc.cc.u32 %6, %6, x1;\n\t"
        "addc.u32 %7, %7, 0;\n\t"
        "}"
        : "+r"(w.e0), "+r"(w.e1), "+r"(w.e2), "+r"(w.e3), "+r"(w.e4), "+r"(w.o1), "+r"(w.o2), "+r"(w.o3)
        : "r"(a0), "r"(a1));
#else
    SB_WIDE(-1);  // the device form has three products
    wide_mac(w, a, a);
#endif
}
// double the accumulated value (cross terms of a squaring)
SB_DEV void wide_double(wide_acc& w) {
    w.e4 = (w.e4 << 1) | (w.e3 >> 31);
    w.e3 = (w.e3 << 1) | (w.e2 >> 31);
    w.e2 = (w.e2 << 1) | (w.e1 >> 31);
    w.e1 = (w.e1 << 1) | (w.e0 >> 31);
    w.e0 <<= 1;
    w.o3 = (w.o3 << 1) | (w.o2 >> 31);
    w.o2 = (w.o2 << 1) | (w.o1 >> 31);
    w.o1 <<= 1;
}

template <bool CANON>
SB_DEV fp_t wide_reduce_t(const wide_acc& w) {
    uint32_t x1, x2, x3, x4;
#if defined(__CUDA_ARCH__)
    asm("add.cc.u32 %0, %4, %8;\n\t"
        "addc.cc.u32 %1, %5, %9;\n\t"
        "addc.cc.u32 %2, %6, %10;\n\t"
        "addc.u32 %3, %7, 0;"
        : "=r"(x1), "=r"(x2), "=r"(x3), "=r"(x4)
        : "r"(w.e1), "r"(w.e2), "r"(w.e3), "r"(w.e4), "r"(w.o1), "r"(w.o2), "r"(w.o3));
#else
    unsigned __int128 hi = ((unsigned __int128)w.e4 << 96) | ((unsigned __int128)w.e3 << 64) | ((uint64_t)w.e2 << 32) | w.e1;
    hi += ((unsigned __int128)w.o3 << 64) | ((uint64_t)w.o2 << 32) | w.o1;
    x1 = (uint32_t)hi;
    x2 = (uint32_t)(hi >> 32);
    x3 = (uint32_t)(hi >> 64);
    x4 = (uint32_t)(hi >> 96);
#endif
    return fp_reduce160_t<CANON>(w.e0, x1, x2, x3, x4);
}
SB_DEV fp_t wide_reduce(const wide_acc& w) { return wide_reduce_t<true>(w); }
// any 64-bit representative of the accumulated value (see fp_reduce96_nc)
SB_DEV fp_t wide_reduce_nc(const wide_acc& w) { return wide_reduce_t<false>(w); }

// w = v (start an accumulation from a 64-bit value instead of zero: a free addition)
SB_DEV void wide_set64(wide_acc& w, uint64_t v) { w = wide_acc{(uint32_t)v, (uint32_t)(v >> 32), 0, 0, 0, 0, 0, 0}; }
// w += v for a 64-bit value v
SB_DEV void wide_add64(wide_acc& w, uint64_t v) {
#if defined(__CUDA_ARCH__)
    asm("add.cc.u32 %0, %0, %5;\n\t"
        "addc.cc.u32 %1, %1, %6;\n\t"
        "addc.cc.u32 %2, %2, 0;\n\t"
        "addc.cc.u32 %3, %3, 0;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+r"(w.e0), "+r"(w.e1), "+r"(w.e2), "+r"(w.e3), "+r"(w.e4)
        : "r"((uint32_t)v), "r"((uint32_t)(v >> 32)));
#else
    unsigned __int128 lo = ((unsigned __int128)w.e3 << 96) | ((unsigned __int128)w.e2 << 64) | ((uint64_t)w.e1 << 32) | w.e0;
    unsigned __int128 s = lo + v;
    if (s < lo) w.e4++;
    w.e0 = (uint32_t)s; w.e1 = (uint32_t)(s >> 32); w.e2 = (uint32_t)(s >> 64); w.e3 = (uint32_t)(s >> 96);
#endif
}

// ---- single products -----------------------------------------------------------------------------
// Dedicated 64x64 multiply / square for the long exponentiation chains (Rescue S-boxes, inversions,
// square roots): 4 (3) IMAD.WIDE, two carry adds and the reduction of fp_reduce160_t.  The *_nc forms
// accept ANY 64-bit representatives and return a value < 2^64 that may be >= p ("not canonical"):
// chains stay in that form and canonicalise once at the end (fp_canon).
SB_DEV fp_t fp_canon(fp_t x) { return x >= FP_P ? x - FP_P : x; }

SB_DEV fp_t fp_mul_nc(fp_t a, fp_t b) {
#if defined(__CUDA_ARCH__)
    uint32_t a0 = (uint32_t)a, a1 = (uint32_t)(a >> 32), b0 = (uint32_t)b, b1 = (uint32_t)(b >> 32), t0, t1;
    asm("{\n\t"
        ".reg .u32 p0, p1, p2, p3, m, m0, c;\n\t"
        "mul.lo.u32 p0, %2, %4;\n\t"
        "mul.hi.u32 p1, %2, %4;\n\t"
        "mul.lo.u32 p2, %3, %5;\n\t"
        "mul.hi.u32 p3, %3, %5;\n\t"
        "mad.lo.cc.u32 p1, %2, %5, p1;\n\t"
        "madc.hi.cc.u32 p2, %2, %5, p2;\n\t"
        "addc.u32 p3, p3, 0;\n\t"
        "mad.lo.cc.u32 p1, %3, %4, p1;\n\t"
        "madc.hi.cc.u32 p2, %3, %4, p2;\n\t"
        "addc.u32 p3, p3, 0;\n\t"
        "sub.cc.u32 %0, p0, p3;\n\t"                  // (p1:p0) - p3                [2^96 == -1]
        "subc.cc.u32 %1, p1, 0;\n\t"
        "subc.u32 m, 0, 0;\n\t"
        "mad.lo.cc.u32 %0, p2, 0xffffffff, %0;\n\t"   // + p2 * (2^32 - 1)           [2^64 == 2^32 - 1]
        "madc.hi.cc.u32 %1, p2, 0xffffffff, %1;\n\t"
        "addc.u32 m0, m, 0;\n\t"                      // net multiple of 2^64 == EPS: -1, 0, 1 (fp_reduce160_t)
        "shr.s32 c, m0, 31;\n\t"
        "sub.cc.u32 %0, %0, m0;\n\t"
        "subc.u32 %1, %1, c;\n\t"
        "add.u32 %1, %1, m0;\n\t"
        "}"
        : "=&r"(t0), "=&r"(t1)
        : "r"(a0), "r"(a1), "r"(b0), "r"(b1));
    return ((uint64_t)t1 << 32) | t0;
#else
    SB_WIDE(4);
    return (fp_t)(((unsigned __int128)a * b) % FP_P);
#endif
}
SB_DEV fp_t fp_sqr_nc(fp_t a) {
#if defined(__CUDA_ARCH__)
    uint32_t a0 = (uint32_t)a, a1 = (uint32_t)(a >> 32), t0, t1;
    asm("{\n\t"
        ".reg .u32 p0, p1, p2, p3, c0, c1, c2, m, m0, c;\n\t"
        "mul.lo.u32 p0, %2, %2;\n\t"
        "mul.hi.u32 p1, %2, %2;\n\t"
        "mul.lo.u32 p2, %3, %3;\n\t"
        "mul.hi.u32 p3, %3, %3;\n\t"
        "mul.lo.u32 c0, %2, %3;\n\t"
        "mul.hi.u32 c1, %2, %3;\n\t"
        "shf.l.clamp.b32 c2, c1, 0, 1;\n\t"   // 2 * cross product (65 bits: c2:c1:c0)
        "shf.l.clamp.b32 c1, c0, c1, 1;\n\t"
        "shl.b32 c0, c0, 1;\n\t"
        "add.cc.u32 p1, p1, c0;\n\t"
        "addc.cc.u32 p2, p2, c1;\n\t"
        "addc.u32 p3, p3, c2;\n\t"
        "sub.cc.u32 %0, p0, p3;\n\t"
        "subc.cc.u32 %1, p1, 0;\n\t"
        "subc.u32 m, 0, 0;\n\t"
        "mad.lo.cc.u32 %0, p2, 0xffffffff, %0;\n\t"
        "madc.hi.cc.u32 %1, p2, 0xffffffff, %1;\n\t"
        "addc.u32 m0, m, 0;\n\t"
        "shr.s32 c, m0, 31;\n\t"
        "sub.cc.u32 %0, %0, m0;\n\t"
        "subc.u32 %1, %1, c;\n\t"
        "add.u32 %1, %1, m0;\n\t"
        "}"
        : "=&r"(t0), "=&r"(t1)
        : "r"(a0), "r"(a1));
    return ((uint64_t)t1 << 32) | t0;
#else
    SB_WIDE(3);
    return (fp_t)(((unsigned __int128)a * a) % FP_P);
#endif
}
SB_DEV fp_t fp_mul(fp_t a, fp_t b) { return fp_canon(fp_mul_nc(a, b)); }
SB_DEV fp_t fp_sqr(fp_t a) { return fp_canon(fp_sqr_nc(a)); }
// a * k for a small constant k < 2^32
SB_DEV fp_t fp_mul_small(fp_t a, uint32_t k) {
    SB_WIDE(2);
    uint64_t lo = (uint64_t)(uint32_t)a * k;
    uint64_t hi = (a >> 32) * k;  // weight 2^32
    uint64_t s = lo + (hi << 32);
    uint32_t c = s < lo;
    uint32_t x2 = (uint32_t)(hi >> 32) + c;  // weight 2^64, < 2^32
    return fp_reduce96((uint32_t)s, (uint32_t)(s >> 32), x2);
}
SB_DEV fp_t fp_mul7(fp_t a) { return fp_mul_small(a, 7); }
// 7a as ANY 64-bit representative (not canonical): only ever fed to wide_mac as a multiplicand
SB_DEV fp_t fp_mul7_nc(fp_t a) {
#if defined(__CUDA_ARCH__)
    uint32_t a0 = (uint32_t)a, a1 = (uint32_t)(a >> 32), t0, t1;
    asm("{\n\t"
        ".reg .u32 x1, x2, c;\n\t"
        "mul.lo.u32 %0, %2, 7;\n\t"
        "mul.hi.u32 x1, %2, 7;\n\t"
        "mad.lo.cc.u32 %1, %3, 7, x1;\n\t"
        "madc.hi.u32 x2, %3, 7, 0;\n\t"
        "mad.lo.cc.u32 %0, x2, 0xffffffff, %0;\n\t"   // + x2 * (2^32 - 1)
        "madc.hi.cc.u32 %1, x2, 0xffffffff, %1;\n\t"
        "addc.u32 c, 0, 0;\n\t"
        "sub.cc.u32 %0, %0, c;\n\t"
        "subc.u32 %1, %1, 0;\n\t"
        "add.u32 %1, %1, c;\n\t"
        "}"
        : "=&r"(t0), "=&r"(t1)
        : "r"(a0), "r"(a1));
    return ((uint64_t)t1 << 32) | t0;
#else
    return fp_mul_small(a, 7);
#endif
}

// a^(2^n)
SB_DEV fp_t fp_sqr_n_nc(fp_t a, int n) {
#pragma unroll 1
    for (int i = 0; i < n; i++) a = fp_sqr_nc(a);
    return a;
}
SB_DEV fp_t fp_sqr_n(fp_t a, int n) { return fp_canon(fp_sqr_n_nc(a, n)); }
// a^-1 = a^(p-2),  p - 2 = 0xfffffffeffffffff = (2^31 - 1) << 33 | (2^32 - 1): 63 squarings + 10 multiplications
SB_DEV_NOINLINE fp_t fp_inv(fp_t a) {
    // t_k = a^(2^k - 1)
    fp_t t2 = fp_mul(fp_sqr(a), a);
    fp_t t4 = fp_mul(fp_sqr_n(t2, 2), t2);
    fp_t t8 = fp_mul(fp_sqr_n(t4, 4), t4);
    fp_t t16 = fp_mul(fp_sqr_n(t8, 8), t8);
    fp_t t32 = fp_mul(fp_sqr_n(t16, 16), t16);
    fp_t t31 = fp_mul(fp_sqr_n(fp_mul(fp_sqr_n(fp_mul(fp_sqr_n(t16, 8), t8), 4), t4), 2), t2);  // 2^30-1
    t31 = fp_mul(fp_sqr(t31), a);                                                                // 2^31-1
    return fp_mul(fp_sqr_n(t31, 33), t32);
}

}  // namespace sb
