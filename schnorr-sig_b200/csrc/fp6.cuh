// Sextic extension Fp6 = Fp[u]/(u^6 - 7) (reference README.md:8; `cheetah::Fp6`, call sites
// src/signature.rs:186,278-282, src/batch.rs:67).  Coefficients c0..c5, canonical.
//
// Multiplication: the wrap-around terms (i + j >= 6) use b pre-scaled by 7, so every output
// coefficient is exactly six 64x64 products accumulated lazily (even/odd accumulators, fp.cuh) and reduced
// once.  24 IMAD.WIDE per coefficient: 144 (+5 for the x7 prescale) per multiplication, 87 per squaring.
#pragma once
#include "fp.cuh"

namespace sb {

struct fp6 {
    fp_t c[6];
};

SB_DEV fp6 fp6_zero() { return fp6{{0, 0, 0, 0, 0, 0}}; }
SB_DEV fp6 fp6_one() { return fp6{{1, 0, 0, 0, 0, 0}}; }
SB_DEV fp6 fp6_add(const fp6& a, const fp6& b) {
    fp6 r;
#pragma unroll
    for (int i = 0; i < 6; i++) r.c[i] = fp_add(a.c[i], b.c[i]);
    return r;
}
SB_DEV fp6 fp6_sub(const fp6& a, const fp6& b) {
    fp6 r;
#pragma unroll
    for (int i = 0; i < 6; i++) r.c[i] = fp_sub(a.c[i], b.c[i]);
    return r;
}
SB_DEV fp6 fp6_neg(const fp6& a) {
    fp6 r;
#pragma unroll
    for (int i = 0; i < 6; i++) r.c[i] = fp_neg(a.c[i]);
    return r;
}
SB_DEV fp6 fp6_dbl(const fp6& a) { return fp6_add(a, a); }
SB_DEV bool fp6_is_zero(const fp6& a) { return (a.c[0] | a.c[1] | a.c[2] | a.c[3] | a.c[4] | a.c[5]) == 0; }
SB_DEV bool fp6_eq(const fp6& a, const fp6& b) {
    uint64_t d = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) d |= a.c[i] ^ b.c[i];
    return d == 0;
}
// every limb canonical?  (Fp6::from_bytes is None otherwise -> the reference panics, src/signature.rs:186)
SB_DEV bool fp6_is_canonical(const fp6& a) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 6; i++) ok &= a.c[i] < FP_P;
    return ok;
}

// CANON = false: the coefficients are returned as arbitrary 64-bit representatives (fp_reduce96_nc) -- for
// products that only feed further multiplications
template <bool CANON = true>
SB_DEV void fp6_mul_body(fp6& r, const fp6& a, const fp6& b) {
    fp_t b7[6];
#pragma unroll
    for (int j = 1; j < 6; j++) b7[j] = fp_mul7_nc(b.c[j]);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        wide_acc w;
        wide_zero(w);
#pragma unroll
        for (int i = 0; i < 6; i++) {
            if (i <= k) wide_mac(w, a.c[i], b.c[k - i]);
            else wide_mac(w, a.c[i], b7[k + 6 - i]);
        }
        r.c[k] = wide_reduce_t<CANON>(w);
    }
}

// Squaring with optional subtracted terms riding in the lazy accumulators (no reduction / subtraction of their own):
//   MODE 0:  a^2
//   MODE 1:  a^2 - 2 A              (A canonical; p - A_k starts the accumulator and is doubled with the cross terms)
//   MODE 2:  a^2 - A - B s          (A, B canonical; s any 64-bit representative of an Fp element)
// These are X3 = L^2 - 2 X m^2 and X3 = L^2 - x1 w3^2 - x2 w3^2 of the point formulas in affine.cuh.
template <int MODE, bool CANON = true>
SB_DEV void fp6_sqr_body_t(fp6& r, const fp6& a, const fp6* A, const fp6* B, fp_t s) {
    fp_t a7[6];
#pragma unroll
    for (int j = 3; j < 6; j++) a7[j] = fp_mul7_nc(a.c[j]);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        wide_acc w;
        if (MODE == 1) wide_set64(w, FP_P - A->c[k]);
        else wide_zero(w);
        // cross terms i < j
#pragma unroll
        for (int i = 0; i < 6; i++) {
#pragma unroll
            for (int j = i + 1; j < 6; j++) {
                if (i + j == k) wide_mac(w, a.c[i], a.c[j]);
                if (i + j == k + 6) wide_mac(w, a.c[i], a7[j]);
            }
        }
        wide_double(w);
        if ((k & 1) == 0) {
            wide_mac_sqr(w, a.c[k / 2]);
            wide_mac(w, a.c[k / 2 + 3], a7[k / 2 + 3]);
        }
        if (MODE == 2) {
            wide_add64(w, FP_P - A->c[k]);
            wide_mac(w, FP_P - B->c[k], s);
        }
        r.c[k] = wide_reduce_t<CANON>(w);
    }
}
SB_DEV void fp6_sqr_body(fp6& r, const fp6& a) { fp6_sqr_body_t<0>(r, a, nullptr, nullptr, 0); }

// a * b - c * s with s in Fp (any 64-bit representative), c canonical: the scaled subtraction rides in the lazy
// accumulators of the product -- six more 64x64 products, but no reduction and no subtraction of its own
// (Y3 = L (A - X3) - Y s of the point formulas in affine.cuh)
SB_DEV void fp6_mul_sub_scaled_body(fp6& r, const fp6& a, const fp6& b, const fp6& c, fp_t s) {
    fp_t b7[6];
#pragma unroll
    for (int j = 1; j < 6; j++) b7[j] = fp_mul7_nc(b.c[j]);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        wide_acc w;
        wide_zero(w);
#pragma unroll
        for (int i = 0; i < 6; i++) {
            if (i <= k) wide_mac(w, a.c[i], b.c[k - i]);
            else wide_mac(w, a.c[i], b7[k + 6 - i]);
        }
        wide_mac(w, FP_P - c.c[k], s);
        r.c[k] = wide_reduce(w);
    }
}

// Out-of-line: one copy of the ~500-instruction bodies per kernel keeps the hot loops inside the
// instruction cache (inlined: 3.65 against 4.78 M/s, profiles/r1_variants.md, v2-D).
SB_DEV_NOINLINE fp6 fp6_mul(fp6 a, fp6 b) {
    fp6 r;
    fp6_mul_body<true>(r, a, b);
    return r;
}
SB_DEV_NOINLINE fp6 fp6_sqr(fp6 a) {
    fp6 r;
    fp6_sqr_body(r, a);
    return r;
}
// (helpers with TWO call sites per kernel stay out of line: duplicating them costs what the calls save,
// profiles/r2_variants.md)
SB_DEV_NOINLINE fp6 fp6_mul_sub_scaled(fp6 a, fp6 b, fp6 c, fp_t s) {
    fp6 r;
    fp6_mul_sub_scaled_body(r, a, b, c, s);
    return r;
}
// a * b with non-canonical coefficients (feeds multiplications only)
SB_DEV_NOINLINE fp6 fp6_mul_nc(fp6 a, fp6 b) {
    fp6 r;
    fp6_mul_body<false>(r, a, b);
    return r;
}
// The three squaring forms below have ONE call site per kernel (the fused doubling / addition, the mixed addition of
// the MSM): inlined there they cost no code and save the argument marshalling of a call (k_verify_fast 75.21
// against 76.33 ms out of line, profiles/r2_variants.md, v16).
// a^2 with non-canonical coefficients
SB_DEV fp6 fp6_sqr_nc(fp6 a) {
    fp6 r;
    fp6_sqr_body_t<0, false>(r, a, nullptr, nullptr, 0);
    return r;
}
// a^2 - 2 A
SB_DEV fp6 fp6_sqr_sub2(fp6 a, fp6 A) {
    fp6 r;
    fp6_sqr_body_t<1>(r, a, &A, nullptr, 0);
    return r;
}
// a^2 - A - B s
SB_DEV fp6 fp6_sqr_sub_scaled(fp6 a, fp6 A, fp6 B, fp_t s) {
    fp6 r;
    fp6_sqr_body_t<2>(r, a, &A, &B, s);
    return r;
}

// ---- cubic subfield Fp3 = Fp[v]/(v^3 - 7), v = u^2, used by inversion and square roots ----
struct fp3 {
    fp_t c[3];
};
// out of line (by value, register ABI): the square-root / inversion code stays compact
SB_DEV_NOINLINE fp3 fp3_mul(fp3 a, fp3 b) {
    fp3 r;
    fp_t b7_1 = fp_mul7_nc(b.c[1]), b7_2 = fp_mul7_nc(b.c[2]);
    wide_acc w;
    wide_zero(w);
    wide_mac(w, a.c[0], b.c[0]);
    wide_mac(w, a.c[1], b7_2);
    wide_mac(w, a.c[2], b7_1);
    r.c[0] = wide_reduce(w);
    wide_zero(w);
    wide_mac(w, a.c[0], b.c[1]);
    wide_mac(w, a.c[1], b.c[0]);
    wide_mac(w, a.c[2], b7_2);
    r.c[1] = wide_reduce(w);
    wide_zero(w);
    wide_mac(w, a.c[0], b.c[2]);
    wide_mac(w, a.c[1], b.c[1]);
    wide_mac(w, a.c[2], b.c[0]);
    r.c[2] = wide_reduce(w);
    return r;
}
// ---- Fp3 squaring, 6 products -------------------------------------------------------------------
SB_DEV fp3 fp3_sqr6(const fp3& a) {
    fp_t a2_7 = fp_mul7_nc(a.c[2]);
    fp3 r;
    wide_acc w;
    wide_zero(w);
    wide_mac(w, a.c[1], a2_7);
    wide_double(w);
    wide_mac_sqr(w, a.c[0]);
    r.c[0] = wide_reduce(w);
    wide_zero(w);
    wide_mac(w, a.c[0], a.c[1]);
    wide_double(w);
    wide_mac(w, a.c[2], a2_7);
    r.c[1] = wide_reduce(w);
    wide_zero(w);
    wide_mac(w, a.c[0], a.c[2]);
    wide_double(w);
    wide_mac_sqr(w, a.c[1]);
    r.c[2] = wide_reduce(w);
    return r;
}

// out of line for the long squaring runs of the square-root code
SB_DEV_NOINLINE fp3 fp3_sqr(fp3 a) { return fp3_sqr6(a); }
SB_DEV fp3 fp3_sub(const fp3& a, const fp3& b) {
    return fp3{{fp_sub(a.c[0], b.c[0]), fp_sub(a.c[1], b.c[1]), fp_sub(a.c[2], b.c[2])}};
}
SB_DEV fp3 fp3_add(const fp3& a, const fp3& b) {
    return fp3{{fp_add(a.c[0], b.c[0]), fp_add(a.c[1], b.c[1]), fp_add(a.c[2], b.c[2])}};
}
SB_DEV fp3 fp3_neg(const fp3& a) { return fp3{{fp_neg(a.c[0]), fp_neg(a.c[1]), fp_neg(a.c[2])}}; }
SB_DEV fp3 fp3_mulv(const fp3& a) { return fp3{{fp_mul7(a.c[2]), a.c[0], a.c[1]}}; }  // * v
SB_DEV fp3 fp3_scale(const fp3& a, fp_t k) { return fp3{{fp_mul(a.c[0], k), fp_mul(a.c[1], k), fp_mul(a.c[2], k)}}; }
SB_DEV bool fp3_is_zero(const fp3& a) { return (a.c[0] | a.c[1] | a.c[2]) == 0; }
// adjugate / norm:  d^-1 = (t0 + t1 v + t2 v^2) / N(d)
SB_DEV void fp3_adj_norm(const fp3& d, fp3& adj, fp_t& norm) {
    fp_t d0 = d.c[0], d1 = d.c[1], d2 = d.c[2];
    fp_t t0 = fp_sub(fp_sqr(d0), fp_mul7(fp_mul(d1, d2)));
    fp_t t1 = fp_sub(fp_mul7(fp_sqr(d2)), fp_mul(d0, d1));
    fp_t t2 = fp_sub(fp_sqr(d1), fp_mul(d0, d2));
    norm = fp_add(fp_mul(d0, t0), fp_mul7(fp_add(fp_mul(d2, t1), fp_mul(d1, t2))));
    adj = fp3{{t0, t1, t2}};
}
SB_DEV fp3 fp3_inv(const fp3& d) {
    fp3 adj;
    fp_t n;
    fp3_adj_norm(d, adj, n);
    return fp3_scale(adj, fp_inv(n));
}
SB_DEV void fp6_split(const fp6& a, fp3& a0, fp3& a1) {  // a = a0 + a1*u over Fp3
    a0 = fp3{{a.c[0], a.c[2], a.c[4]}};
    a1 = fp3{{a.c[1], a.c[3], a.c[5]}};
}
SB_DEV fp6 fp6_join(const fp3& a0, const fp3& a1) { return fp6{{a0.c[0], a1.c[0], a0.c[1], a1.c[1], a0.c[2], a1.c[2]}}; }

// a^-1 through the tower Fp6 = Fp3[u]/(u^2 - v):  (a0 + a1 u)^-1 = (a0 - a1 u) / (a0^2 - v a1^2).
// Returns 0 for a = 0.
SB_DEV_NOINLINE fp6 fp6_inv(fp6 a) {
    fp3 a0, a1;
    fp6_split(a, a0, a1);
    fp3 d = fp3_sub(fp3_sqr(a0), fp3_mulv(fp3_sqr(a1)));
    fp3 di = fp3_inv(d);
    return fp6_join(fp3_mul(a0, di), fp3_mul(fp3_neg(a1), di));
}

// "lexicographically largest": decided by the highest non-zero coefficient (oracle/pyref.py
// f6_lex_largest; [RECALLED] convention of cheetah's compressed encoding)
SB_DEV bool fp6_lex_largest(const fp6& a) {
    bool res = false, decided = false;
#pragma unroll
    for (int i = 5; i >= 0; i--) {
        bool nz = a.c[i] != 0;
        bool big = a.c[i] > (FP_P - 1) / 2;
        res = decided ? res : (nz & big);
        decided |= nz;
    }
    return res;
}

// ---------------------------------------------------------------------------------------------
// Square roots (used by AffinePoint::from_compressed: src/batch.rs:104, src/public.rs:55).
// Which root is returned is irrelevant: the caller fixes the sign with the flag bit.

// a^(2^32 - 1)
SB_DEV fp_t fp_pow_2_32_m1(fp_t a) {
    fp_t t2 = fp_mul(fp_sqr(a), a);
    fp_t t4 = fp_mul(fp_sqr_n(t2, 2), t2);
    fp_t t8 = fp_mul(fp_sqr_n(t4, 4), t4);
    fp_t t16 = fp_mul(fp_sqr_n(t8, 8), t8);
    return fp_mul(fp_sqr_n(t16, 16), t16);
}
// Legendre symbol: a^((p-1)/2) == 1 (a != 0);  (p-1)/2 = 2^31 * (2^32 - 1)
SB_DEV bool fp_is_square(fp_t a) {
    if (a == 0) return true;
    return fp_sqr_n(fp_pow_2_32_m1(a), 31) == 1;
}
// Tonelli-Shanks in Fp with a WINDOWED discrete logarithm: p - 1 = 2^32 t, t = 2^32 - 1, g = 7^t generates the
// 2-power torsion.  For a != 0: x = a^((t+1)/2), b = a^t = g^e, and sqrt(a) = x g^(-e/2) when e is even (a is a
// non-residue when e is odd).  e is read eight bits at a time: (b g^-(e0 + ... ))^(2^(24-8i)) lies in the subgroup of
// order 256, whose discrete log is one lookup in a perfect-hash table (include/fp_sqrt_tables.h, generated by
// tools/gen_params.py).  48 squarings + 8 multiplications, uniform control flow -- the textbook loop needs ~300
// squarings on average and diverges between the lanes of a warp.
#if defined(__CUDACC__)
#define FP_TABLE_QUAL __device__
#endif
}  // namespace sb
#include "../../include/fp_sqrt_tables.h"
namespace sb {
static constexpr fp_t FP_NONE = ~0ULL;  // not a canonical element: "no square root"
SB_DEV_NOINLINE fp_t fp_sqrt_or_none(fp_t a) {
    if (a == 0) return 0;
    fp_t x = fp_sqr_n(a, 31);        // a^((t+1)/2)
    fp_t c = fp_pow_2_32_m1(a);      // a^t, in the 2-power torsion
    uint32_t e[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        fp_t bi = fp_sqr_n(c, 24 - 8 * i);  // order divides 256
        e[i] = FP_SQRT_DLOG[(bi * FP_SQRT_DLOG_MUL) >> FP_SQRT_DLOG_SHIFT];
        c = fp_mul(c, FP_SQRT_GINV[256 * i + e[i]]);
    }
    if (e[0] & 1) return FP_NONE;
    fp_t r = fp_mul(x, FP_SQRT_GINV[e[0] >> 1]);
#pragma unroll
    for (int i = 1; i < 4; i++) r = fp_mul(r, FP_SQRT_HALF[256 * (i - 1) + e[i]]);
    return r;
}
SB_DEV bool fp_sqrt(fp_t a, fp_t& out) {
    fp_t r = fp_sqrt_or_none(a);
    if (r == FP_NONE) return false;
    out = r;
    return true;
}

SB_DEV fp3 fp3_sqr_n(fp3 a, int n) {
#pragma unroll 1
    for (int i = 0; i < n; i++) a = fp3_sqr(a);
    return a;
}
SB_DEV fp_t fp3_norm(const fp3& a) {
    fp3 adj;
    fp_t n;
    fp3_adj_norm(a, adj, n);
    return n;
}
// a is a square in Fp3  <=>  N(a) is a square in Fp  (odd-degree extension)
SB_DEV bool fp3_is_square(const fp3& a) { return fp_is_square(fp3_norm(a)); }
// sqrt in Fp3 through the norm: with e = p^2 + p + 1 (odd), a^e = N(a) in Fp and
//   sqrt(a) = a^((e+1)/2) / sqrt(N(a)),   a^((e+1)/2) = Frob(a^((p+1)/2)) * a,  (p+1)/2 = 2^31 (2^32-1) + 1
SB_DEV_NOINLINE fp3 fp3_sqrt_or_none(fp3 a) {
    if (fp3_is_zero(a)) return a;
    fp_t s;
    if (!fp_sqrt(fp3_norm(a), s)) return fp3{{FP_NONE, 0, 0}};
    // c = a^(2^32 - 1)
    fp3 t2 = fp3_mul(fp3_sqr(a), a);
    fp3 t4 = fp3_mul(fp3_sqr_n(t2, 2), t2);
    fp3 t8 = fp3_mul(fp3_sqr_n(t4, 4), t4);
    fp3 t16 = fp3_mul(fp3_sqr_n(t8, 8), t8);
    fp3 c = fp3_mul(fp3_sqr_n(t16, 16), t16);
    c = fp3_mul(fp3_sqr_n(c, 31), a);  // a^((p+1)/2)
    const fp_t w = 0xfffffffe00000001ULL;  // FP_OMEGA3: v^p = w v
    const fp_t w2 = fp_sqr(w);
    fp3 f = fp3{{c.c[0], fp_mul(c.c[1], w), fp_mul(c.c[2], w2)}};  // Frobenius
    return fp3_scale(fp3_mul(f, a), fp_inv(s));
}
SB_DEV bool fp3_sqrt(const fp3& a, fp3& out) {
    fp3 r = fp3_sqrt_or_none(a);
    if (r.c[0] == FP_NONE) return false;
    out = r;
    return true;
}

// sqrt in Fp6 = Fp3[u]/(u^2 - v) by the complex method.  Returns false if a is not a square.
SB_DEV bool fp6_sqrt(const fp6& a, fp6& out) {
    fp3 a0, a1;
    fp6_split(a, a0, a1);
    const fp_t half = 0x7fffffff80000001ULL;  // 2^-1 mod p
    if (fp3_is_zero(a1)) {
        // a in Fp3: a square there, or v * square (then the root is a multiple of u)
        fp3 r;
        if (fp3_sqrt(a0, r)) {
            out = fp6_join(r, fp3{{0, 0, 0}});
            return true;
        }
        // a0 / v = (c1, c2, c0/7): sqrt(a0) = sqrt(a0/v) * u
        const fp_t inv7 = 0x249249246db6db6eULL;  // 7^-1 mod p
        fp3 q = fp3{{a0.c[1], a0.c[2], fp_mul(a0.c[0], inv7)}};
        if (!fp3_sqrt(q, r)) return false;  // cannot happen
        out = fp6_join(fp3{{0, 0, 0}}, r);
        return true;
    }
    fp3 nrm = fp3_sub(fp3_sqr(a0), fp3_mulv(fp3_sqr(a1)));
    fp3 n;
    if (!fp3_sqrt(nrm, n)) return false;
    fp3 d = fp3_scale(fp3_add(a0, n), half);
    if (!fp3_is_square(d)) d = fp3_scale(fp3_sub(a0, n), half);
    fp3 x0;
    if (!fp3_sqrt(d, x0)) return false;
    fp3 x1 = fp3_mul(a1, fp3_inv(fp3_add(x0, x0)));
    out = fp6_join(x0, x1);
    return fp6_eq(fp6_sqr(out), a);
}

}  // namespace sb
