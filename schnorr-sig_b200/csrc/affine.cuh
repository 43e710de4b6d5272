// Fast path of the verification (Signature::verify, src/signature.rs:181-205): point arithmetic in
// "(X, Y, w)" coordinates -- affine formulas whose field inversions are replaced by a denominator kept in
// the BASE field.
//
// In Fp6 the inverse of d is c / n with the cofactor c in Fp6 and the norm n in Fp (tower Fp6 -> Fp3 -> Fp,
// ~42 base-field products).  Keeping x = X / w^2, y = Y / w^3 with w in Fp lets every slope denominator be
// absorbed into w, and scaling by an Fp element costs a sixth of an Fp6 multiplication: an addition is
// 2M + 1S + cofactor + 7 scalings instead of the 11M + 5S of a Jacobian addition, a doubling 2M + 2S +
// cofactor + 2 scalings, and no inversion is ever performed.  (A first version used true affine points with
// Montgomery-shared Fp inversions: one 74-product inversion per chain step made it only 10 % faster than
// the Jacobian kernel -- profiles/r1_variants.md.)
//
// The affine group law has exceptional inputs (P + P, P + (-P), the identity).  They cannot occur for
// honest keys except with negligible probability, but adversarial small-order keys reach them, so the
// fast path DETECTS every such event (a zero norm, an identity operand it cannot represent)
// and reports FAST_EXCEPTIONAL; the caller then re-runs that signature through the exact Jacobian
// routine (curve.cuh: torsion_check_and_mul).  A result that is not flagged is the exact group
// element, so verdicts stay bit-identical to the reference.
#pragma once
#include "curve.cuh"

namespace sb {

// adjugate and norm of d in Fp3 with lazily accumulated products (12 products, 4 reductions):
//   d^-1 = (t0 + t1 v + t2 v^2) / n,   t0 = d0^2 - 7 d1 d2,  t1 = 7 d2^2 - d0 d1,  t2 = d1^2 - d0 d2,
//   n = d0 t0 + 7 (d2 t1 + d1 t2)
SB_DEV void fp3_adj_norm_lazy(const fp3& d, fp3& adj, fp_t& norm) {
    fp_t d0 = d.c[0], d1 = d.c[1], d2 = d.c[2];
    fp_t d1_7 = fp_mul7_nc(d1), d2_7 = fp_mul7_nc(d2);
    fp_t nd0 = FP_P - d0, nd1 = FP_P - d1;  // negatives as 64-bit representatives (p itself for 0)
    wide_acc w;
    wide_zero(w);
    wide_mac_sqr(w, d0);
    wide_mac(w, nd1, d2_7);
    fp_t t0 = wide_reduce_nc(w);  // the adjugate only feeds products: any 64-bit representative will do
    wide_zero(w);
    wide_mac(w, d2, d2_7);
    wide_mac(w, nd0, d1);
    fp_t t1 = wide_reduce_nc(w);
    wide_zero(w);
    wide_mac_sqr(w, d1);
    wide_mac(w, nd0, d2);
    fp_t t2 = wide_reduce_nc(w);
    wide_zero(w);
    wide_mac(w, d0, t0);
    wide_mac(w, d2_7, t1);
    wide_mac(w, d1_7, t2);
    norm = wide_reduce(w);
    adj = fp3{{t0, t1, t2}};
}

// ---- Jacobian coordinates with the denominator in the BASE field -------------------------------------
// (X, Y, w), x = X / w^2, y = Y / w^3 with w in Fp*.  The slope of a chord / tangent has a denominator d in Fp6;
// instead of inverting it, write 1/d = c / n with the cofactor c = n / d in Fp6 and the norm n in Fp (tower
// Fp6 -> Fp3 -> Fp, ~42 base-field products) and push n into the new w.  Scaling by an Fp element costs 6
// products (a sixth of an Fp6 multiplication), so
//     doubling  = 2M + 2S + cofactor + 2 scalings        (Jacobian dbl-2007-bl: 1M + 8S)
//     addition  = 2M + 1S + cofactor + 7 scalings        (Jacobian add-2007-bl: 11M + 5S)
// and no field inversion is ever needed.
struct jf_pt {
    fp6 X, Y;
    fp_t w;
};

// a * b in Fp3 with the wrap-around multiples 7 b1, 7 b2 supplied by the caller (shared by several products);
// coefficients returned as arbitrary 64-bit representatives (the cofactor only feeds a multiplication)
SB_DEV fp3 fp3_mul_pre(const fp3& a, const fp3& b, fp_t b7_1, fp_t b7_2) {
    fp3 r;
    wide_acc w;
    wide_zero(w);
    wide_mac(w, a.c[0], b.c[0]);
    wide_mac(w, a.c[1], b7_2);
    wide_mac(w, a.c[2], b7_1);
    r.c[0] = wide_reduce_nc(w);
    wide_zero(w);
    wide_mac(w, a.c[0], b.c[1]);
    wide_mac(w, a.c[1], b.c[0]);
    wide_mac(w, a.c[2], b7_2);
    r.c[1] = wide_reduce_nc(w);
    wide_zero(w);
    wide_mac(w, a.c[0], b.c[2]);
    wide_mac(w, a.c[1], b.c[1]);
    wide_mac(w, a.c[2], b.c[0]);
    r.c[2] = wide_reduce_nc(w);
    return r;
}

// d * c = n,  c in Fp6 (coefficients NOT canonical: c only ever feeds a multiplication), n in Fp canonical;
// n == 0 <=> d == 0.  d canonical.
//   d = x + y u over Fp3 (x = (d0, d2, d4), y = (d1, d3, d5)),  1/d = (x - y u) / N,  N = x^2 - v y^2 in Fp3,
//   v (t0, t1, t2) = (7 t2, t0, t1).  The three coefficients of N are accumulated directly (12 products, three
//   reductions, no subtraction: the y terms enter through p - y_i):
//     N0 = x0^2 + 2 x1 7x2 - 2 y0 7y2 - y1 7y1      N1 = 2 x0 x1 + x2 7x2 - y0^2 - 2 y1 7y2
//     N2 = 2 x0 x2 + x1^2 - 2 y0 y1 - y2 7y2
// Operand and results travel in registers (a by-value struct): the pointer form cost a 13-word round trip through
// thread-local memory per call (403 calls per verification; ncu: 0.7 % of the kernel in load stalls behind them).
struct fp6_cof {
    fp6 c;
    fp_t n;
};
SB_DEV fp6_cof fp6_cofactor_norm_body(const fp6& d) {
    fp6_cof out;
    fp6* c = &out.c;
    fp_t* n = &out.n;
    fp3 x, y, adj;
    fp6_split(d, x, y);
    fp3 ny = fp3{{FP_P - y.c[0], FP_P - y.c[1], FP_P - y.c[2]}};
    fp_t x2_7 = fp_mul7_nc(x.c[2]), y1_7 = fp_mul7_nc(y.c[1]), y2_7 = fp_mul7_nc(y.c[2]);
    fp3 nn;
    wide_acc w;
    wide_zero(w);
    wide_mac(w, x.c[1], x2_7);
    wide_mac(w, ny.c[0], y2_7);
    wide_double(w);
    wide_mac_sqr(w, x.c[0]);
    wide_mac(w, ny.c[1], y1_7);
    nn.c[0] = wide_reduce(w);
    wide_zero(w);
    wide_mac(w, x.c[0], x.c[1]);
    wide_mac(w, ny.c[1], y2_7);
    wide_double(w);
    wide_mac(w, x.c[2], x2_7);
    wide_mac(w, ny.c[0], y.c[0]);
    nn.c[1] = wide_reduce(w);
    wide_zero(w);
    wide_mac(w, x.c[0], x.c[2]);
    wide_mac(w, ny.c[0], y.c[1]);
    wide_double(w);
    wide_mac_sqr(w, x.c[1]);
    wide_mac(w, ny.c[2], y2_7);
    nn.c[2] = wide_reduce(w);
    fp3_adj_norm_lazy(nn, adj, *n);  // 1/N = adj / n
    fp_t adj7_1 = fp_mul7_nc(adj.c[1]), adj7_2 = fp_mul7_nc(adj.c[2]);
    *c = fp6_join(fp3_mul_pre(x, adj, adj7_1, adj7_2), fp3_mul_pre(ny, adj, adj7_1, adj7_2));
    return out;
}
SB_DEV_NOINLINE fp6_cof fp6_cofactor_norm_v(fp6 d) { return fp6_cofactor_norm_body(d); }
SB_DEV void fp6_cofactor_norm(const fp6* d, fp6* c, fp_t* n) {
    fp6_cof r = fp6_cofactor_norm_v(*d);
    *c = r.c;
    *n = r.n;
}
// The slope of a chord / tangent up to its base-field denominator: L = num * (n / d), n = norm(d).  Cofactor and product
// in ONE out-of-line function (the fused doubling and addition both end in this pair): the cofactor never leaves the
// registers and one call with its argument marshalling is saved per point operation (k_verify_fast 74.61 against
// 75.38 ms with two calls, profiles/r2_variants.md, v17).  L not canonical.
SB_DEV_NOINLINE fp6_cof fp6_slope_nc(fp6 num, fp6 d) {
    fp6_cof r = fp6_cofactor_norm_body(d);
    fp6 L;
    fp6_mul_body<false>(L, num, r.c);
    r.c = L;
    return r;
}

// The scaling helpers are inlined into jf_add / jf_dbl: 50.2 against 50.65 ms out of line (profiles/r1_variants.md).
// a * s for s in Fp (any 64-bit representative)
SB_DEV fp6 fp6_scale(fp6 a, fp_t s) {
    fp6 r;
#pragma unroll
    for (int i = 0; i < 6; i++) r.c[i] = fp_mul(a.c[i], s);
    return r;
}
// a * s - b * t  (s, t any 64-bit representatives; a, b canonical)
SB_DEV fp6 fp6_scale_diff(fp6 a, fp_t s, fp6 b, fp_t t) {
    fp6 r;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        wide_acc w;
        wide_zero(w);
        wide_mac(w, a.c[i], s);
        wide_mac(w, FP_P - b.c[i], t);
        r.c[i] = wide_reduce(w);
    }
    return r;
}

// a * s - b * t with non-canonical coefficients (feeds a multiplication only)
SB_DEV fp6 fp6_scale_diff_nc(fp6 a, fp_t s, fp6 nb, fp_t t) {  // nb = a representative of -b (p - b, or b itself
    fp6 r;                                                     // when the caller wants a s + b t)
#pragma unroll
    for (int i = 0; i < 6; i++) {
        wide_acc w;
        wide_zero(w);
        wide_mac(w, a.c[i], s);
        wide_mac(w, nb.c[i], t);
        r.c[i] = wide_reduce_nc(w);
    }
    return r;
}

// p <- 2 p.  Returns true on the exceptional input (a point of order 2: the result would be the identity).
// FUSED (k_verify_fast): X3 = L^2 - 2 A and Y3 = L (A - X3) - Y m^3 each come out of ONE lazy accumulation
// (fp6_sqr_sub2, fp6_mul_sub_scaled), L and the cofactor stay non-canonical.  The MSM kernels keep the plain
// form: the fused helpers take 38 argument registers, which costs k_msm_segment_sum a resident block.
template <bool FUSED = false>
SB_DEV_NOINLINE bool jf_dbl(jf_pt* p) {
#if defined(__CUDA_ARCH__)
    // The fused form is only ever handed a shared-memory slot (the running point of k_verify_fast): telling the compiler
    // turns 26 generic accesses -- each with its own descriptor set-up (two R2UR) -- into LDS / STS.
    if (FUSED) __builtin_assume(__isShared(p));
#endif
    fp6 X = p->X, Y = p->Y, c;
    fp_t w = p->w, n;
    if (FUSED) {
        // slope = (3 X^2 + w^4) c / (2 n w) = (X^2 + w^4 / 3) c / (m w) with m = 2 n / 3 and 1 / (2 Y) = c / (2 n): the
        // factor 3 moves into the denominator (one product by a constant) instead of tripling the six coefficients of X^2
        const fp_t inv3 = 0xaaaaaaaa00000001ULL, two_thirds = 0x5555555500000001ULL;
        fp_t w4 = fp_mul(fp_sqr_nc(fp_sqr_nc(w)), inv3);
        fp6 num = fp6_sqr_nc(X);
        num.c[0] = fp_add(num.c[0], w4);    // (a non-canonical minuend is fine, fp_sub)
        fp6_cof sl = fp6_slope_nc(num, Y);
        fp6 L = sl.c;                       // slope = L / (m w)
        n = sl.n;
        fp_t m = fp_mul(n, two_thirds);
        fp_t m2 = fp_sqr_nc(m), m3 = fp_mul_nc(m2, m);
        fp6 A = fp6_scale(X, m2);
        fp6 X3 = fp6_sqr_sub2(L, A);
        p->Y = fp6_mul_sub_scaled(L, fp6_sub(A, X3), Y, m3);
        p->X = X3;
        p->w = fp_mul(m, w);
        return n == 0;
    }
    fp6_cofactor_norm(&Y, &c, &n);          // 1 / (2 Y) = c / (2 n)
    fp_t m = fp_add(n, n);
    fp_t w4 = fp_sqr(fp_sqr_nc(w));
    fp6 xx = fp6_sqr(X);
    fp6 num = fp6_add(fp6_dbl(xx), xx);
    num.c[0] = fp_add(num.c[0], w4);        // 3 X^2 + a w^4, a = 1
    fp_t m2 = fp_sqr_nc(m), m3 = fp_mul_nc(m2, m);
    fp6 A = fp6_scale(X, m2);
    fp6 L = fp6_mul(num, c);
    fp6 X3 = fp6_sub(fp6_sub(fp6_sqr(L), A), A);
    fp6 Y3 = fp6_sub(fp6_mul(L, fp6_sub(A, X3)), fp6_scale(Y, m3));
    p->X = X3;
    p->Y = Y3;
    p->w = fp_mul(m, w);
    return n == 0;
}

// Per-thread mode of an addition (data-dependent, evaluated with selects: control flow stays uniform)
enum jf_mode : uint8_t {
    JOP_NOP = 0,     // leave acc unchanged (the addend is the identity / a zero digit)
    JOP_ADD = 1,     // acc <- acc + src
    JOP_SUB = 2,     // acc <- acc - src
    JOP_SET = 3,     // acc <- src   (acc was the identity)
    JOP_SETNEG = 4,  // acc <- -src
};
SB_DEV uint8_t jf_add_mode(bool acc_empty, bool src_empty, bool neg) {
    return src_empty ? JOP_NOP : (acc_empty ? (neg ? JOP_SETNEG : JOP_SET) : (neg ? JOP_SUB : JOP_ADD));
}

// acc <- acc (+|-) src according to `mode`.  Returns true when an ACTIVE addition met x(acc) == x(src)
// (P + P or P - P): the fast path cannot represent / evaluate those and must be abandoned.
template <bool FUSED = false>
SB_DEV_NOINLINE bool jf_add(jf_pt* acc, const jf_pt* src, uint8_t mode) {
    fp6 X1 = acc->X, Y1 = acc->Y, X2 = src->X, Y2 = src->Y;
    fp_t w1 = acc->w, w2 = src->w;
    bool negate = mode == JOP_SUB || mode == JOP_SETNEG;
    fp_t w1s = fp_sqr_nc(w1), w1c = fp_mul_nc(w1s, w1), w2s = fp_sqr_nc(w2), w2c = fp_mul_nc(w2s, w2);
    fp6 d = fp6_scale_diff(X1, w2s, X2, w1s);    // U1 - U2,  U1 = X1 w2^2,  U2 = X2 w1^2
    fp6 c;
    fp_t n;
    bool wanted = mode == JOP_ADD || mode == JOP_SUB;
    bool set = mode == JOP_SET || mode == JOP_SETNEG;
    if (FUSED) {
        // S1 - (+|-) S2: the sign of src enters through the representative of -Y2 handed to the accumulation
        fp6 nY2;
#pragma unroll
        for (int i = 0; i < 6; i++) nY2.c[i] = negate ? Y2.c[i] : FP_P - Y2.c[i];
        fp6 num = fp6_scale_diff_nc(Y1, w2c, nY2, w1c);
        fp6_cof sl = fp6_slope_nc(num, d);
        fp6 L = sl.c;                                // slope = L / (n w1 w2)
        n = sl.n;
        fp_t n2 = fp_sqr_nc(n), n3 = fp_mul_nc(n2, n);
        fp6 A = fp6_scale(X1, fp_mul_nc(n2, w2s));   // n^2 U1 = x1 w3^2
        fp6 X3 = fp6_sqr_sub_scaled(L, A, X2, fp_mul_nc(n2, w1s));            // L^2 - x1 w3^2 - x2 w3^2
        fp6 Y3 = fp6_mul_sub_scaled(L, fp6_sub(A, X3), Y1, fp_mul_nc(n3, w2c));  // L (x1 w3^2 - X3) - y1 w3^3
        fp_t w3 = fp_mul(fp_mul_nc(n, w1), w2);
        if (wanted && n != 0) {  // on the exceptional input acc is left untouched
            acc->X = X3;
            acc->Y = Y3;
            acc->w = w3;
        } else if (set) {
            acc->X = X2;
#pragma unroll
            for (int i = 0; i < 6; i++) acc->Y.c[i] = negate ? fp_neg(Y2.c[i]) : Y2.c[i];
            acc->w = w2;
        }
        return wanted && n == 0;
    }
    if (negate) Y2 = fp6_neg(Y2);
    fp6 num = fp6_scale_diff(Y1, w2c, Y2, w1c);  // S1 - S2
    fp6_cofactor_norm(&d, &c, &n);
    fp6 L = fp6_mul(num, c);                     // slope = L / (n w1 w2)
    fp_t n2 = fp_sqr_nc(n), n3 = fp_mul_nc(n2, n);
    fp6 A = fp6_scale(X1, fp_mul_nc(n2, w2s));   // n^2 U1 = x1 w3^2
    fp6 B = fp6_scale(X2, fp_mul_nc(n2, w1s));   // n^2 U2 = x2 w3^2
    fp6 X3 = fp6_sub(fp6_sub(fp6_sqr(L), A), B);
    fp6 Y3 = fp6_sub(fp6_mul(L, fp6_sub(A, X3)), fp6_scale(Y1, fp_mul_nc(n3, w2c)));  // L (x1 w3^2 - X3) - y1 w3^3
    fp_t w3 = fp_mul(fp_mul_nc(n, w1), w2);
    bool active = wanted && n != 0;  // on the exceptional input acc is left untouched
#pragma unroll
    for (int i = 0; i < 6; i++) {
        acc->X.c[i] = active ? X3.c[i] : (set ? X2.c[i] : X1.c[i]);
        acc->Y.c[i] = active ? Y3.c[i] : (set ? Y2.c[i] : Y1.c[i]);
    }
    acc->w = active ? w3 : (set ? w2 : w1);
    return wanted && n == 0;
}

// acc <- acc (+|-) (x2, y2) for an AFFINE addend (denominator 1): the mixed form of jf_add<true> -- no powers of w2,
// U1 = X1 and S1 = Y1 need no scaling (14 base-field products less), the same lazily accumulated X3 / Y3.
// `acc` must be finite.  Returns true (acc untouched) when x(acc) == x2.
SB_DEV_NOINLINE bool jf_madd(jf_pt* acc, const jf_pt* t, bool neg) {
    fp6 X1 = acc->X, Y1 = acc->Y, X2 = t->X, Y2 = t->Y;
    fp_t w1 = acc->w;
    fp_t w1s = fp_sqr_nc(w1), w1c = fp_mul_nc(w1s, w1);
    fp6 d, num;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        wide_acc w;
        wide_set64(w, X1.c[i]);                       // U1 - U2 = X1 - x2 w1^2
        wide_mac(w, FP_P - X2.c[i], w1s);
        d.c[i] = wide_reduce(w);
        wide_set64(w, Y1.c[i]);                       // S1 - (+|-) S2 = Y1 -+ y2 w1^3
        wide_mac(w, neg ? Y2.c[i] : FP_P - Y2.c[i], w1c);
        num.c[i] = wide_reduce_nc(w);
    }
    fp_t n;
    fp6_cof sl = fp6_slope_nc(num, d);
    fp6 L = sl.c;                                     // slope = L / (n w1)
    n = sl.n;
    fp_t n2 = fp_sqr_nc(n), n3 = fp_mul_nc(n2, n);
    fp6 A = fp6_scale(X1, n2);                        // x1 w3^2
    fp6 X3 = fp6_sqr_sub_scaled(L, A, X2, fp_mul_nc(n2, w1s));
    fp6 Y3 = fp6_mul_sub_scaled(L, fp6_sub(A, X3), Y1, n3);
    if (n == 0) return true;
    acc->X = X3;
    acc->Y = Y3;
    acc->w = fp_mul(n, w1);
    return false;
}

// Exact accumulation for the Pippenger buckets (batch.cuh): acc += (+|-) t with t affine (t->w == 1).
// The identity is w == 0; P + P and P - P (repeated signers put equal points into one bucket,
// src/batch.rs:167-169) are resolved on a rarely taken branch.
SB_DEV void jf_madd_exact(jf_pt* acc, const jf_pt* t, bool neg) {
    if (acc->w == 0) {  // first point of the bucket
        acc->X = t->X;
        acc->Y = neg ? fp6_neg(t->Y) : t->Y;
        acc->w = 1;
        return;
    }
    bool exc = jf_madd(acc, t, neg);
    if (__builtin_expect(exc, 0)) {
        fp_t w = acc->w;
        fp6 ty = fp6_scale(neg ? fp6_neg(t->Y) : t->Y, fp_mul_nc(fp_sqr_nc(w), w));
        bool same = fp6_eq(acc->Y, ty);
        if (!same || jf_dbl(acc)) acc->w = 0;  // P - P, or the doubling of a 2-torsion point
    }
}

// a == b as points (both finite)
SB_DEV bool jf_eq_neg(const jf_pt& a, const jf_pt& b, bool& x_eq) {
    fp_t was = fp_sqr_nc(a.w), wbs = fp_sqr_nc(b.w);
    x_eq = fp6_eq(fp6_scale(a.X, wbs), fp6_scale(b.X, was));
    return x_eq && fp6_eq(fp6_scale(a.Y, fp_mul_nc(wbs, b.w)), fp6_neg(fp6_scale(b.Y, fp_mul_nc(was, a.w))));
}

// General exact addition acc += src of two (X, Y, w) points, either of which may be the identity (w == 0).
SB_DEV void jf_add_exact(jf_pt* acc, const jf_pt* src) {
    bool exc = jf_add(acc, src, jf_add_mode(acc->w == 0, src->w == 0, false));
    if (__builtin_expect(exc, 0)) {
        // x(acc) == x(src):  Y1 w2^3 == Y2 w1^3  <=>  the same point (doubling), otherwise opposite points
        fp_t w1 = acc->w, w2 = src->w;
        fp6 a = fp6_scale(acc->Y, fp_mul_nc(fp_sqr_nc(w2), w2)), b = fp6_scale(src->Y, fp_mul_nc(fp_sqr_nc(w1), w1));
        if (!fp6_eq(a, b) || jf_dbl(acc)) acc->w = 0;
    }
}
// acc <- 2 acc, exact (identity and 2-torsion points give the identity)
SB_DEV void jf_dbl_exact(jf_pt* acc) {
    if (acc->w == 0) return;
    if (jf_dbl(acc)) acc->w = 0;
}

enum fast_result : int {
    FAST_TORSION_FREE = 0,      // [q]P == O, h*P + e*G computed
    FAST_NOT_TORSION_FREE = 1,  // [q]P != O
    FAST_EXCEPTIONAL = 2,       // an exceptional case was met: use the exact routine
};

// [q]P == O ?  and  R = h*P + e*G, sharing the doubling chain D_j = 2^j P as torsion_check_and_mul does, in the
// (X, Y, w) coordinates above.  Caller-provided storage (shared memory in the kernels): `Dp` for D_j, and `Bh` for the
// buckets of the challenge digits of magnitude 1..FAST_BH_SHARED -- bucket b of this thread at Bh[b * bh_stride].  Those
// buckets are indexed by a PER-THREAD digit: in thread-local memory a warp's 32 accesses scatter over 32 different
// lines (ncu: 13 of 32 bytes per sector used, 7 GB of DRAM write-backs per 2^20 signatures, 5 % of the kernel time),
// in shared memory the 104-byte slots are conflict-free for 64-bit accesses whatever the bucket index is
// (bank = 26 tid + 2 k mod 32: sixteen distinct even banks per half-warp).  The buckets of the subgroup check are
// indexed by the constant digits of q -- warp-uniform, hence coalesced -- and stay in thread-local memory, as does the
// bucket of magnitude 8 (one digit in sixteen; two blocks of 128 threads x 8 slots fill the SM's shared memory).
// On FAST_TORSION_FREE / FAST_NOT_TORSION_FREE, *R is the result (never the identity: that is reported as exceptional).
// 7 shared buckets: 79.73 ms against 80.25 with 6 and 82.59 with 8 (profiles/r2_variants.md, v12).
static constexpr int FAST_BH_SHARED = 7;
SB_DEV int verify_core_fast(const fp6& px, const fp6& py, const scalar& h, const scalar& e,
                            const uint64_t* __restrict__ gtab, jf_pt* R, jf_pt* Dp, jf_pt* Bh, int bh_stride) {
    jf_pt Bq[8], Bhl[8 - FAST_BH_SHARED];
#define SB_BH(b) ((b) < FAST_BH_SHARED ? Bh + (size_t)(b) * bh_stride : &Bhl[(b) - FAST_BH_SHARED])
    int h_carry = 0;  // signed 4-bit digits of h are recoded on the fly (recode_signed_w4), least significant first
    scalar hs = h;    // shifted right by one nibble per window: a dynamically indexed h.l[j >> 5] would live in local memory
    uint32_t q_seen = 0, h_seen = 0;
    bool exc = false;
#pragma unroll 1
    for (int b = 0; b < 8; b++) {  // dummy (masked) operations read empty buckets: give them defined contents
        Bq[b] = jf_pt{fp6_zero(), fp6_zero(), 1};
        *SB_BH(b) = Bq[b];
    }
    Dp->X = px;
    Dp->Y = py;
    Dp->w = 1;
#pragma unroll 1
    for (int j = 0; j < SB_CHAIN_STEPS; j++) {
        SB_PHASE_SYNC();  // every step: 77.45 against 77.80 ms every 4th (profiles/r2_variants.md, v14)
        int dq = SB_QWNAF(j);
        if (dq != 0) {  // warp-uniform
            int idx = (dq < 0 ? -dq : dq) >> 1;
            if ((q_seen >> idx) & 1) {
                exc |= jf_add<true>(&Bq[idx], Dp, dq < 0 ? JOP_SUB : JOP_ADD);
            } else {  // first digit of this bucket: a copy (warp-uniform, q is a constant)
                Bq[idx] = *Dp;
                if (dq < 0) Bq[idx].Y = fp6_neg(Bq[idx].Y);
                q_seen |= 1u << idx;
            }
        }
        if ((j & 3) == 0) {
            int raw = (int)(hs.l[0] & 15) + h_carry;   // j = 4 i: nibble i of h
#pragma unroll
            for (int k = 0; k < 7; k++) hs.l[k] = (hs.l[k] >> 4) | (hs.l[k + 1] << 28);
            hs.l[7] >>= 4;
            h_carry = raw > 8;
            int dh = h_carry ? raw - 16 : raw;
            int mag = dh < 0 ? -dh : dh;
            int idx = mag ? mag - 1 : 0;
            exc |= jf_add<true>(SB_BH(idx), Dp, jf_add_mode(!((h_seen >> idx) & 1), mag == 0, dh < 0));
            if (mag) h_seen |= 1u << idx;
        }
        if (j < SB_CHAIN_STEPS - 1) exc |= jf_dbl<true>(Dp);
    }
    // Bucket aggregation (R_k = sum_{m>=k} B_m, O_k = sum_{m>=k} R_m):
    //   q (odd digits 2k+1):  [q]P = 2 O_1 + R_0        h (digits m = k+1):  h*P = O_0
    // The running sums R live IN PLACE in the top buckets and O_h in the caller's result slot: no extra copies in
    // thread-local memory (the buckets are not needed any more once they have been folded in).
    jf_pt* Rq = &Bq[7];
    jf_pt* Rh = SB_BH(7);
    jf_pt* Oh = R;
    jf_pt& Oq = *Dp;   // the chain is over: its slot (shared memory, what jf_dbl<true> expects) holds O_q from here on
    Oq = Bq[7];
    *Oh = *Rh;
    bool eRq = !((q_seen >> 7) & 1), eOq = eRq, eRh = !((h_seen >> 7) & 1), eOh = eRh;
    // `same_h`: O_h and R_h are the same (finite) point.  It happens whenever the buckets below the highest used
    // digit magnitude are empty (~2e-4 of random challenges): O += R is then a doubling, taken on a divergent
    // branch by those few threads instead of being handed to the exact kernel.
    bool same_h = !eRh;
#pragma unroll 1
    for (int b = 6; b >= 0; b--) {
        SB_PHASE_SYNC();
        bool eb = !((q_seen >> b) & 1);
        exc |= jf_add<true>(Rq, &Bq[b], jf_add_mode(eRq, eb, false));
        eRq = eRq && eb;
        if (b >= 1) {
            exc |= jf_add<true>(&Oq, Rq, jf_add_mode(eOq, eRq, false));
            eOq = eOq && eRq;
        }
        eb = !((h_seen >> b) & 1);
        exc |= jf_add<true>(Rh, SB_BH(b), jf_add_mode(eRh, eb, false));
        if (!eb && !eRh) same_h = false;  // a real addition changed R
        eRh = eRh && eb;
        if (__builtin_expect(same_h && !eOh, 0)) {
            jf_pt keep = Oq;                   // O == R: O + R = 2 O, doubled through the shared slot
            Oq = *Oh;
            exc |= jf_dbl<true>(&Oq);
            *Oh = Oq;
            Oq = keep;
            same_h = false;
        } else {
            exc |= jf_add<true>(Oh, Rh, jf_add_mode(eOh, eRh, false));
            same_h = eOh && !eRh;         // O was empty and has just been set to R
        }
        eOh = eOh && eRh;
    }
    if (eOq || eRq) exc = true;  // degenerate digit pattern: leave it to the exact routine
    else exc |= jf_dbl<true>(&Oq);
    // [q]P = 2 O_1 + R_0 is the identity  <=>  2 O_1 == -R_0
    bool x_eq;
    bool torsion_free = jf_eq_neg(Oq, *Rq, x_eq);
    if (x_eq && !torsion_free) exc = true;  // 2 O_1 == R_0: a doubling the fast path does not evaluate

    // + e*G: 20 table points (affine, w = 1) added to h*P (which already sits in *R)
    bool e_acc = eOh;
    {
        int carry = 0;
        jf_pt T;
        T.w = 1;
#pragma unroll 1
        for (int i = 0; i < GTAB_WINDOWS; i++) {
            if ((i & 3) == 0) SB_PHASE_SYNC();
            int raw = (int)sc_bits(e, GTAB_W * i, GTAB_W) + carry;
            bool neg = raw > (1 << (GTAB_W - 1));
            carry = neg ? 1 : 0;
            int dg = neg ? (1 << GTAB_W) - raw : raw;
            const uint64_t* ent = gtab + ((size_t)i * GTAB_ENTRIES + (dg ? dg : 1)) * GTAB_ENTRY_U64;
#if defined(__CUDA_ARCH__)
            const ulonglong2* e2 = reinterpret_cast<const ulonglong2*>(ent);
            ulonglong2 a = e2[0], b = e2[1], c = e2[2], dd = e2[3], ee = e2[4], f = e2[5];
            T.X = fp6{{a.x, a.y, b.x, b.y, c.x, c.y}};
            T.Y = fp6{{dd.x, dd.y, ee.x, ee.y, f.x, f.y}};
#else
            for (int c = 0; c < 6; c++) {
                T.X.c[c] = ent[c];
                T.Y.c[c] = ent[6 + c];
            }
#endif
            exc |= jf_add<true>(R, &T, jf_add_mode(e_acc, dg == 0, neg));
            e_acc = e_acc && dg == 0;
        }
    }
    if (e_acc) exc = true;  // the result is the identity: exact routine
#undef SB_BH
    if (exc) return FAST_EXCEPTIONAL;
    return torsion_free ? FAST_TORSION_FREE : FAST_NOT_TORSION_FREE;
}

}  // namespace sb
