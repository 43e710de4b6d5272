// Cheetah curve  y^2 = x^3 + x + (u + 395)  over Fp6 (reference README.md:4-8; `cheetah::AffinePoint`
// / `ProjectivePoint`, call sites src/signature.rs:182,196-200, src/batch.rs:98-123).
//
// Jacobian coordinates (X, Y, Z), x = X/Z^2, y = Y/Z^3, identity <=> Z = 0.  The verification
// result is compared through its affine x only (src/signature.rs:200), so any algorithm producing
// the same group element is bit-exact after normalisation.
//
// The exceptional inputs (identity operands, P + P, P + (-P)) are handled exactly, on rarely taken
// branches, because adversarial public keys of small order DO reach them (the reference's own test
// uses an off-subgroup key, src/signature.rs:385-406).
//
// Code-size discipline: the hot loops call ONE out-of-line copy each of jac_dbl_mem / jac_add_mem /
// jac_madd_mem (operating on points held in thread-local memory), which in turn call one copy of
// fp6_mul / fp6_sqr: small instruction-cache footprint, and no point pins 36 registers across calls.
#pragma once
#include "fp6.cuh"
#include "scalar.cuh"

namespace sb {

struct jac_pt {
    fp6 X, Y, Z;
};

SB_DEV jac_pt jac_identity() { return jac_pt{fp6_one(), fp6_one(), fp6_zero()}; }
SB_DEV bool jac_is_identity(const jac_pt& p) { return fp6_is_zero(p.Z); }
SB_DEV jac_pt jac_from_affine(const fp6& x, const fp6& y, bool inf) {
    jac_pt r{x, y, fp6_one()};
    if (inf) r = jac_identity();
    return r;
}

// dbl-2007-bl with a = 1: 1M + 8S.  Complete: Z = 0 or Y = 0 (order-2 point) both give Z3 = 0.
SB_DEV jac_pt jac_dbl(const jac_pt& p) {
    fp6 XX = fp6_sqr(p.X);
    fp6 YY = fp6_sqr(p.Y);
    fp6 YYYY = fp6_sqr(YY);
    fp6 ZZ = fp6_sqr(p.Z);
    fp6 t = fp6_sqr(fp6_add(p.X, YY));
    fp6 S = fp6_dbl(fp6_sub(fp6_sub(t, XX), YYYY));
    fp6 M = fp6_add(fp6_add(fp6_dbl(XX), XX), fp6_sqr(ZZ));
    jac_pt r;
    r.X = fp6_sub(fp6_sqr(M), fp6_dbl(S));
    fp6 y8 = fp6_dbl(fp6_dbl(fp6_dbl(YYYY)));
    r.Y = fp6_sub(fp6_mul(M, fp6_sub(S, r.X)), y8);
    r.Z = fp6_sub(fp6_sub(fp6_sqr(fp6_add(p.Y, p.Z)), YY), ZZ);
    return r;
}

// add-2007-bl: 11M + 5S.  `same` is set (and p returned) when p == q: the caller doubles instead -- kept
// out of this function so that the rare case does not drag a second copy of the doubling code along.
SB_DEV jac_pt jac_add_core(const jac_pt& p, const jac_pt& q, bool& same) {
    same = false;
    bool p_inf = fp6_is_zero(p.Z), q_inf = fp6_is_zero(q.Z);
    if (p_inf | q_inf) return p_inf ? q : p;  // rare
    fp6 Z1Z1 = fp6_sqr(p.Z);
    fp6 Z2Z2 = fp6_sqr(q.Z);
    fp6 U1 = fp6_mul(p.X, Z2Z2);
    fp6 U2 = fp6_mul(q.X, Z1Z1);
    fp6 S1 = fp6_mul(fp6_mul(p.Y, q.Z), Z2Z2);
    fp6 S2 = fp6_mul(fp6_mul(q.Y, p.Z), Z1Z1);
    fp6 H = fp6_sub(U2, U1);
    fp6 rr = fp6_sub(S2, S1);
    if (fp6_is_zero(H)) {  // rare: same x
        same = fp6_is_zero(rr);
        return same ? p : jac_identity();
    }
    fp6 I = fp6_sqr(fp6_dbl(H));
    fp6 J = fp6_mul(H, I);
    fp6 r2 = fp6_dbl(rr);
    fp6 V = fp6_mul(U1, I);
    jac_pt r;
    r.X = fp6_sub(fp6_sub(fp6_sqr(r2), J), fp6_dbl(V));
    r.Y = fp6_sub(fp6_mul(r2, fp6_sub(V, r.X)), fp6_dbl(fp6_mul(S1, J)));
    r.Z = fp6_mul(fp6_sub(fp6_sub(fp6_sqr(fp6_add(p.Z, q.Z)), Z1Z1), Z2Z2), H);
    return r;
}

SB_DEV jac_pt jac_add(const jac_pt& p, const jac_pt& q) {
    bool same;
    jac_pt r = jac_add_core(p, q, same);
    return same ? jac_dbl(p) : r;
}

// madd-2007-bl (q affine): 7M + 4S
SB_DEV jac_pt jac_madd_core(const jac_pt& p, const fp6& qx, const fp6& qy, bool q_inf, bool& same) {
    same = false;
    if (q_inf) return p;
    if (fp6_is_zero(p.Z)) return jac_pt{qx, qy, fp6_one()};
    fp6 Z1Z1 = fp6_sqr(p.Z);
    fp6 U2 = fp6_mul(qx, Z1Z1);
    fp6 S2 = fp6_mul(fp6_mul(qy, p.Z), Z1Z1);
    fp6 H = fp6_sub(U2, p.X);
    fp6 rr = fp6_sub(S2, p.Y);
    if (fp6_is_zero(H)) {  // rare: same x
        same = fp6_is_zero(rr);
        return same ? p : jac_identity();
    }
    fp6 HH = fp6_sqr(H);
    fp6 I = fp6_dbl(fp6_dbl(HH));
    fp6 J = fp6_mul(H, I);
    fp6 r2 = fp6_dbl(rr);
    fp6 V = fp6_mul(p.X, I);
    jac_pt r;
    r.X = fp6_sub(fp6_sub(fp6_sqr(r2), J), fp6_dbl(V));
    r.Y = fp6_sub(fp6_mul(r2, fp6_sub(V, r.X)), fp6_dbl(fp6_mul(p.Y, J)));
    r.Z = fp6_sub(fp6_sub(fp6_sqr(fp6_add(p.Z, H)), Z1Z1), HH);
    return r;
}

SB_DEV jac_pt jac_madd(const jac_pt& p, const fp6& qx, const fp6& qy, bool q_inf) {
    bool same;
    jac_pt r = jac_madd_core(p, qx, qy, q_inf, same);
    return same ? jac_dbl(p) : r;
}

// ---- out-of-line, in-memory forms used by every loop -------------------------------------------
SB_DEV_NOINLINE void jac_dbl_mem(jac_pt* p) { *p = jac_dbl(*p); }
SB_DEV_NOINLINE void jac_add_mem(jac_pt* acc, const jac_pt* q, bool q_neg) {
    jac_pt t = *q;
    if (q_neg) t.Y = fp6_neg(t.Y);
    // (the rare P + P case is inlined here on purpose: measured 2 % faster in k_verify than calling
    // jac_dbl_mem, while the mixed addition below is 14 % faster with the out-of-line form)
    *acc = jac_add(*acc, t);
}
// affine operand read from a table of 12 x u64 entries (x || y)
SB_DEV_NOINLINE void jac_madd_mem(jac_pt* acc, const uint64_t* __restrict__ ent, bool q_neg, bool q_skip) {
    fp6 qx, qy;
#if defined(__CUDA_ARCH__)
    const ulonglong2* e2 = reinterpret_cast<const ulonglong2*>(ent);
    ulonglong2 a = e2[0], b = e2[1], c = e2[2], d = e2[3], e = e2[4], f = e2[5];
    qx = fp6{{a.x, a.y, b.x, b.y, c.x, c.y}};
    qy = fp6{{d.x, d.y, e.x, e.y, f.x, f.y}};
#else
    for (int k = 0; k < 6; k++) {
        qx.c[k] = ent[k];
        qy.c[k] = ent[6 + k];
    }
#endif
    if (q_neg) qy = fp6_neg(qy);
    bool same;
    *acc = jac_madd_core(*acc, qx, qy, q_skip, same);
    if (__builtin_expect(same, 0)) jac_dbl_mem(acc);  // rare: P + P
}

SB_DEV void jac_to_affine(const jac_pt& p, fp6& x, fp6& y, bool& inf) {
    inf = fp6_is_zero(p.Z);
    fp6 zi = fp6_inv(p.Z);  // 0 for the identity -> x = y = 0
    fp6 zi2 = fp6_sqr(zi);
    x = fp6_mul(p.X, zi2);
    y = fp6_mul(p.Y, fp6_mul(zi2, zi));
}
// X == x * Z^2 without an inversion (final comparison of verify); the identity reads as x = 0
// (SURVEY.md §8 a9), so it compares equal to x = 0 only.
SB_DEV bool jac_x_equals(const jac_pt& p, const fp6& x) {
    if (fp6_is_zero(p.Z)) return fp6_is_zero(x);
    return fp6_eq(p.X, fp6_mul(x, fp6_sqr(p.Z)));
}

#if defined(__CUDACC__)
__constant__ int8_t c_q_wnaf5[256];  // CHEETAH_Q_WNAF5, filled at context creation
#define SB_QWNAF(i) c_q_wnaf5[i]
#else
#define SB_QWNAF(i) CHEETAH_Q_WNAF5[i]
#endif

// Fixed-base table of G (the reference's BASEPOINT_TABLE): signed 13-bit windows,
//   gtab[i][d] = d * 2^(13 i) * G   (affine x || y, 12 x u64),  i < 20,  1 <= d <= 4096  (slot 0 unused)
// 20 x 4097 x 96 B = 7.9 MB, L2 resident.  k = sum_i d_i 2^(13 i) with d_i in [-4096, 4096].
static constexpr int GTAB_ENTRY_U64 = 12;
static constexpr int GTAB_W = 13;
static constexpr int GTAB_WINDOWS = 20;
static constexpr int GTAB_ENTRIES = (1 << (GTAB_W - 1)) + 1;  // 4097

// acc += k * G: 20 mixed additions, no doublings
SB_DEV void fixed_base_accumulate(jac_pt* acc, const scalar& k, const uint64_t* __restrict__ gtab) {
    int carry = 0;
#pragma unroll 1
    for (int i = 0; i < GTAB_WINDOWS; i++) {
        int raw = (int)sc_bits(k, GTAB_W * i, GTAB_W) + carry;
        bool neg = raw > (1 << (GTAB_W - 1));
        carry = neg ? 1 : 0;
        int d = neg ? (1 << GTAB_W) - raw : raw;
        jac_madd_mem(acc, gtab + ((size_t)i * GTAB_ENTRIES + (d ? d : 1)) * GTAB_ENTRY_U64, neg, d == 0);
    }
}

// k*G (BASEPOINT_TABLE * scalar: src/public.rs:29, src/signature.rs:67,116, src/batch.rs:98-100)
SB_DEV jac_pt fixed_base_mul(const scalar& k, const uint64_t* __restrict__ gtab) {
    jac_pt acc = jac_identity();
    fixed_base_accumulate(&acc, k, gtab);
    return acc;
}

// ---------------------------------------------------------------------------------------------
// Shared-doubling ("Yao" / bucket) evaluation of the two variable-base products of a verification:
// the subgroup check [q]P and the challenge product h*P use the SAME chain D_i = 16^i P
// (252 doublings instead of 2 x 254), each scalar in signed 4-bit windows d_i in [-8, 8]:
//     B[|d_i|] += sign(d_i) * D_i        then        k*P = sum_{m=1..8} m * B[m]   (14 additions)
// q's digits are constants (warp-uniform additions); h's digits are per thread.
// q is taken in its width-5 NAF, 8 buckets of odd multiples (44 + 14 additions): 7.84 against 7.74 M/s at width 4
// (profiles/r1_variants.md).
static constexpr int SB_Q_BUCKETS = 8;
// Steps of the shared doubling chain D_j = 2^j P: the last 4-bit window of the challenge starts at bit 252, and the
// generated width-5 digits of q end at bit 251 (tools/gen_params.py: fold_top), so D_253..D_255 are never needed.
static constexpr int SB_CHAIN_STEPS = 253;
static_assert(CHEETAH_Q_WNAF5_LEN <= SB_CHAIN_STEPS, "digits of q above the last challenge window");

// Keeping the warps of a block in the same phase of the loop lets them share instruction-cache lines
// (the point routines are ~4k instructions, larger than the cache): a block barrier per point
// operation, +11 % on k_verify (profiles/r1_variants.md).  Exited threads do not take part in barriers, divergent
// branches contain none.
#if defined(__CUDA_ARCH__)
#define SB_PHASE_SYNC() __syncthreads()
#else
#define SB_PHASE_SYNC() do { } while (0)
#endif

// k < 2^255  ->  64 signed digits, k = sum d_i 16^i, |d_i| <= 8
SB_DEV void recode_signed_w4(const scalar& k, int8_t* d /*64*/) {
    int carry = 0;
#pragma unroll 1
    for (int i = 0; i < 64; i++) {
        int raw = (int)((k.l[i >> 3] >> (4 * (i & 7))) & 15) + carry;
        carry = raw > 8;
        d[i] = (int8_t)(carry ? raw - 16 : raw);
    }
}
// out = sum_{m=1..8} m * B[m-1]
SB_DEV void bucket_aggregate(const jac_pt* B, jac_pt* out) {
    jac_pt running = B[7];
    *out = B[7];
#pragma unroll 1
    for (int m = 6; m >= 0; m--) {
        jac_add_mem(&running, &B[m], false);
        jac_add_mem(out, &running, false);
    }
}
// out = sum_{k<nb} (2k+1) * B[k]  =  2 * sum k B[k] + sum B[k]      (2 nb - 3 additions + 1 doubling)
SB_DEV void bucket_aggregate_odd(const jac_pt* B, int nb, jac_pt* out) {
    jac_pt running = B[nb - 1];
    *out = B[nb - 1];
#pragma unroll 1
    for (int k = nb - 2; k >= 1; k--) {
        jac_add_mem(&running, &B[k], false);
        jac_add_mem(out, &running, false);
    }
    jac_add_mem(&running, &B[0], false);
    jac_dbl_mem(out);
    jac_add_mem(out, &running, false);
}
// returns [q]P == O (AffinePoint::is_torsion_free, src/signature.rs:182) and writes h*P.
// One doubling chain D_j = 2^j P, j = 0..SB_CHAIN_STEPS-1.  q is consumed in its constant width-w NAF (non-zero odd
// digits at arbitrary bit positions -> 2^(w-2) buckets of odd multiples, warp-uniform control flow);
// h in signed 4-bit windows at every fourth step (per-thread digits, uniform trip count).
// `Dp` is caller-provided storage for the running point D_j (the kernels place it in shared memory: it is
// touched by every doubling and every addition, i.e. 70 % of the thread-local traffic).
SB_DEV bool torsion_check_and_mul(const jac_pt& P, const scalar& h, jac_pt* hP, jac_pt* Dp) {
    jac_pt Bq[SB_Q_BUCKETS], Bh[8];
#pragma unroll 1
    for (int b = 0; b < 8; b++) Bh[b] = jac_identity();
#pragma unroll 1
    for (int b = 0; b < SB_Q_BUCKETS; b++) Bq[b] = jac_identity();
    int8_t hd[64];
    recode_signed_w4(h, hd);
    *Dp = P;
#pragma unroll 1
    for (int j = 0; j < SB_CHAIN_STEPS; j++) {
        if ((j & 3) == 0) SB_PHASE_SYNC();
        if (j != 0) jac_dbl_mem(Dp);
        int dq = SB_QWNAF(j);
        if (dq != 0) jac_add_mem(&Bq[(dq < 0 ? -dq : dq) >> 1], Dp, dq < 0);  // warp-uniform
        if ((j & 3) == 0) {
            int dh = hd[j >> 2];
            if (dh != 0) jac_add_mem(&Bh[(dh < 0 ? -dh : dh) - 1], Dp, dh < 0);
        }
    }
    jac_pt tq;
    bucket_aggregate_odd(Bq, SB_Q_BUCKETS, &tq);
    bucket_aggregate(Bh, hP);
    return jac_is_identity(tq);
}

// AffinePoint::from_compressed (src/batch.rs:104, src/public.rs:55): 48 bytes of x + flag byte
// (bit 7 infinity, bit 6 "y is the lexicographically largest root", other bits must be 0).
// x arrives already split into limbs; returns false when the record does not decode.
SB_DEV bool decompress_point(const fp6& x, uint8_t flags, fp6& ox, fp6& oy, bool& inf) {
    ox = fp6_zero();
    oy = fp6_zero();
    inf = true;
    if (flags & 0x3f) return false;
    if (!fp6_is_canonical(x)) return false;
    bool f_inf = (flags >> 7) & 1, f_sign = (flags >> 6) & 1;
    if (f_inf) return fp6_is_zero(x) && !f_sign;
    fp6 rhs = fp6_add(fp6_mul(fp6_sqr(x), x), x);
    rhs.c[0] = fp_add(rhs.c[0], 395);
    rhs.c[1] = fp_add(rhs.c[1], 1);
    fp6 y;
    if (!fp6_sqrt(rhs, y)) return false;
    if (fp6_lex_largest(y) != f_sign) y = fp6_neg(y);
    ox = x;
    oy = y;
    inf = false;
    return true;
}
// AffinePoint::to_compressed flag byte
SB_DEV uint8_t compress_flags(const fp6& y, bool inf) { return inf ? 0x80 : (fp6_lex_largest(y) ? 0x40 : 0x00); }

}  // namespace sb
