// Warp-cooperative ("distributed") verification for SMALL calls: one signature per group of six lanes.
//
// The throughput kernel (k_verify_fast) runs one signature per thread: ~1.6 M dependent instructions, i.e. ~2 ms
// of latency however few signatures a call holds, and it needs ~38 k signatures to fill a B200.  Here an Fp6 value
// is DISTRIBUTED over six lanes (lane k holds coefficient k), so that a product is one coefficient per lane (six
// 64x64 products and one reduction) with the operands exchanged by warp shuffles, the Fp3 steps of the
// cofactor/norm computation run on the two 3-lane halves side by side, the 12-element Rescue state is held two
// elements per lane, and everything coefficient-wise (additions, scalings by Fp elements, selects) is one
// operation per lane.  Same algorithm, coordinates, exceptional-case policy and verdicts as affine.cuh /
// verify_points_fast; ~4x shorter dependency chain and 6x more parallelism for a given number of signatures, at
// ~1.5x the total instruction count (replicated scalar work, shuffles) -- which is why large calls keep the
// one-signature-per-thread kernel.
//
// All shuffles name only the six lanes of the group in their mask, so the groups of a warp are independent
// (different message lengths -> different trip counts in the hash).  Device-only code (no host build).
#pragma once
#include "verify.cuh"

namespace sb {

__device__ __forceinline__ fp_t dshfl(unsigned mask, fp_t v, int src) { return __shfl_sync(mask, v, src); }

// coefficient k of a * b in Fp6; a, b = the lane's coefficients of the two operands.  Step i: lane k needs a_i and
// b'_(k - i mod 6); the source lane j is read by lane (j + i) mod 6, which wraps (needs 7 b_j) iff j + i >= 6.
__device__ __noinline__ fp_t dfp6_mul(unsigned mask, fp_t a, fp_t b, int k, int gbase) {
    fp_t b7 = fp_mul7_nc(b);
    wide_acc w;
    wide_zero(w);
#pragma unroll
    for (int i = 0; i < 6; i++) {
        fp_t send = (k + i >= 6) ? b7 : b;
        int j = k - i;
        j += j < 0 ? 6 : 0;
        wide_mac(w, dshfl(mask, a, gbase + i), dshfl(mask, send, gbase + j));
    }
    return wide_reduce(w);
}
// Fp3 = Fp[v]/(v^3 - 7) products on the two 3-lane halves of a group at once: lanes of parity `par` hold the
// coefficients t = k >> 1 of one Fp3 operand pair (even lanes: the c0,c2,c4 part of an Fp6 value, odd: c1,c3,c5)
__device__ __noinline__ fp_t dfp3_mul(unsigned mask, fp_t a, fp_t b, int k, int gbase) {
    int par = k & 1, t = k >> 1;
    fp_t b7 = fp_mul7_nc(b);
    wide_acc w;
    wide_zero(w);
#pragma unroll
    for (int i = 0; i < 3; i++) {
        fp_t send = (t + i >= 3) ? b7 : b;
        int j = t - i;
        j += j < 0 ? 3 : 0;
        wide_mac(w, dshfl(mask, a, gbase + 2 * i + par), dshfl(mask, send, gbase + 2 * j + par));
    }
    return wide_reduce(w);
}
__device__ __forceinline__ bool dall(unsigned mask, int gbase, bool v) {
    return ((__ballot_sync(mask, v) >> gbase) & 0x3fu) == 0x3fu;
}

// d * c = n (fp6_cofactor_norm of affine.cuh): e = the lane's coefficient of d; returns the lane's coefficient of c
// and the norm n (replicated)
__device__ __noinline__ fp_t dfp6_cofactor_norm(unsigned mask, fp_t e, int k, int gbase, fp_t* n_out) {
    int par = k & 1, t = k >> 1;
    fp_t s = dfp3_mul(mask, e, e, k, gbase);  // even lanes: (a0^2)_t, odd lanes: (a1^2)_t
    // N = a0^2 - v a1^2,  (v x)_t = x_(t-1), times 7 for t = 0; computed by both halves (replicated)
    int tm = t == 0 ? 2 : t - 1;
    fp_t s0 = dshfl(mask, s, gbase + 2 * t), s1 = dshfl(mask, s, gbase + 2 * tm + 1);
    fp_t s1_7 = fp_mul7(s1);
    fp_t N = fp_sub(s0, t == 0 ? s1_7 : s1);
    fp_t d0 = dshfl(mask, N, gbase), d1 = dshfl(mask, N, gbase + 2), d2 = dshfl(mask, N, gbase + 4);
    fp_t d1_7 = fp_mul7_nc(d1), d2_7 = fp_mul7_nc(d2);
    // adjugate: t0 = d0^2 - 7 d1 d2,  t1 = 7 d2^2 - d0 d1,  t2 = d1^2 - d0 d2   (operands picked by selects)
    fp_t x = t == 0 ? d0 : (t == 1 ? d2 : d1);
    fp_t xp = t == 0 ? d0 : (t == 1 ? d2_7 : d1);
    fp_t y = FP_P - (t == 0 ? d1 : d0);
    fp_t yp = t == 0 ? d2_7 : (t == 1 ? d1 : d2);
    wide_acc w;
    wide_zero(w);
    wide_mac(w, x, xp);
    wide_mac(w, y, yp);
    fp_t adj = wide_reduce(w);
    fp_t a0 = dshfl(mask, adj, gbase), a1 = dshfl(mask, adj, gbase + 2), a2 = dshfl(mask, adj, gbase + 4);
    wide_zero(w);
    wide_mac(w, d0, a0);
    wide_mac(w, d2_7, a1);
    wide_mac(w, d1_7, a2);
    *n_out = wide_reduce(w);
    // c = (a0 - a1 u) * adj
    fp_t r = dfp3_mul(mask, e, adj, k, gbase);
    return par ? fp_neg(r) : r;
}

struct dpt {  // the lane's coefficients of X and Y; w (in Fp) replicated
    fp_t X, Y, w;
};

// p <- 2 p (jf_dbl of affine.cuh); returns true on a 2-torsion point
__device__ __noinline__ bool djf_dbl(unsigned mask, dpt* p, int k, int gbase) {
    fp_t X = p->X, Y = p->Y, w = p->w, n;
    fp_t c = dfp6_cofactor_norm(mask, Y, k, gbase, &n);
    fp_t m = fp_add(n, n);
    fp_t w4 = fp_sqr(fp_sqr_nc(w));
    fp_t xx = dfp6_mul(mask, X, X, k, gbase);
    fp_t num = fp_add(fp_dbl(xx), xx);
    num = fp_add(num, k == 0 ? w4 : 0);
    fp_t L = dfp6_mul(mask, num, c, k, gbase);
    fp_t m2 = fp_sqr_nc(m), m3 = fp_mul_nc(m2, m);
    fp_t A = fp_mul(X, m2);
    fp_t X3 = fp_sub(fp_sub(dfp6_mul(mask, L, L, k, gbase), A), A);
    fp_t Y3 = fp_sub(dfp6_mul(mask, L, fp_sub(A, X3), k, gbase), fp_mul(Y, m3));
    p->X = X3;
    p->Y = Y3;
    p->w = fp_mul(m, w);
    return n == 0;
}

// acc <- acc (+|-) src by mode (jf_add of affine.cuh)
__device__ __noinline__ bool djf_add(unsigned mask, dpt* acc, const dpt* src, uint8_t mode, int k, int gbase) {
    fp_t X1 = acc->X, Y1 = acc->Y, w1 = acc->w, X2 = src->X, Y2 = src->Y, w2 = src->w;
    if (mode == JOP_SUB || mode == JOP_SETNEG) Y2 = fp_neg(Y2);
    fp_t w1s = fp_sqr_nc(w1), w1c = fp_mul_nc(w1s, w1), w2s = fp_sqr_nc(w2), w2c = fp_mul_nc(w2s, w2);
    wide_acc wa;
    wide_zero(wa);
    wide_mac(wa, X1, w2s);
    wide_mac(wa, FP_P - X2, w1s);
    fp_t d = wide_reduce(wa);
    wide_zero(wa);
    wide_mac(wa, Y1, w2c);
    wide_mac(wa, FP_P - Y2, w1c);
    fp_t num = wide_reduce(wa);
    fp_t n;
    fp_t c = dfp6_cofactor_norm(mask, d, k, gbase, &n);
    fp_t L = dfp6_mul(mask, num, c, k, gbase);
    fp_t n2 = fp_sqr_nc(n), n3 = fp_mul_nc(n2, n);
    fp_t A = fp_mul(X1, fp_mul_nc(n2, w2s));
    fp_t B = fp_mul(X2, fp_mul_nc(n2, w1s));
    fp_t X3 = fp_sub(fp_sub(dfp6_mul(mask, L, L, k, gbase), A), B);
    fp_t Y3 = fp_sub(dfp6_mul(mask, L, fp_sub(A, X3), k, gbase), fp_mul(Y1, fp_mul_nc(n3, w2c)));
    fp_t w3 = fp_mul(fp_mul_nc(n, w1), w2);
    bool wanted = mode == JOP_ADD || mode == JOP_SUB;
    bool active = wanted && n != 0;
    bool set = mode == JOP_SET || mode == JOP_SETNEG;
    acc->X = active ? X3 : (set ? X2 : X1);
    acc->Y = active ? Y3 : (set ? Y2 : Y1);
    acc->w = active ? w3 : (set ? w2 : w1);
    return wanted && n == 0;
}

// Exact forms for the reduction stages of the batch MSM (batch.cuh): the identity is w == 0; P + P and P - P are
// resolved on a rarely taken, group-uniform branch (jf_add_exact / jf_dbl_exact of affine.cuh).
__device__ __forceinline__ void djf_dbl_exact(unsigned mask, dpt* p, int k, int gbase) {
    if (p->w == 0) return;
    if (djf_dbl(mask, p, k, gbase)) p->w = 0;
}
__device__ __forceinline__ void djf_add_exact(unsigned mask, dpt* acc, const dpt* src, int k, int gbase) {
    bool exc = djf_add(mask, acc, src, jf_add_mode(acc->w == 0, src->w == 0, false), k, gbase);
    if (__builtin_expect(exc, 0)) {  // x(acc) == x(src): the same point (doubling) or opposite points (identity)
        fp_t w1 = acc->w, w2 = src->w;
        bool same = dall(mask, gbase,
                         fp_mul(acc->Y, fp_mul_nc(fp_sqr_nc(w2), w2)) == fp_mul(src->Y, fp_mul_nc(fp_sqr_nc(w1), w1)));
        if (!same || djf_dbl(mask, acc, k, gbase)) acc->w = 0;
    }
}

// ---- Rescue-Prime with the state held two elements per lane: lane k has s[k] (lo) and s[k + 6] (hi) ----
// y = M s + ark: every lane gathers the 12 inputs by shuffles and forms its two rows of the circulant matrix;
// `mds2` = the MDS row twice (shared memory): M[i][j] = row[(j - i) mod 12] = mds2[j - i + 12]
__device__ __forceinline__ void drescue_mds_ark(unsigned mask, fp_t& lo, fp_t& hi, int ark_row, int k, int gbase,
                                                const uint32_t* mds2) {
    uint64_t alo = 0, ahi = 0, blo = 0, bhi = 0;  // rows k (a) and k + 6 (b): low / high input halves, no carries
#pragma unroll
    for (int j = 0; j < 12; j++) {
        fp_t v = dshfl(mask, j < 6 ? lo : hi, gbase + (j % 6));
        uint32_t ma = mds2[j - k + 12], mb = mds2[j - k + 6];
        alo += (uint64_t)(uint32_t)v * ma;
        ahi += (v >> 32) * ma;
        blo += (uint64_t)(uint32_t)v * mb;
        bhi += (v >> 32) * mb;
    }
    uint64_t mid = (alo >> 32) + ahi;
    lo = fp_add(fp_reduce96((uint32_t)alo, (uint32_t)mid, (uint32_t)(mid >> 32)), SB_ARK(ark_row * 12 + k));
    mid = (blo >> 32) + bhi;
    hi = fp_add(fp_reduce96((uint32_t)blo, (uint32_t)mid, (uint32_t)(mid >> 32)), SB_ARK(ark_row * 12 + k + 6));
}
__device__ __noinline__ void drescue_permutation(unsigned mask, fp_t* lo_hi, int k, int gbase, const uint32_t* mds2) {
    fp_t s[2] = {lo_hi[0], lo_hi[1]};
#pragma unroll 1
    for (int r = 0; r < RESCUE_ROUNDS; r++) {
        s[0] = rescue_sbox(s[0]);
        s[1] = rescue_sbox(s[1]);
        drescue_mds_ark(mask, s[0], s[1], 2 * r, k, gbase, mds2);
        rescue_inv_sbox_lanes<2>(s);
        drescue_mds_ark(mask, s[0], s[1], 2 * r + 1, k, gbase, mds2);
    }
    lo_hi[0] = s[0];
    lo_hi[1] = s[1];
}
// hash_message (rescue.cuh) on six lanes; rx, px, py = the lane's coefficients (py: only lane 0's P.y[0] is used);
// msg/len are the group's message; the digest (4 elements) is returned on every lane
__device__ void dhash_message(unsigned mask, fp_t rx, fp_t px, fp_t py, const uint8_t* msg, uint64_t len, int k, int gbase,
                              const uint32_t* mds2, fp_t* d) {
    fp_t s[2];
    s[0] = rx;               // s[0..5] = R.x
    s[1] = k < 2 ? px : 0;   // s[6], s[7] = P.x[0..1]; capacity = 0
    drescue_permutation(mask, s, k, gbase, mds2);
    // s[0..3] += P.x[2..5], s[4] += P.y[0]
    fp_t t1 = dshfl(mask, px, gbase + (k + 2 < 6 ? k + 2 : 5)), t2 = dshfl(mask, py, gbase);
    s[0] = fp_add(s[0], k < 4 ? t1 : (k == 4 ? t2 : 0));
    int pos = 5;
    uint64_t nb = len / 7;
    int rem = (int)(len - 7 * nb);
    uint64_t total = nb + (rem ? 1 : 0);
    for (uint64_t cidx = 0; cidx < total; cidx++) {
        uint64_t chunk = cidx < nb ? load_le_bytes(msg + 7 * cidx, 7) : (load_le_bytes(msg + 7 * nb, rem) | (1ULL << (8 * rem)));
        fp_t v = (k == pos % 6) ? chunk : 0;
        if (pos >= 6) s[1] = fp_add(s[1], v);
        else s[0] = fp_add(s[0], v);
        if (++pos == 8) {
            drescue_permutation(mask, s, k, gbase, mds2);
            pos = 0;
        }
    }
    if (pos > 0) {  // a single '1' element of padding when the last block is partial
        fp_t v = (k == pos % 6) ? 1 : 0;
        if (pos >= 6) s[1] = fp_add(s[1], v);
        else s[0] = fp_add(s[0], v);
        drescue_permutation(mask, s, k, gbase, mds2);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) d[i] = dshfl(mask, s[0], gbase + i);
}
// challenge scalar (verify.cuh: challenge_scalar)
__device__ scalar dchallenge_scalar(unsigned mask, fp_t rx, fp_t px, fp_t py, const uint8_t* msg, uint64_t len, int k,
                                    int gbase, const uint32_t* mds2) {
    fp_t d[4];
    dhash_message(mask, rx, px, py, msg, len, k, gbase, mds2, d);
    return digest_to_scalar(d);
}

// verify_core_fast (affine.cuh) on six lanes.  px, py = the lane's coefficients of the public key.
__device__ int dverify_core(unsigned mask, fp_t px, fp_t py, const scalar& h, const scalar& e,
                            const uint64_t* __restrict__ gtab, dpt* R, int k, int gbase) {
    dpt Bq[8], Bh[8], D;
    int8_t hd[64];
    recode_signed_w4(h, hd);
    uint32_t q_seen = 0, h_seen = 0;
    bool exc = false;
#pragma unroll 1
    for (int b = 0; b < 8; b++) {
        Bq[b] = dpt{0, 0, 1};
        Bh[b] = Bq[b];
    }
    D = dpt{px, py, 1};
#pragma unroll 1
    for (int j = 0; j < SB_CHAIN_STEPS; j++) {
        if ((j & 3) == 0) SB_PHASE_SYNC();
        int dq = SB_QWNAF(j);
        if (dq != 0) {
            int idx = (dq < 0 ? -dq : dq) >> 1;
            if ((q_seen >> idx) & 1) {
                exc |= djf_add(mask, &Bq[idx], &D, dq < 0 ? JOP_SUB : JOP_ADD, k, gbase);
            } else {
                Bq[idx] = D;
                if (dq < 0) Bq[idx].Y = fp_neg(D.Y);
                q_seen |= 1u << idx;
            }
        }
        if ((j & 3) == 0) {
            int dh = hd[j >> 2];
            int mag = dh < 0 ? -dh : dh;
            int idx = mag ? mag - 1 : 0;
            exc |= djf_add(mask, &Bh[idx], &D, jf_add_mode(!((h_seen >> idx) & 1), mag == 0, dh < 0), k, gbase);
            if (mag) h_seen |= 1u << idx;
        }
        if (j < SB_CHAIN_STEPS - 1) exc |= djf_dbl(mask, &D, k, gbase);
    }
    dpt Rq = Bq[7], Oq = Bq[7], Rh = Bh[7], Oh = Bh[7];
    bool eRq = !((q_seen >> 7) & 1), eOq = eRq, eRh = !((h_seen >> 7) & 1), eOh = eRh;
    bool same_h = !eRh;
#pragma unroll 1
    for (int b = 6; b >= 0; b--) {
        SB_PHASE_SYNC();
        bool eb = !((q_seen >> b) & 1);
        exc |= djf_add(mask, &Rq, &Bq[b], jf_add_mode(eRq, eb, false), k, gbase);
        eRq = eRq && eb;
        if (b >= 1) {
            exc |= djf_add(mask, &Oq, &Rq, jf_add_mode(eOq, eRq, false), k, gbase);
            eOq = eOq && eRq;
        }
        eb = !((h_seen >> b) & 1);
        exc |= djf_add(mask, &Rh, &Bh[b], jf_add_mode(eRh, eb, false), k, gbase);
        if (!eb && !eRh) same_h = false;
        eRh = eRh && eb;
        if (same_h && !eOh) {  // group-uniform (h is per signature)
            exc |= djf_dbl(mask, &Oh, k, gbase);
            same_h = false;
        } else {
            exc |= djf_add(mask, &Oh, &Rh, jf_add_mode(eOh, eRh, false), k, gbase);
            same_h = eOh && !eRh;
        }
        eOh = eOh && eRh;
    }
    if (eOq || eRq) exc = true;
    else exc |= djf_dbl(mask, &Oq, k, gbase);
    // [q]P == O  <=>  2 O_1 == -R_0:  X_O w_R^2 == X_R w_O^2  and  Y_O w_R^3 == -Y_R w_O^3
    fp_t wos = fp_sqr_nc(Oq.w), wrs = fp_sqr_nc(Rq.w);
    bool x_eq = dall(mask, gbase, fp_mul(Oq.X, wrs) == fp_mul(Rq.X, wos));
    bool y_opp = dall(mask, gbase, fp_mul(Oq.Y, fp_mul_nc(wrs, Rq.w)) == fp_neg(fp_mul(Rq.Y, fp_mul_nc(wos, Oq.w))));
    bool torsion_free = x_eq && y_opp;
    if (x_eq && !torsion_free) exc = true;

    bool e_acc = eOh;
    *R = Oh;
    int carry = 0;
    dpt T;
    T.w = 1;
#pragma unroll 1
    for (int i = 0; i < GTAB_WINDOWS; i++) {
        if ((i & 3) == 0) SB_PHASE_SYNC();
        int raw = (int)sc_bits(e, GTAB_W * i, GTAB_W) + carry;
        bool neg = raw > (1 << (GTAB_W - 1));
        carry = neg ? 1 : 0;
        int dg = neg ? (1 << GTAB_W) - raw : raw;
        const uint64_t* ent = gtab + ((size_t)i * GTAB_ENTRIES + (dg ? dg : 1)) * GTAB_ENTRY_U64;
        T.X = ent[k];
        T.Y = ent[6 + k];
        exc |= djf_add(mask, R, &T, jf_add_mode(e_acc, dg == 0, neg), k, gbase);
        e_acc = e_acc && dg == 0;
    }
    if (e_acc) exc = true;
    if (exc) return FAST_EXCEPTIONAL;
    return torsion_free ? FAST_TORSION_FREE : FAST_NOT_TORSION_FREE;
}

}  // namespace sb
