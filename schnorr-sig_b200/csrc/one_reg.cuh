// Lowest-latency form of Signature::verify (src/signature.rs:181-205) against a REGISTERED key (keyset.cuh): one thread
// block per signature, for calls of a few signatures (schnorr_b200_set_one_threshold).
//
// Registration froze the key's doubling chain into its table ktab[key][window][|d|] = |d| 2^(KT_W window) P and its
// subgroup check into the status byte, so what is left of a verification is the challenge hash, 32 table terms for h*P
// and e*G.  k_verify_reg runs that on one thread per signature as a serial chain (hash + 52 table additions); here the
// four warps of a block share the work of ONE signature in three barrier-separated phases:
//   A  warp 0: the challenge hash on six lanes and the 32 signed KT_W-bit digits of h (the recoding of
//      jf_table_accumulate);   warp 1: e*G from the fixed-base table on six lanes (reg_one_e_stage, as in
//      k_verify_one)  -- side by side
//   B  the h*P tree: warp w loads the terms of windows 8w .. 8w+7 (entry |d| of the key's table, y negated for a
//      negative digit, the identity for d = 0) and adds them pairwise on 24 lanes (jac_add_dist_exact of batch.cuh);
//      then (0..7 + 8..15) and (16..23 + 24..31) on two warps, then their sum: 31 additions in 9 sequential rounds
//   C  warp 0: h*P + e*G, the x-only comparison against sig.x
// Latency = the hash + 10 sequential additions.  Every addition of the tree and the final one is exact (an identity
// operand or equal x takes the complete per-thread routine of curve.cuh), so the only items handed to k_verify are
// those k_verify_one hands back: the identity key, and a collision in the e*G stage (never for a reduced scalar).
// Additions are only re-associated with respect to verify_points: same group elements, same verdicts.
#pragma once
#include "one.cuh"
#include "keyset.cuh"

namespace sb {

static_assert(KT_WINDOWS == 32, "the h*P tree gives eight windows to each of the four warps of a block");
static constexpr int REG_ONE_WARP_WINDOWS = KT_WINDOWS / (ONE_THREADS / 32);

struct reg_one_shared {
    fp_t px[KT_WINDOWS][6], py[KT_WINDOWS][6], pz[KT_WINDOWS][6];  // window terms of h*P, then the partial sums of the tree
    fp_t ex[6], ey[6], ew;                                         // e*G as (X, Y, w): a Jacobian point with Z = w
    uint32_t mds2[24];
    int16_t hd[KT_WINDOWS];                                        // signed digits of h, -2^(KT_W-1) < d <= 2^(KT_W-1)
    int e_empty;                                                   // reg_one_e_stage: 0, 1 (e = 0) or 2 (collision)
};

// h = sum_i d_i 2^(KT_W i): the signed recoding of jf_table_accumulate, carry into the next window included
__device__ __forceinline__ void recode_signed_kt(const scalar& h, int16_t* d) {
    int carry = 0;
#pragma unroll 1
    for (int i = 0; i < KT_WINDOWS; i++) {
        int raw = (int)sc_bits(h, KT_W * i, KT_W) + carry;
        bool neg = raw > (1 << (KT_W - 1));
        carry = neg ? 1 : 0;
        d[i] = (int16_t)(neg ? raw - (1 << KT_W) : raw);
    }
}

// e*G into S on lanes k = 0..5 of one warp (phase A): k_verify_one's e*G stage, the same (X, Y, w) additions on six
// lanes, so that a collision (never for a reduced scalar) is handed back as k_verify_one hands it back.  A copy on
// purpose: factoring the loop out of k_verify_one changed that kernel's SASS (its stack frame).
__device__ __forceinline__ void reg_one_e_stage(reg_one_shared& S, const scalar& e, const uint64_t* __restrict__ gtab, int k) {
    dpt R{0, 0, 1}, T;
    T.w = 1;
    bool e_acc = true, exc = false;
    int carry = 0;
#pragma unroll 1
    for (int w = 0; w < GTAB_WINDOWS; w++) {
        int raw = (int)sc_bits(e, GTAB_W * w, GTAB_W) + carry;
        bool neg = raw > (1 << (GTAB_W - 1));
        carry = neg ? 1 : 0;
        int dg = neg ? (1 << GTAB_W) - raw : raw;
        const uint64_t* ent = gtab + ((size_t)w * GTAB_ENTRIES + (dg ? dg : 1)) * GTAB_ENTRY_U64;
        T.X = ent[k];
        T.Y = ent[6 + k];
        exc |= djf_add(0x3fu, &R, &T, jf_add_mode(e_acc, dg == 0, neg), k, 0);
        e_acc = e_acc && dg == 0;
    }
    S.ex[k] = R.X;
    S.ey[k] = R.Y;
    if (k == 0) {
        S.ew = R.w;
        S.e_empty = exc ? 2 : (e_acc ? 1 : 0);   // 1: e = 0 (R is not a point), 2: the table points collided
    }
}

// Phases B and C on the digits S.hd and e*G in S: every thread of the block calls this after the barrier that ends
// phase A.  On return the lanes k of warp 0 (all four groups) hold coefficient k of h*P + e*G in (x, y, z), Jacobian.
__device__ __forceinline__ void reg_one_point_stage(reg_one_shared& S, const uint64_t* __restrict__ ktab_key, fp_t& x,
                                                    fp_t& y, fp_t& z) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool in24 = lane < 24;
    const int g = in24 ? lane / 6 : 0, k = lane % 6;
    const int first = REG_ONE_WARP_WINDOWS * warp;
    // the warp's terms, loaded side by side: entry |d| (entry 1 for d = 0, a point whose z = 0 makes it the identity)
#pragma unroll 1
    for (int t = lane; t < REG_ONE_WARP_WINDOWS * 12; t += 32) {
        const int j = first + t / 12, c = t % 12, d = S.hd[j], m = d < 0 ? -d : d;
        fp_t v = ktab_key[((size_t)j * KT_ENTRIES + (m ? m : 1)) * 12 + c];
        if (c < 6) S.px[j][c] = v;
        else S.py[j][c - 6] = d < 0 ? fp_neg(v) : v;
    }
#pragma unroll 1
    for (int t = lane; t < REG_ONE_WARP_WINDOWS * 6; t += 32) {
        const int j = first + t / 6, c = t % 6;
        S.pz[j][c] = (c == 0 && S.hd[j] != 0) ? 1 : 0;
    }
    __syncwarp();
    // the tree: at stride s, sum j += sum j + s for j = 0 mod 2s, each warp over the windows it owns at that level
#pragma unroll 1
    for (int s = 1; s < KT_WINDOWS; s <<= 1) {
        const int span = s < REG_ONE_WARP_WINDOWS ? REG_ONE_WARP_WINDOWS : 2 * s;
        if (in24 && (warp + 1) * span <= KT_WINDOWS) {
#pragma unroll 1
            for (int j = warp * span; j < (warp + 1) * span; j += 2 * s) {
                x = S.px[j][k];
                y = S.py[j][k];
                z = S.pz[j][k];
                jac_add_dist_exact(x, y, z, S.px[j + s][k], S.py[j + s][k], S.pz[j + s][k], g, k);
                if (g == 0) {
                    S.px[j][k] = x;
                    S.py[j][k] = y;
                    S.pz[j][k] = z;
                }
                __syncwarp(HORNER_MASK);
            }
        }
        __syncthreads();
    }
    if (warp == 0 && in24) {
        fp_t ez = (S.e_empty == 0 && k == 0) ? S.ew : 0;
        x = S.px[0][k];
        y = S.py[0][k];
        z = S.pz[0][k];
        jac_add_dist_exact(x, y, z, S.ex[k], S.ey[k], ez, g, k);
    }
}

// MINB = resident blocks per SM the register allocation must allow, as in k_verify_one.  Only 2 is launched (246
// registers, no spills): at 3 or 4 per SM (168 / 128 registers) the kernel body spills (44 / 64 bytes per thread), so
// calls above 2 x SMs signatures run in a second wave instead.  LOOKUP: the items of a keyed call (k_keyed_split_lookup),
// where key_idx[i] == KEYSET_MISS marks a record whose key is not in the set: it is handed to k_verify, which reads the
// key decompressed into the planes.
// Verdicts with the precedence of reg_verdict (keyset.cuh): malformed record, identity key (handed back), key of status
// KEY_NOT_TORSION_FREE, non-canonical sig.x, then the comparison -- the first four without any point arithmetic.
template <int MINB, bool LOOKUP>
__global__ void __launch_bounds__(ONE_THREADS, MINB) k_verify_reg_one(soa_batch in, const uint32_t* __restrict__ key_idx,
                                                                  const uint8_t* __restrict__ key_status,
                                                                  const uint64_t* __restrict__ ktab,
                                                                  const uint8_t* __restrict__ msgs,
                                                                  const uint64_t* __restrict__ msg_off,
                                                                  const uint64_t* __restrict__ gtab,
                                                                  uint8_t* __restrict__ verdicts,
                                                                  uint32_t* __restrict__ work_list,
                                                                  uint32_t* __restrict__ work_count) {
    __shared__ reg_one_shared S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, k = lane % 6;
    const size_t i = blockIdx.x, n = in.n;
    const uint8_t fl = in.flags[i];          // block-uniform from here on
    uint32_t key = 0;
    uint8_t v = 0;
    bool decided = true;
    if (fl & FL_MALFORMED) v = VERDICT_MALFORMED;
    else if (fl & FL_PK_INF) v = VERDICT_NEEDS_EXACT;   // the identity key is the exact kernel's business
    else if (LOOKUP && (key = key_idx[i]) == KEYSET_MISS) v = VERDICT_NEEDS_EXACT;
    else {
        // a record that is not malformed has an index inside the set (k_keyset_gather)
        key = key_idx[i];
        if (key_status[key] == KEY_NOT_TORSION_FREE) v = VERDICT_INVALID_PUBLIC_KEY;
        else if (fl & FL_X_BAD) v = VERDICT_MALFORMED;
        else decided = false;
    }
    if (decided) {
        if (tid == 0) {
            verdicts[i] = v;
            if (v == VERDICT_NEEDS_EXACT) work_list[atomicAdd(work_count, 1u)] = (uint32_t)i;
        }
        return;
    }
    if (tid < 24) S.mds2[tid] = c_mds_row[tid % 12];
    __syncthreads();
    const uint64_t* pl = reinterpret_cast<const uint64_t*>(in.planes);
    fp_t sx = pl[((size_t)(0 + (k >> 1)) * n + i) * 2 + (k & 1)];

    // ---- phase A: challenge | e*G -------------------------------------------------------------------------------
    if (warp == 0) {
        if (lane < 6) {
            fp_t px = pl[((size_t)(5 + (k >> 1)) * n + i) * 2 + (k & 1)];
            fp_t py = pl[((size_t)(8 + (k >> 1)) * n + i) * 2 + (k & 1)];
            uint64_t off = msg_off[i];
            scalar h = dchallenge_scalar(0x3fu, sx, px, py, msgs + off, msg_off[i + 1] - off, k, 0, S.mds2);
            if (k == 0) recode_signed_kt(h, S.hd);
        }
    } else if (warp == 1) {
        if (lane < 6) reg_one_e_stage(S, load_scalar_planes(in.planes, 3, n, i), gtab, k);
    }
    __syncthreads();

    // ---- phases B and C: the h*P tree, + e*G, x-only comparison ---------------------------------------------------
    fp_t x, y, z;
    reg_one_point_stage(S, ktab + (size_t)key * KT_KEY_U64, x, y, z);
    if (warp == 0 && lane < 24) {
        // x-only comparison (src/signature.rs:200) as jac_x_equals, on the 24 lanes: X == sig.x Z^2, the identity reading
        // as x = 0 (every value here is canonical)
        const int gbase = 6 * (lane / 6);
        const bool r_inf = __ballot_sync(HORNER_MASK, z == 0) == HORNER_MASK;
        fp_t rhs = dfp6_mul(HORNER_MASK, sx, dfp6_mul(HORNER_MASK, z, z, k, gbase), k, gbase);
        v = __ballot_sync(HORNER_MASK, r_inf ? sx == 0 : x == rhs) == HORNER_MASK ? VERDICT_OK : VERDICT_INVALID_SIGNATURE;
        if (S.e_empty == 2) v = VERDICT_NEEDS_EXACT;
        if (lane == 0) {
            verdicts[i] = v;
            if (v == VERDICT_NEEDS_EXACT) work_list[atomicAdd(work_count, 1u)] = (uint32_t)i;
        }
    }
}

}  // namespace sb
