// Registration of a FEW keys (schnorr_b200_keyset_create / _append / _replace): one thread block per key.
//
// k_keyset_register + k_tab_bases give each key one thread that walks two serial chains of ~250 Jacobian doublings
// (the exact subgroup check, then the window bases of the table): a call of a few keys is latency-bound on them.  Here
// the four warps of a block share the work of ONE key in the phases of k_verify_one (one.cuh):
//   A  warp 0: the doubling chain D_j = 2^j P on 24 lanes (jac_dbl_dist of batch.cuh), every D_j stored to shared
//      memory;   warp 1: the lists of chain steps of the eight buckets of the subgroup check (odd wNAF digits of q)
//   B  the eight bucket accumulations, two per warp (jac_add_dist_exact)
//   C  warp 0: aggregation of the buckets and the test [q]P == O -> the status byte;   warps 1-3: the window bases
//      2^(KT_W i) P = D_(KT_W i) to global memory, where the unchanged k_tab_fill builds the table from them.
// Additions are only re-associated with respect to torsion_check_and_mul and every exceptional operand falls back to
// the complete routines of curve.cuh, so the status and the group elements of the bases are those of
// k_keyset_register / k_tab_bases; the table entries are normalised to affine (tab_entry), so the table bytes are the
// same.  That holds for points off the curve too: the formulas never use the curve constant b.
// A separate copy of the phase code on purpose: sharing it with k_verify_one would change that tuned kernel.
#pragma once
#include "one.cuh"

namespace sb {

static_assert(KT_W * (KT_WINDOWS - 1) < SB_CHAIN_STEPS, "the window bases are steps of the doubling chain");
static_assert(CHEETAH_Q_WNAF5_LEN <= SB_CHAIN_STEPS, "the digits of q are steps of the doubling chain");

static constexpr int KREG_SLOTS = 8;  // buckets of the subgroup check: odd digits 2b + 1 of q, b < 8

struct keyreg_shared {
    fp_t cx[SB_CHAIN_STEPS][6], cy[SB_CHAIN_STEPS][6], cz[SB_CHAIN_STEPS][6];  // the chain D_j (Jacobian)
    fp_t bx[KREG_SLOTS][6], by[KREG_SLOTS][6], bz[KREG_SLOTS][6];             // bucket sums
    uint8_t lst[KREG_SLOTS][64];
    uint8_t neg[KREG_SLOTS][64];
    int cnt[KREG_SLOTS];
    int torsion_free;
};

// status[k] and skip[k] as k_keyset_register writes them, bases[k][i] = 2^(KT_W i) P_k as k_tab_bases writes them
// (for keys with skip[k] = 0).  One block of ONE_THREADS per key.
__global__ void __launch_bounds__(ONE_THREADS, 2) k_keyset_register_block(size_t n_keys, const uint64_t* __restrict__ pk12,
                                                                       const uint8_t* __restrict__ pk_inf,
                                                                       uint8_t* __restrict__ status, uint8_t* __restrict__ skip,
                                                                       jac_pt* __restrict__ bases) {
    __shared__ keyreg_shared S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool in24 = lane < 24;
    const int g = in24 ? lane / 6 : 0, k = lane % 6;
    const size_t key = blockIdx.x;
    if (key >= n_keys) return;
    const uint64_t* pk = pk12 + 12 * key;
    const bool inf = pk_inf[key] != 0;
    bool canonical = true;
#pragma unroll
    for (int c = 0; c < 12; c++) canonical &= pk[c] < FP_P;
    if (inf || !canonical) {  // block-uniform: keyset_key_status decides these without the chain
        if (tid == 0) {
            status[key] = inf ? KEY_OK : KEY_MALFORMED;
            skip[key] = 1;
        }
        return;
    }

    // ---- phase A: doubling chain | bucket lists ----------------------------------------------------------------
    if (warp == 0) {
        if (in24) {
            fp_t x = pk[k], y = pk[6 + k], z = k == 0 ? 1 : 0;
#pragma unroll 1
            for (int j = 0; j < SB_CHAIN_STEPS; j++) {
                if (g == 0) {
                    S.cx[j][k] = x;
                    S.cy[j][k] = y;
                    S.cz[j][k] = z;
                }
                if (j < SB_CHAIN_STEPS - 1) jac_dbl_dist(x, y, z, g, k);
            }
        }
    } else if (warp == 1 && lane < KREG_SLOTS) {
        const int slot = lane;
        int c = 0;
#pragma unroll 1
        for (int j = 0; j < CHEETAH_Q_WNAF5_LEN; j++) {
            int dq = SB_QWNAF(j);
            if (dq != 0 && ((dq < 0 ? -dq : dq) >> 1) == slot) {
                S.lst[slot][c] = (uint8_t)j;
                S.neg[slot][c] = dq < 0;
                c++;
            }
        }
        S.cnt[slot] = c;
    }
    __syncthreads();

    // ---- phase B: eight bucket accumulations, two per warp -------------------------------------------------------
    if (in24) {
#pragma unroll 1
        for (int q2 = 0; q2 < 2; q2++) {
            const int slot = warp * 2 + q2;
            const int cnt = S.cnt[slot];
            fp_t x = 1, y = 1, z = 0;  // identity (curve.cuh: jac_identity; only z matters)
#pragma unroll 1
            for (int t = 0; t < cnt; t++) {
                int j = S.lst[slot][t];
                fp_t x2 = S.cx[j][k], y2 = S.cy[j][k], z2 = S.cz[j][k];
                if (S.neg[slot][t]) y2 = fp_neg(y2);
                if (t == 0) {
                    x = x2;
                    y = y2;
                    z = z2;
                } else {
                    jac_add_dist_exact(x, y, z, x2, y2, z2, g, k);
                }
            }
            if (g == 0) {
                S.bx[slot][k] = x;
                S.by[slot][k] = y;
                S.bz[slot][k] = z;
            }
        }
    }
    __syncthreads();

    // ---- phase C: [q]P = 2 O_1 + R_0 (odd digits 2b + 1) | window bases ------------------------------------------
    if (warp == 0) {
        if (in24) {
            fp_t rx = S.bx[7][k], ry = S.by[7][k], rz = S.bz[7][k];
            fp_t ox = rx, oy = ry, oz = rz;
#pragma unroll 1
            for (int b = 6; b >= 0; b--) {
                jac_add_dist_exact(rx, ry, rz, S.bx[b][k], S.by[b][k], S.bz[b][k], g, k);
                if (b >= 1) jac_add_dist_exact(ox, oy, oz, rx, ry, rz, g, k);
            }
            jac_dbl_dist(ox, oy, oz, g, k);
            jac_add_dist_exact(ox, oy, oz, rx, ry, rz, g, k);
            bool ident = __ballot_sync(HORNER_MASK, oz == 0) == HORNER_MASK;
            if (lane == 0) S.torsion_free = ident;
        }
    } else {
        uint64_t* out = reinterpret_cast<uint64_t*>(bases + key * KT_WINDOWS);
#pragma unroll 1
        for (int t = tid - 32; t < KT_WINDOWS * 18; t += ONE_THREADS - 32) {
            const int i = t / 18, c = t % 18, j = KT_W * i;
            out[t] = c < 6 ? S.cx[j][c] : (c < 12 ? S.cy[j][c - 6] : S.cz[j][c - 12]);
        }
    }
    __syncthreads();
    if (tid == 0) {
        uint8_t st = S.torsion_free ? KEY_OK : KEY_NOT_TORSION_FREE;
        status[key] = st;
        skip[key] = st != KEY_OK;
    }
}

}  // namespace sb
