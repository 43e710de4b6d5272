// Rescue-Prime over Goldilocks, state 12 / rate 8 / capacity 4 -- the `hash::rescue_64_12_8::RescueHash`
// the reference calls at src/signature.rs:303-305 -- and the reference's own `hash_message`
// (src/signature.rs:274-306).  Instance parameters: include/cheetah_params.h (provenance in
// params/params.json; rounds/MDS/padding are "parity unpinned", see DESIGN.md).
//
// One message per thread; the 12-element state lives in registers; the circulant MDS row and the
// 168 round constants sit in __constant__ memory (uniform across the warp -> constant-cache
// broadcast, no shared-memory staging needed).
#pragma once
#include "../../include/cheetah_params.h"
#include "fp6.cuh"
#include "scalar.cuh"

namespace sb {

// circulant first row (RESCUE_MDS_ROW) and round constants (RESCUE_ARK) of cheetah_params.h
SB_CONSTANT uint32_t c_mds_row[12] = RESCUE_MDS_ROW_INIT;
// rescue_mds_ark below sums twelve (32-bit half) x (matrix entry) products in one 64-bit register without carries and
// indexes the first row cyclically: both properties are checked where the parameters are generated and again here
static_assert(RESCUE_MDS_IS_CIRCULANT == 1, "rescue_mds_ark needs a circulant MDS matrix");
static_assert(RESCUE_MDS_MAX_ENTRY < (1u << 28), "MDS entries too large for the carry-free accumulation of rescue_mds_ark");
#if defined(__CUDACC__)
__constant__ uint64_t c_ark[2 * RESCUE_ROUNDS * 12];  // filled from RESCUE_ARK at context creation
#define SB_ARK(i) c_ark[i]
#else
#define SB_ARK(i) RESCUE_ARK[i]
#endif

// x^7
// (result not canonical: the MDS layer that follows accepts any 64-bit representative)
SB_DEV fp_t rescue_sbox(fp_t x) {
    fp_t x2 = fp_sqr_nc(x);
    fp_t x3 = fp_mul_nc(x2, x);
    fp_t x4 = fp_sqr_nc(x2);
    return fp_mul_nc(x3, x4);
}

// y = M * s + k  with M circulant, entries < 2^28 (26 for the shipped parameters): the low and high 32-bit halves of the
// inputs are accumulated separately in 64-bit registers (12 * 2^28 * 2^32 < 2^64: no carries), one reduction per output.
SB_DEV void rescue_mds_ark(fp_t* s, int ark_row) {
    fp_t t[12];
#pragma unroll
    for (int i = 0; i < 12; i++) {
        uint64_t lo = 0, hi = 0;
#pragma unroll
        for (int j = 0; j < 12; j++) {
            uint32_t m = c_mds_row[(j - i + 12) % 12];
            lo += (uint64_t)(uint32_t)s[j] * m;
            hi += (s[j] >> 32) * m;
        }
        // value = lo + hi * 2^32 < 2^74
        uint64_t mid = (lo >> 32) + hi;  // weight 2^32, < 2^43
        fp_t r = fp_reduce96((uint32_t)lo, (uint32_t)mid, (uint32_t)(mid >> 32));
        t[i] = fp_add(r, SB_ARK(ark_row * 12 + i));
    }
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = t[i];
}

// x^(1/7) = x^0x92492491b6db6db7 = "100" x 10, "0", then "110" x 10 + "111" in binary:
// 63 squarings + 9 multiplications, evaluated on LANES independent elements at once (instruction-
// level parallelism) with rolled squaring loops (compact code: the whole round stays in the
// instruction cache).
template <int LANES>
SB_DEV void sqr_n_lanes(fp_t* v, int n) {
#pragma unroll 1
    for (int i = 0; i < n; i++) {
#pragma unroll
        for (int l = 0; l < LANES; l++) v[l] = fp_sqr_nc(v[l]);
    }
}
template <int LANES>
SB_DEV void rescue_inv_sbox_lanes(fp_t* x) {
    fp_t t1[LANES], t2[LANES], t3[LANES], t6[LANES], w[LANES];
#pragma unroll
    for (int l = 0; l < LANES; l++) {
        t1[l] = fp_sqr_nc(x[l]);   // 10b
        t2[l] = fp_sqr_nc(t1[l]);  // 100b
        w[l] = t2[l];
    }
    sqr_n_lanes<LANES>(w, 3);
#pragma unroll
    for (int l = 0; l < LANES; l++) t3[l] = w[l] = fp_mul_nc(w[l], t2[l]);  // 100100b
    sqr_n_lanes<LANES>(w, 6);
#pragma unroll
    for (int l = 0; l < LANES; l++) w[l] = fp_mul_nc(w[l], t3[l]);  // (100)x4
    fp_t t4[LANES];
#pragma unroll
    for (int l = 0; l < LANES; l++) t4[l] = w[l];
    sqr_n_lanes<LANES>(w, 12);
#pragma unroll
    for (int l = 0; l < LANES; l++) w[l] = fp_mul_nc(w[l], t4[l]);  // (100)x8
    sqr_n_lanes<LANES>(w, 6);
#pragma unroll
    for (int l = 0; l < LANES; l++) t6[l] = w[l] = fp_mul_nc(w[l], t3[l]);  // (100)x10
    sqr_n_lanes<LANES>(w, 31);
#pragma unroll
    for (int l = 0; l < LANES; l++) w[l] = fp_mul_nc(fp_sqr_nc(fp_mul_nc(w[l], t6[l])), t6[l]);  // t7^2 * t6
    sqr_n_lanes<LANES>(w, 2);
#pragma unroll
    for (int l = 0; l < LANES; l++) x[l] = fp_mul_nc(w[l], fp_mul_nc(fp_mul_nc(t1[l], t2[l]), x[l]));
}
SB_DEV fp_t rescue_inv_sbox(fp_t x) {
    rescue_inv_sbox_lanes<1>(&x);
    return fp_canon(x);
}

// Code-size discipline (ncu: the fully unrolled permutation was 4.9 k instructions and ran at a 76 % instruction-cache
// hit rate, "no instruction" being the top stall of k_hash and k_batch_prepare): ONE copy of the MDS layer, of the
// forward S-box group and of the inverse S-box group, driven by rolled loops over the two half-rounds and the two
// groups of six state elements.
// state elements per S-box group (independent chains interleaved for ILP; smaller = less code)
static constexpr int SBOX_LANES = 6;
// `sync`: block barrier per half-round.  Warps that run the permutation in step share instruction-cache lines (same
// effect as SB_PHASE_SYNC in the point loops); only legal when EVERY live thread of the block runs the same number of
// permutations -- the kernels vote on that (block_hash_vote, schnorr_b200.cu) and pass false otherwise; threads without work
// of their own hash along on a stand-in message so that the whole block reaches every barrier.
#if defined(__CUDA_ARCH__)
#define SB_HASH_SYNC(flag) do { if (flag) __syncthreads(); } while (0)
#else
#define SB_HASH_SYNC(flag) do { (void)(flag); } while (0)
#endif
SB_DEV_NOINLINE void rescue_permutation(fp_t* s, bool sync = false) {
#pragma unroll 1
    for (int hr = 0; hr < 2 * RESCUE_ROUNDS; hr++) {
        SB_HASH_SYNC(sync);
        if ((hr & 1) == 0) {
#pragma unroll 1
            for (int g = 0; g < 12; g += SBOX_LANES) {
#pragma unroll
                for (int i = 0; i < SBOX_LANES; i++) s[g + i] = rescue_sbox(s[g + i]);
            }
        } else {
            // inverse S-box: 6 independent chains at a time (ILP), one rolled copy of the code for both halves
#pragma unroll 1
            for (int g = 0; g < 12; g += SBOX_LANES) rescue_inv_sbox_lanes<SBOX_LANES>(s + g);
        }
        rescue_mds_ark(s, hr);
    }
}

// Streaming sponge = RescueHash::hash_field: additive absorption into state[0..8], permutation per
// full block, a single '1' element of padding only when the last block is partial, digest = state[0..4].
struct rescue_sponge {
    fp_t s[12];
    int i;
    bool sync;
};
SB_DEV void sponge_init(rescue_sponge& sp, bool sync = false) {
#pragma unroll
    for (int k = 0; k < 12; k++) sp.s[k] = 0;
    sp.i = 0;
    sp.sync = sync;
}
// number of permutations hash_message runs for a message of `len` bytes (13 fixed elements + ceil(len / 7), rate 8)
SB_DEV int hash_message_permutations(uint64_t len) { return (int)((13 + (len + 6) / 7 + 7) / 8); }
SB_DEV void sponge_absorb(rescue_sponge& sp, fp_t e) {
    // dynamic index into a register array would spill: select statically
#pragma unroll
    for (int k = 0; k < 8; k++)
        if (k == sp.i) sp.s[k] = fp_add(sp.s[k], e);
    if (++sp.i == 8) {
        rescue_permutation(sp.s, sp.sync);
        sp.i = 0;
    }
}
SB_DEV void sponge_finish(rescue_sponge& sp) {
    if (sp.i > 0) {
#pragma unroll
        for (int k = 0; k < 8; k++)
            if (k == sp.i) sp.s[k] = fp_add(sp.s[k], 1);
        rescue_permutation(sp.s, sp.sync);
    }
}

// load up to 7 message bytes as a little-endian integer
SB_DEV uint64_t load_le_bytes(const uint8_t* p, int n) {
    uint64_t v = 0;
    for (int k = 0; k < n; k++) v |= (uint64_t)p[k] << (8 * k);
    return v;
}

// hash_message (src/signature.rs:274-306): absorb R.x (6), P.x (6), P.y[0] (1), then the message in
// 7-byte little-endian chunks; a short tail chunk gets a 0x01 marker byte after its last byte.
// Returns the digest as 4 field elements (Digest::to_bytes = their little-endian bytes).
SB_DEV void hash_message(const fp6& rx, const fp6& px, fp_t py0, const uint8_t* msg, uint64_t len, fp_t* digest,
                         bool sync = false) {
    rescue_sponge sp;
    sponge_init(sp, sync);
    // first block is always full: 8 of the 13 fixed elements
    sp.s[0] = rx.c[0]; sp.s[1] = rx.c[1]; sp.s[2] = rx.c[2]; sp.s[3] = rx.c[3];
    sp.s[4] = rx.c[4]; sp.s[5] = rx.c[5]; sp.s[6] = px.c[0]; sp.s[7] = px.c[1];
    rescue_permutation(sp.s, sync);
    sp.s[0] = fp_add(sp.s[0], px.c[2]); sp.s[1] = fp_add(sp.s[1], px.c[3]);
    sp.s[2] = fp_add(sp.s[2], px.c[4]); sp.s[3] = fp_add(sp.s[3], px.c[5]);
    sp.s[4] = fp_add(sp.s[4], py0);
    sp.i = 5;
    uint64_t nb = len / 7;
    for (uint64_t c = 0; c < nb; c++) sponge_absorb(sp, load_le_bytes(msg + 7 * c, 7));
    int rem = (int)(len - 7 * nb);
    if (rem) sponge_absorb(sp, load_le_bytes(msg + 7 * nb, rem) | (1ULL << (8 * rem)));
    sponge_finish(sp);
#pragma unroll
    for (int k = 0; k < 4; k++) digest[k] = sp.s[k];
}

// digest (4 canonical field elements, little-endian) -> Scalar::from_bits_vartime = integer mod q
SB_DEV scalar digest_to_scalar(const fp_t* d) { return sc_from_u256(sc_from_u64x4(d[0], d[1], d[2], d[3])); }

}  // namespace sb
