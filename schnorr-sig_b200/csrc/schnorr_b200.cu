// schnorr_b200 -- kernels, host orchestration and the C ABI (include/schnorr_b200.h).
//
// Kernel inventory (SURVEY.md §2, "kernels the new build must create"):
//   k_ingest          AoS wire records -> SoA limb planes (coalesced 128-bit stores), input checks
//   k_hash            K1  hash_message per thread
//   k_verify          K2  Signature::verify per thread (challenge hash + subgroup check + h*P + e*G)
//   k_keygen / k_sign K5  fixed-base multiplication; device signer for synthetic inputs
//   k_tab_*               signed-window tables of affine multiples: the fixed-base table of G at context creation,
//                         the per-key tables of registered key sets
//   k_keyset_register     registration of a key set (status + subgroup check per key)
//   k_keyset_register_block  the same for a few keys, one thread block per key, with the table's window bases
//   k_keyset_scatter      replaced slots of a key set: records, status and tables from a compact registration
//   k_keyset_gather       key records of the items of a registered call (ahead of k_ingest)
//   k_verify_reg          Signature::verify against registered keys (table additions, no doubling chain)
//   k_keyset_encode       the lookup table of a key set's compressed encodings (sorted on the host)
//   k_keyset_lookup       compressed keys -> indices into a registered key set (binary search)
//   k_keyed_split_lookup  KeyedSignature records against a registered key set: registered record on a hit, decompressed
//                         key on a miss, ahead of k_ingest
//   k_keyed_bad_records   batches over KeyedSignature records: an undecodable key -> the record of an index outside a set
//   k_imad_peak       K6  integer-multiply roofline calibration
//   batch kernels     K3/K4  in batch.cuh (Pippenger MSM)
// No CPU fallback exists: every entry point needs a live CUDA context.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/cheetah_params.h"
#include "../../include/schnorr_b200.h"
#include "verify.cuh"
#include "keyset.cuh"
#include "dist.cuh"
#include "debug_ops.cuh"
#include "derive.cuh"

using namespace sb;

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
static constexpr size_t GTAB_U64 = (size_t)GTAB_WINDOWS * GTAB_ENTRIES * 12;
// Batches against a registered key set sum the key side per key (one table product per key instead of one MSM point
// per signature) when they hold at least this many signatures per key of the set; others run the per-signature
// pipeline on the gathered key records (schnorr_b200_set_registered_batch_threshold).  Measured on a B200 (1000 W,
// 1965 MHz; profiles/r4_registered_batch.md), summed per key against per signature: 64 per key wins at every size
// (2^12 / 64 keys 0.89 against 0.91 ms, 2^16 / 1024 keys 2.31 against 2.51 ms, 2^20 / 16 384 keys 20.9 against
// 23.0 ms), 16 per key loses (2^10 / 64 keys 0.82 against 0.80 ms), 4 per key loses (2^16 / 16 384 keys 2.83
// against 2.51 ms): the key terms of a warp per key cost more than the MSM points they remove.
static constexpr size_t REG_BATCH_MIN_PER_KEY = 64;
// Registrations (keyset_create / _append / _replace) of at most this many keys run one thread block per key
// (k_keyset_register_block), larger ones one thread per key (k_keyset_register, k_tab_bases); the tables are then built
// by k_tab_fill either way (schnorr_b200_set_keyset_block_threshold).  Measured on a B200 (1000 W, 1965 MHz;
// profiles/r6_keyset_update.md), warm replace calls, block against thread kernels: 1 key 0.64 / 3.46 ms, 64 keys
// 1.67 / 4.53 ms, 512 keys 10.3 / 12.8 ms, 4096 keys 81.5 / 79.5 ms (sets of 64 to 16 384 keys).
static constexpr size_t KEYSET_BLOCK_MAX = 512;

// N, O: batches against registered key sets (gathered key records; key-side accumulators and terms), which run
// batch_partial_impl (A-G, I-L) on inputs staged in H or M
enum scratch_slot { SL_A = 0, SL_B, SL_C, SL_D, SL_E, SL_F, SL_G, SL_H, SL_I, SL_J, SL_K, SL_L, SL_M, SL_N, SL_O, SL_COUNT };

struct schnorr_b200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    uint64_t* gtab = nullptr;
    void* scratch[SL_COUNT] = {};
    size_t scratch_cap[SL_COUNT] = {};
    uint64_t launches = 0;
    int sm_count = 148;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // bracket the dominant kernel of the last call
    size_t verify_wave = 148 * 256;                 // signatures resident at once in k_verify (filled at creation)
    cudaStream_t copy_stream = nullptr;             // host->device staging of the pipelined host entry points
    cudaStream_t aux_stream = nullptr;              // second compute stream: consecutive pipeline chunks alternate between
    cudaEvent_t ev_aux = nullptr;                   // the two, so a chunk's blocks fill the SMs the previous chunk drains
    bool exact_only = false;                        // schnorr_b200_set_exact_only: skip the fast path (A/B measurements, tests)
    int msm_c_override = 0;                         // schnorr_b200_set_msm_geometry (tests): forced window width / segment length
    uint32_t msm_t_override = 0;
    int last_msm_c = 0, last_msm_K = 0;             // Pippenger geometry of the last batch call (schnorr_b200_last_batch_plan)
    uint32_t last_msm_T = 0;
    uint64_t last_batch_points = 0;                 // MSM points of the last batch call (schnorr_b200_last_batch_points)
    size_t reg_batch_min_per_key = REG_BATCH_MIN_PER_KEY;
    size_t keyset_block_max = KEYSET_BLOCK_MAX;     // registrations of up to this many keys: k_keyset_register_block
    size_t dist_max = 10240;                        // calls up to this many signatures use the six-lanes-per-signature kernel
    size_t one_max = 512;                           // ... and up to this many the block-per-signature kernel (one.cuh)
    size_t batch_dist_max = (size_t)1 << 18;        // batches up to this size hash their challenges on six lanes per signature
    size_t batch_small_max = 256;                   // batches up to this size run one thread block per signature (k_batch_small)
    int exact_counters_used = 0;                    // work-list counters written by the last verify call
    static constexpr int MAX_CHUNKS = 16;
    cudaEvent_t ev_chunk[MAX_CHUNKS] = {};
    std::string err;
    // multi-device context (schnorr_b200_create_multi): one single-device context per listed device; empty otherwise
    std::vector<schnorr_b200_ctx*> shards;
};

#define CUDA_TRY(ctx, expr)                                                                      \
    do {                                                                                         \
        cudaError_t e_ = (expr);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e_);                     \
            return SCHNORR_B200_ECUDA;                                                           \
        }                                                                                        \
    } while (0)

static int ensure_scratch(schnorr_b200_ctx* ctx, int slot, size_t bytes, void** out) {
    if (bytes == 0) bytes = 16;
    if (ctx->scratch_cap[slot] < bytes) {
        if (ctx->scratch[slot]) {
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            CUDA_TRY(ctx, cudaFree(ctx->scratch[slot]));
            ctx->scratch[slot] = nullptr;
            ctx->scratch_cap[slot] = 0;
        }
        size_t cap = bytes + bytes / 8;
        CUDA_TRY(ctx, cudaMalloc(&ctx->scratch[slot], cap));
        ctx->scratch_cap[slot] = cap;
    }
    *out = ctx->scratch[slot];
    return 0;
}

// ------------------------------------------------------------------------------------------------
// SoA device layout: plane-major ulonglong2, plane p of an Fp6 holds coefficients (2p, 2p+1).
//   sx[3][n] sig.x   se[2][n] sig.e   px[3][n] py[3][n] public key   fl[n] flags
// A warp reads 32 x 16 B = 512 contiguous bytes per plane.
// ------------------------------------------------------------------------------------------------
static constexpr uint8_t FL_PK_INF = 1;     // public key is the identity
static constexpr uint8_t FL_X_BAD = 2;      // sig.x has a non-canonical limb
static constexpr uint8_t FL_MALFORMED = 4;  // e >= q or non-canonical public-key limb
static constexpr int SOA_PLANES = 11;

struct soa_batch {
    ulonglong2* planes;  // [11][n]: 0-2 sx, 3-4 se, 5-7 px, 8-10 py
    uint8_t* flags;      // [n]
    uint8_t* sig_flag;   // [n] byte 48 of the compressed point (used by batch verification only)
    size_t n;
};

// The planes are read exactly once per launch: streaming loads (evict-first) keep them from displacing the thread-local
// bucket lines that the L2 is really caching in these kernels.
__device__ __forceinline__ ulonglong2 load_plane(const ulonglong2* p) {
    return __ldcs(p);
}
__device__ __forceinline__ fp6 load_fp6_planes(const ulonglong2* planes, int first_plane, size_t n, size_t i) {
    ulonglong2 a = load_plane(&planes[(size_t)(first_plane + 0) * n + i]);
    ulonglong2 b = load_plane(&planes[(size_t)(first_plane + 1) * n + i]);
    ulonglong2 c = load_plane(&planes[(size_t)(first_plane + 2) * n + i]);
    return fp6{{a.x, a.y, b.x, b.y, c.x, c.y}};
}
__device__ __forceinline__ scalar load_scalar_planes(const ulonglong2* planes, int first_plane, size_t n, size_t i) {
    ulonglong2 a = load_plane(&planes[(size_t)(first_plane + 0) * n + i]);
    ulonglong2 b = load_plane(&planes[(size_t)(first_plane + 1) * n + i]);
    return sc_from_u64x4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ uint64_t load_u64_le(const uint8_t* p) {
    uint64_t v = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) v |= (uint64_t)p[k] << (8 * k);
    return v;
}

// Block-wide agreement on the challenge hash.  The permutation takes a block barrier per half-round when every hashing
// thread of the block runs the same number of Rescue permutations (rescue.cuh: the warps then share instruction-cache
// lines), and barriers need EVERY thread of the block: threads without work of their own (past the end of the batch,
// malformed items, identity keys) therefore hash along on the message of the block's first hashing thread and drop the
// result.  Must be called by all threads of the block.
//   np         this thread's permutation count, -1 if it has nothing to hash
//   off / len  in: this thread's message; out: the message to hash (its own, or the first hasher's)
//   returns    sync  = all hashing threads agree on the count (take the barriers)
//              any   = at least one thread of the block hashes
struct hash_vote {
    bool sync, any;
};
__device__ __forceinline__ hash_vote block_hash_vote(int np, uint64_t& off, uint64_t& len) {
    __shared__ int s_np_min, s_np_max, s_first;
    __shared__ uint64_t s_off, s_len;
    if (threadIdx.x == 0) {
        s_np_min = 1 << 30;
        s_np_max = -1;
        s_first = 1 << 30;
    }
    __syncthreads();
    if (np >= 0) {
        atomicMin(&s_np_min, np);
        atomicMax(&s_np_max, np);
        atomicMin(&s_first, (int)threadIdx.x);
    }
    __syncthreads();
    if ((int)threadIdx.x == s_first) {
        s_off = off;
        s_len = len;
    }
    __syncthreads();
    hash_vote v;
    v.any = s_np_max >= 0;
    v.sync = v.any && s_np_min >= s_np_max;
    if (np < 0 && v.any) {
        off = s_off;
        len = s_len;
    }
    return v;
}

// AoS -> SoA.  The 81-byte signature records of a block are staged through shared memory with
// coalesced 16-byte loads; public keys (96 B, 8-byte aligned) are read directly.
static constexpr int INGEST_THREADS = 128;
__global__ void __launch_bounds__(INGEST_THREADS) k_ingest(size_t n, const uint8_t* __restrict__ sigs81,
                                                           const uint8_t* __restrict__ pk96,
                                                           const uint8_t* __restrict__ pk_inf, soa_batch out) {
    __shared__ __align__(16) uint8_t s_sig[INGEST_THREADS * 81];
    size_t base = (size_t)blockIdx.x * INGEST_THREADS;
    size_t cnt = n - base < (size_t)INGEST_THREADS ? n - base : (size_t)INGEST_THREADS;
    size_t bytes = cnt * 81;
    const uint8_t* src = sigs81 + base * 81;
    if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        size_t nv = bytes / 16;
        for (size_t k = threadIdx.x; k < nv; k += INGEST_THREADS)
            reinterpret_cast<uint4*>(s_sig)[k] = reinterpret_cast<const uint4*>(src)[k];
        for (size_t k = nv * 16 + threadIdx.x; k < bytes; k += INGEST_THREADS) s_sig[k] = src[k];
    } else {
        for (size_t k = threadIdx.x; k < bytes; k += INGEST_THREADS) s_sig[k] = src[k];
    }
    __syncthreads();
    size_t i = base + threadIdx.x;
    if (i >= n) return;
    const uint8_t* rec = s_sig + threadIdx.x * 81;
    uint64_t x[6], e[4];
#pragma unroll
    for (int k = 0; k < 6; k++) x[k] = load_u64_le(rec + 8 * k);
#pragma unroll
    for (int k = 0; k < 4; k++) e[k] = load_u64_le(rec + 49 + 8 * k);
    const uint64_t* pk = reinterpret_cast<const uint64_t*>(pk96 + i * 96);
    uint64_t p[12];
#pragma unroll
    for (int k = 0; k < 12; k++) p[k] = pk[k];
    uint8_t fl = 0;
    bool inf = pk_inf != nullptr && pk_inf[i] != 0;
    if (inf) fl |= FL_PK_INF;
    bool x_ok = true, pk_ok = true;
#pragma unroll
    for (int k = 0; k < 6; k++) x_ok &= x[k] < FP_P;
#pragma unroll
    for (int k = 0; k < 12; k++) pk_ok &= p[k] < FP_P;
    if (!x_ok) fl |= FL_X_BAD;
    if ((!pk_ok && !inf) || sc_geq_q(sc_from_u64x4(e[0], e[1], e[2], e[3]))) fl |= FL_MALFORMED;
    size_t N = out.n;
    ulonglong2* pl = out.planes;
    pl[0 * N + i] = make_ulonglong2(x[0], x[1]);
    pl[1 * N + i] = make_ulonglong2(x[2], x[3]);
    pl[2 * N + i] = make_ulonglong2(x[4], x[5]);
    pl[3 * N + i] = make_ulonglong2(e[0], e[1]);
    pl[4 * N + i] = make_ulonglong2(e[2], e[3]);
#pragma unroll
    for (int k = 0; k < 6; k++) pl[(size_t)(5 + k) * N + i] = make_ulonglong2(p[2 * k], p[2 * k + 1]);
    out.flags[i] = fl;
    out.sig_flag[i] = rec[48];
}

// ------------------------------------------------------------------------------------------------
// K2: Signature::verify, one signature per thread
// ------------------------------------------------------------------------------------------------
#ifndef VERIFY_THREADS_N
#define VERIFY_THREADS_N 128
#endif
static constexpr int VERIFY_THREADS = VERIFY_THREADS_N;
#ifndef VERIFY_MIN_BLOCKS
#define VERIFY_MIN_BLOCKS 2
#endif
__global__ void __launch_bounds__(VERIFY_THREADS, VERIFY_MIN_BLOCKS) k_verify(soa_batch in, const uint8_t* __restrict__ msgs,
                                                           const uint64_t* __restrict__ msg_off,
                                                           const uint64_t* __restrict__ gtab,
                                                           uint8_t* __restrict__ verdicts,
                                                           const uint32_t* __restrict__ work_list,
                                                           const uint32_t* __restrict__ work_count) {
    // running point D_j of each thread: shared memory, padded to 152 B per thread (2-way bank conflicts at most)
    struct d_slot {
        jac_pt p;
        uint64_t pad;
    };
    __shared__ d_slot s_d[VERIFY_THREADS];
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (work_list) {  // exact pass over the items the fast path handed back
        if (i >= *work_count) return;
        i = work_list[i];
    }
    if (i >= in.n) return;
    uint8_t fl = in.flags[i];
    if (fl & FL_MALFORMED) {
        verdicts[i] = VERDICT_MALFORMED;
        return;
    }
    fp6 sx = load_fp6_planes(in.planes, 0, in.n, i);
    scalar e = load_scalar_planes(in.planes, 3, in.n, i);
    fp6 px = load_fp6_planes(in.planes, 5, in.n, i);
    fp6 py = load_fp6_planes(in.planes, 8, in.n, i);
    bool pk_inf = fl & FL_PK_INF;
    bool x_ok = !(fl & FL_X_BAD);
    uint64_t off = msg_off[i];
    scalar h = sc_zero();
    if (x_ok) h = challenge_scalar(sx, px, py, pk_inf, msgs + off, msg_off[i + 1] - off);
    verdicts[i] = verify_points(sx, x_ok, e, px, py, pk_inf, h, gtab, &s_d[threadIdx.x].p);
}

// K2 fast path: the same verdicts through point arithmetic in (X, Y, w) coordinates, w in Fp (affine.cuh).
// Items that meet an exceptional case of the chord-and-tangent formulas (identity / small-order keys, colliding
// partial sums: ~0.1 % of honest inputs) are appended to `work_list` and finished by k_verify.
#ifndef VERIFY_FAST_MIN_BLOCKS
#define VERIFY_FAST_MIN_BLOCKS 2
#endif
static constexpr size_t VERIFY_FAST_SMEM = (size_t)(1 + FAST_BH_SHARED) * VERIFY_THREADS * sizeof(jf_pt);  // 106 496 B: two blocks per SM
__global__ void __launch_bounds__(VERIFY_THREADS, VERIFY_FAST_MIN_BLOCKS) k_verify_fast(soa_batch in, const uint8_t* __restrict__ msgs,
                                                           const uint64_t* __restrict__ msg_off,
                                                           const uint64_t* __restrict__ gtab,
                                                           uint8_t* __restrict__ verdicts,
                                                           uint32_t* __restrict__ work_list,
                                                           uint32_t* __restrict__ work_count) {
    // dynamic shared memory (VERIFY_FAST_SMEM bytes): the running point D_j of every thread, then FAST_BH_SHARED
    // challenge buckets per thread, bucket-major.  A slot is 104 bytes: 64-bit accesses of a half-warp fall into sixteen
    // distinct even banks whatever bucket each thread addresses.
    extern __shared__ __align__(16) unsigned char s_fast[];
    jf_pt* s_d = reinterpret_cast<jf_pt*>(s_fast);
    jf_pt* s_bh = s_d + VERIFY_THREADS;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool live = i < in.n;
    uint8_t fl = live ? in.flags[i] : FL_MALFORMED;
    // `work`: this thread has a verification of its own.  Every other thread of the block (past the end of the batch,
    // malformed record, identity key) runs the SAME instruction stream on stand-in inputs -- the generator as the key,
    // zero scalars, the first hashing thread's message -- so that all 128 threads reach every barrier of the hash and of
    // the point loops; its result is dropped.
    bool work = live && !(fl & (FL_MALFORMED | FL_PK_INF));
    uint64_t off = work ? msg_off[i] : 0, len = work ? msg_off[i + 1] - off : 0;
    hash_vote hv = block_hash_vote(work ? hash_message_permutations(len) : -1, off, len);
    fp6 sx = fp6_zero(), px, py;
    scalar e = sc_zero();
    if (work) {
        sx = load_fp6_planes(in.planes, 0, in.n, i);
        e = load_scalar_planes(in.planes, 3, in.n, i);
        px = load_fp6_planes(in.planes, 5, in.n, i);
        py = load_fp6_planes(in.planes, 8, in.n, i);
    } else {  // 1 * G, the first entry of the fixed-base table
        const uint64_t* g = gtab + (size_t)1 * GTAB_ENTRY_U64;
#pragma unroll
        for (int k = 0; k < 6; k++) {
            px.c[k] = g[k];
            py.c[k] = g[6 + k];
        }
    }
    bool x_ok = !(fl & FL_X_BAD);
    scalar h = sc_zero();
    if (hv.any) {  // block-uniform.  An item with a malformed x hashes too (result unused)
        h = challenge_scalar(sx, px, py, false, msgs + off, len, hv.sync);
        if (!x_ok || !work) h = sc_zero();
    }
    uint8_t v = verify_points_fast(sx, x_ok, e, px, py, false, h, gtab, s_d + threadIdx.x, s_bh + threadIdx.x, VERIFY_THREADS);
    if (!live) return;
    if (fl & FL_MALFORMED) v = VERDICT_MALFORMED;
    else if (fl & FL_PK_INF) v = VERDICT_NEEDS_EXACT;   // the identity key is the exact kernel's business
    verdicts[i] = v;
    if (v == VERDICT_NEEDS_EXACT) work_list[atomicAdd(work_count, 1u)] = (uint32_t)i;
}

// K2 for small calls: one signature per group of six lanes (dist.cuh), five signatures per warp.  Same verdicts and
// the same hand-back list as k_verify_fast.
static constexpr int DIST_THREADS = 128;
static constexpr int DIST_SIGS_PER_BLOCK = (DIST_THREADS / 32) * 5;
__global__ void __launch_bounds__(DIST_THREADS) k_verify_dist(soa_batch in, const uint8_t* __restrict__ msgs,
                                                              const uint64_t* __restrict__ msg_off,
                                                              const uint64_t* __restrict__ gtab,
                                                              uint8_t* __restrict__ verdicts,
                                                              uint32_t* __restrict__ work_list,
                                                              uint32_t* __restrict__ work_count) {
    __shared__ uint32_t s_mds2[24];  // the circulant MDS row twice: M[i][j] = s_mds2[j - i + 12]
    if (threadIdx.x < 24) s_mds2[threadIdx.x] = c_mds_row[threadIdx.x % 12];
    __syncthreads();
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int g = lane / 6, k = lane % 6;
    if (g >= 5) return;  // lanes 30, 31 idle
    size_t i = ((size_t)blockIdx.x * (DIST_THREADS / 32) + warp) * 5 + g;
    if (i >= in.n) return;
    int gbase = 6 * g;
    unsigned mask = 0x3fu << gbase;
    uint8_t fl = in.flags[i];
    if (fl & FL_MALFORMED) {
        if (k == 0) verdicts[i] = VERDICT_MALFORMED;
        return;
    }
    uint8_t v;
    if (fl & FL_PK_INF) {
        v = VERDICT_NEEDS_EXACT;
    } else {
        bool x_ok = !(fl & FL_X_BAD);
        // the lane's coefficient k of an Fp6 held in planes p0..p0+2 (ulonglong2 = two coefficients)
        const uint64_t* pl = reinterpret_cast<const uint64_t*>(in.planes);
        size_t n = in.n;
        fp_t sx = pl[((size_t)(0 + (k >> 1)) * n + i) * 2 + (k & 1)];
        fp_t px = pl[((size_t)(5 + (k >> 1)) * n + i) * 2 + (k & 1)];
        fp_t py = pl[((size_t)(8 + (k >> 1)) * n + i) * 2 + (k & 1)];
        scalar e = load_scalar_planes(in.planes, 3, n, i);
        uint64_t off = msg_off[i];
        scalar h = sc_zero();
        if (x_ok) h = dchallenge_scalar(mask, sx, px, py, msgs + off, msg_off[i + 1] - off, k, gbase, s_mds2);
        dpt r;
        int fr = dverify_core(mask, px, py, h, e, gtab, &r, k, gbase);
        bool eq = dall(mask, gbase, r.X == fp_mul(sx, fp_sqr_nc(r.w)));  // x(R) == sig.x  <=>  X == sig.x w^2
        v = fr == FAST_EXCEPTIONAL ? VERDICT_NEEDS_EXACT
            : (fr == FAST_NOT_TORSION_FREE ? VERDICT_INVALID_PUBLIC_KEY
               : (!x_ok ? VERDICT_MALFORMED : (eq ? VERDICT_OK : VERDICT_INVALID_SIGNATURE)));
    }
    if (k == 0) {
        verdicts[i] = v;
        if (v == VERDICT_NEEDS_EXACT) work_list[atomicAdd(work_count, 1u)] = (uint32_t)i;
    }
}


// ------------------------------------------------------------------------------------------------
// K1: hash_message, one message per thread (AoS inputs: 8-byte aligned records)
// ------------------------------------------------------------------------------------------------
static constexpr int HASH_THREADS = 128;
__global__ void __launch_bounds__(HASH_THREADS) k_hash(size_t n, const uint8_t* __restrict__ rx48,
                                                       const uint8_t* __restrict__ pk96,
                                                       const uint8_t* __restrict__ msgs,
                                                       const uint64_t* __restrict__ msg_off,
                                                       uint8_t* __restrict__ digests) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool live = i < n;
    uint64_t off = live ? msg_off[i] : 0, len = live ? msg_off[i + 1] - off : 0;
    // threads past the end of the batch hash the first live thread's message along (every thread reaches the barriers)
    hash_vote hv = block_hash_vote(live ? hash_message_permutations(len) : -1, off, len);
    size_t src = live ? i : (size_t)blockIdx.x * blockDim.x;   // the block's first item always exists
    const uint64_t* r = reinterpret_cast<const uint64_t*>(rx48 + src * 48);
    const uint64_t* p = reinterpret_cast<const uint64_t*>(pk96 + src * 96);
    fp6 rx, px;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        rx.c[k] = r[k];
        px.c[k] = p[k];
    }
    fp_t py0 = p[6];
    fp_t d[4];
    hash_message(rx, px, py0, msgs + off, len, d, hv.sync);
    if (!live) return;
    ulonglong2* o = reinterpret_cast<ulonglong2*>(digests + i * 32);
    o[0] = make_ulonglong2(d[0], d[1]);
    o[1] = make_ulonglong2(d[2], d[3]);
}

// K1 for small calls: one message per group of six lanes (dist.cuh), five messages per warp
__global__ void __launch_bounds__(DIST_THREADS) k_hash_dist(size_t n, const uint8_t* __restrict__ rx48,
                                                            const uint8_t* __restrict__ pk96,
                                                            const uint8_t* __restrict__ msgs,
                                                            const uint64_t* __restrict__ msg_off,
                                                            uint8_t* __restrict__ digests) {
    __shared__ uint32_t s_mds2[24];
    if (threadIdx.x < 24) s_mds2[threadIdx.x] = c_mds_row[threadIdx.x % 12];
    __syncthreads();
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int g = lane / 6, k = lane % 6;
    if (g >= 5) return;
    size_t i = ((size_t)blockIdx.x * (DIST_THREADS / 32) + warp) * 5 + g;
    if (i >= n) return;
    int gbase = 6 * g;
    unsigned mask = 0x3fu << gbase;
    const uint64_t* r = reinterpret_cast<const uint64_t*>(rx48 + i * 48);
    const uint64_t* p = reinterpret_cast<const uint64_t*>(pk96 + i * 96);
    uint64_t off = msg_off[i];
    fp_t d[4];
    dhash_message(mask, r[k], p[k], p[6 + k], msgs + off, msg_off[i + 1] - off, k, gbase, s_mds2, d);
    if (k < 4) reinterpret_cast<uint64_t*>(digests + i * 32)[k] = d[k];
}

// ------------------------------------------------------------------------------------------------
// K5: fixed-base multiplication -> key generation and the device signer
// ------------------------------------------------------------------------------------------------
static constexpr int SIGN_THREADS = 128;
__device__ __forceinline__ void store_point96(uint8_t* dst, const fp6& x, const fp6& y) {
    uint64_t* o = reinterpret_cast<uint64_t*>(dst);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        o[k] = x.c[k];
        o[6 + k] = y.c[k];
    }
}
__global__ void __launch_bounds__(SIGN_THREADS) k_keygen(size_t n, const uint8_t* __restrict__ sk32,
                                                         const uint64_t* __restrict__ gtab, uint8_t* __restrict__ pk96,
                                                         uint8_t* __restrict__ pk_inf) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    scalar k = sc_from_u256(sc_load_le(sk32 + 32 * i));
    jac_pt P = fixed_base_mul(k, gtab);
    fp6 x, y;
    bool inf;
    jac_to_affine(P, x, y, inf);
    store_point96(pk96 + 96 * i, x, y);
    if (pk_inf) pk_inf[i] = inf ? 1 : 0;
}
__global__ void __launch_bounds__(SIGN_THREADS) k_sign(size_t n, const uint8_t* __restrict__ sk32,
                                                       const uint8_t* __restrict__ pk96,
                                                       const uint8_t* __restrict__ pk_inf,
                                                       const uint8_t* __restrict__ msgs,
                                                       const uint64_t* __restrict__ msg_off,
                                                       const uint8_t* __restrict__ nonce32,
                                                       const uint64_t* __restrict__ gtab, uint8_t* __restrict__ sigs81) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    scalar sk = sc_from_u256(sc_load_le(sk32 + 32 * i));
    scalar r = sc_from_u256(sc_load_le(nonce32 + 32 * i));
    const uint64_t* p = reinterpret_cast<const uint64_t*>(pk96 + i * 96);
    fp6 px, py;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        px.c[k] = p[k];
        py.c[k] = p[6 + k];
    }
    bool inf = pk_inf != nullptr && pk_inf[i] != 0;
    jac_pt R = fixed_base_mul(r, gtab);
    fp6 x, y;
    bool r_inf;
    jac_to_affine(R, x, y, r_inf);  // identity -> x = y = 0
    uint64_t off = msg_off[i];
    scalar h = challenge_scalar(x, px, py, inf, msgs + off, msg_off[i + 1] - off);
    scalar e = sc_sub(r, sc_mul(sk, h));
    uint8_t* o = sigs81 + 81 * i;
#pragma unroll
    for (int k = 0; k < 6; k++)
#pragma unroll
        for (int b = 0; b < 8; b++) o[8 * k + b] = (uint8_t)(x.c[k] >> (8 * b));
    o[48] = compress_flags(y, r_inf);
#pragma unroll
    for (int k = 0; k < 8; k++)
#pragma unroll
        for (int b = 0; b < 4; b++) o[49 + 4 * k + b] = (uint8_t)(e.l[k] >> (8 * b));
}

// ------------------------------------------------------------------------------------------------
// compressed point codecs (PublicKey::from_bytes / to_bytes, src/public.rs:49-56)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_decompress(size_t n, const uint8_t* __restrict__ in49, uint8_t* __restrict__ pk96,
                                                    uint8_t* __restrict__ pk_inf, uint8_t* __restrict__ ok) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* rec = in49 + 49 * i;
    fp6 x;
#pragma unroll
    for (int k = 0; k < 6; k++) x.c[k] = load_u64_le(rec + 8 * k);
    fp6 ox, oy;
    bool inf;
    bool good = decompress_point(x, rec[48], ox, oy, inf);
    store_point96(pk96 + 96 * i, ox, oy);
    pk_inf[i] = inf ? 1 : 0;
    ok[i] = good ? 1 : 0;
}
__global__ void __launch_bounds__(128) k_compress(size_t n, const uint8_t* __restrict__ pk96,
                                                  const uint8_t* __restrict__ pk_inf, uint8_t* __restrict__ out49) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t* p = reinterpret_cast<const uint64_t*>(pk96 + i * 96);
    bool inf = pk_inf != nullptr && pk_inf[i] != 0;
    fp6 y;
#pragma unroll
    for (int k = 0; k < 6; k++) y.c[k] = p[6 + k];
    uint8_t* o = out49 + 49 * i;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        uint64_t v = inf ? 0 : p[k];
#pragma unroll
        for (int b = 0; b < 8; b++) o[8 * k + b] = (uint8_t)(v >> (8 * b));
    }
    o[48] = compress_flags(y, inf);
}

// KeyedSignature wire records (src/signature.rs:237-271): 49-byte compressed public key || 81-byte
// signature.  The key is decompressed on the device; records whose key does not decode get verdict 3
// (KeyedSignature::from_bytes returns None for them).
__global__ void __launch_bounds__(128) k_split_keyed(size_t n, const uint8_t* __restrict__ keyed130, uint8_t* __restrict__ pk96,
                                                     uint8_t* __restrict__ pk_inf, uint8_t* __restrict__ ok,
                                                     uint8_t* __restrict__ sigs81) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* rec = keyed130 + 130 * i;
    fp6 x;
#pragma unroll
    for (int k = 0; k < 6; k++) x.c[k] = load_u64_le(rec + 8 * k);
    fp6 ox, oy;
    bool inf;
    bool good = decompress_point(x, rec[48], ox, oy, inf);
    store_point96(pk96 + 96 * i, ox, oy);
    pk_inf[i] = inf ? 1 : 0;
    ok[i] = good ? 1 : 0;
    for (int k = 0; k < 81; k++) sigs81[81 * i + k] = rec[49 + k];
}
__global__ void k_mask_verdicts(size_t n, const uint8_t* __restrict__ ok, uint8_t* __restrict__ verdicts) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !ok[i]) verdicts[i] = VERDICT_MALFORMED;
}
// Batches over keyed records: a record whose key does not decode gets the record of an index outside a set
// (k_keyset_gather), all-ones limbs and identity flag 0, which k_ingest flags as malformed: the batch is malformed, as
// unwrapping KeyedSignature::from_bytes on such a record panics.
__global__ void __launch_bounds__(128) k_keyed_bad_records(size_t n, const uint8_t* __restrict__ ok, uint64_t* __restrict__ pk12,
                                                           uint8_t* __restrict__ pk_inf) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || ok[i]) return;
#pragma unroll
    for (int c = 0; c < 12; c++) pk12[12 * i + c] = ~0ULL;
    pk_inf[i] = 0;
}

// ------------------------------------------------------------------------------------------------
// f4: hierarchical deterministic derivation (src/derivation.rs:66-277), one child per thread (derive.cuh)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_derive_master(size_t n, const uint8_t* __restrict__ seeds32, uint8_t* __restrict__ xsk64,
                                                       uint8_t* __restrict__ ok) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ok[i] = derive_master(seeds32 + 32 * i, xsk64 + 64 * i) ? 1 : 0;
}
// parent49 = PublicKey::from(parent sk).to_bytes(), computed once by k_parent_public below
__global__ void __launch_bounds__(128) k_derive_private(size_t n, const uint8_t* __restrict__ parent_xsk64,
                                                        const uint8_t* __restrict__ parent49, const uint32_t* __restrict__ indices,
                                                        uint8_t* __restrict__ children64, uint8_t* __restrict__ ok) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ok[i] = derive_private_child(parent_xsk64, parent49, indices[i], children64 + 64 * i) ? 1 : 0;
}
__global__ void k_parent_public(const uint8_t* __restrict__ parent_xsk64, const uint64_t* __restrict__ gtab, uint8_t* __restrict__ out49) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    scalar k = sc_from_u256(sc_load_le(parent_xsk64));
    jac_pt P = fixed_base_mul(k, gtab);
    fp6 x, y;
    bool inf;
    jac_to_affine(P, x, y, inf);
    for (int c = 0; c < 6; c++)
        for (int b = 0; b < 8; b++) out49[8 * c + b] = (uint8_t)((inf ? 0 : x.c[c]) >> (8 * b));
    out49[48] = compress_flags(y, inf);
}
// children81 = 49-byte compressed child key || 32-byte chain code; parent96 / parent_inf = the decompressed parent key
__global__ void __launch_bounds__(SIGN_THREADS) k_derive_public(size_t n, const uint8_t* __restrict__ parent_xpk81,
                                                                const uint8_t* __restrict__ parent96,
                                                                const uint8_t* __restrict__ parent_inf,
                                                                const uint32_t* __restrict__ indices,
                                                                const uint64_t* __restrict__ gtab, uint8_t* __restrict__ children81,
                                                                uint8_t* __restrict__ ok) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t index = indices[i];
    uint8_t* o = children81 + 81 * i;
    const uint64_t* p = reinterpret_cast<const uint64_t*>(parent96);
    fp6 px, py;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        px.c[k] = p[k];
        py.c[k] = p[6 + k];
    }
    // the tweak hashes PublicKey::to_bytes of the decoded parent (:255), not the bytes it was given: a 2-torsion parent
    // (y = 0) decodes under either sign bit and re-encodes with the bit clear.  The x limbs of a decodable record are
    // already its canonical encoding.
    uint8_t pk49[49];
    for (int k = 0; k < 48; k++) pk49[k] = parent_xpk81[k];
    pk49[48] = compress_flags(py, parent_inf[0] != 0);
    scalar t = derive_public_tweak(pk49, parent_xpk81 + 49, index, o + 49);
    jac_pt acc = fixed_base_mul(t, gtab);                       // I_L G   (src/derivation.rs:263)
    bool tweak_inf = jac_is_identity(acc);
    acc = jac_madd(acc, px, py, parent_inf[0] != 0);            // + parent key (:264)
    fp6 x, y;
    bool inf;
    jac_to_affine(acc, x, y, inf);
#pragma unroll
    for (int k = 0; k < 6; k++)
#pragma unroll
        for (int b = 0; b < 8; b++) o[8 * k + b] = (uint8_t)((inf ? 0 : x.c[k]) >> (8 * b));
    o[48] = compress_flags(y, inf);
    ok[i] = (!tweak_inf && (index >> 31) == 0) ? 1 : 0;         // :270-275
}

// ------------------------------------------------------------------------------------------------
// signed-window tables of affine multiples (keyset.cuh: tab_bases / tab_entry), for a list of base points:
//   tab[p][i][d] = d * 2^(w i) * P_p,  i < windows,  d < 2^(w-1) + 1  (slot 0 unused)
// The fixed-base table of G (curve.cuh: w = 13, 20 windows) and the per-key tables of registered key sets (KT_W).
// skip[p] != 0 (skip may be NULL): no table for point p (its slots are left as they are).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_tab_bases(size_t n_pts, const uint64_t* __restrict__ pts12, const uint8_t* __restrict__ skip,
                                                   int w, int windows, jac_pt* __restrict__ bases) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pts || (skip && skip[p])) return;
    tab_bases(pts12 + 12 * p, w, windows, bases + p * windows);
}
__global__ void __launch_bounds__(128) k_tab_fill(size_t n_pts, const uint8_t* __restrict__ skip, int w, int windows,
                                                  const jac_pt* __restrict__ bases, uint64_t* __restrict__ tab) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t entries = ((size_t)1 << (w - 1)) + 1, per_pt = (size_t)windows * entries;
    if (t >= n_pts * per_pt) return;
    size_t p = t / per_pt;
    if (skip && skip[p]) return;
    tab_entry(bases[t / entries], w, (int)(t % entries), tab + t * 12);
}

// ------------------------------------------------------------------------------------------------
// registered key sets (keyset.cuh)
// ------------------------------------------------------------------------------------------------
// one thread per key: status (canonical limbs, exact subgroup check) and skip = no table (status != 0 or identity)
__global__ void __launch_bounds__(128) k_keyset_register(size_t n_keys, const uint64_t* __restrict__ pk12,
                                                         const uint8_t* __restrict__ pk_inf, uint8_t* __restrict__ status,
                                                         uint8_t* __restrict__ skip) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_keys) return;
    bool inf = pk_inf[k] != 0;
    jac_pt d;
    uint8_t st = keyset_key_status(pk12 + 12 * k, inf, &d);
    status[k] = st;
    skip[k] = st != KEY_OK || inf;
}
// per item: the key record of key_idx[i] for k_ingest.  An index outside the set gets all-ones limbs, which k_ingest
// flags as malformed (verdict 3: indexing past the end of a slice panics in the reference).
__global__ void __launch_bounds__(128) k_keyset_gather(size_t n, const uint32_t* __restrict__ key_idx, size_t n_keys,
                                                       const uint64_t* __restrict__ ks_pk12, const uint8_t* __restrict__ ks_inf,
                                                       uint64_t* __restrict__ pk12, uint8_t* __restrict__ pk_inf) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k = key_idx[i];
    bool in = k < n_keys;
#pragma unroll
    for (int c = 0; c < 12; c++) pk12[12 * i + c] = in ? ks_pk12[12 * (size_t)k + c] : ~0ULL;
    pk_inf[i] = in ? ks_inf[k] : 0;
}
// one thread per key: the key's lookup entry (keyset_encode) and whether it is findable
__global__ void __launch_bounds__(128) k_keyset_encode(size_t n_keys, const uint64_t* __restrict__ pk12,
                                                       const uint8_t* __restrict__ pk_inf, keyset_entry* __restrict__ entries,
                                                       uint8_t* __restrict__ findable) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_keys) return;
    keyset_entry e;
    uint8_t flag;
    findable[k] = keyset_encode(pk12 + 12 * k, pk_inf[k] != 0, e.x, flag) ? 1 : 0;
    e.flag = flag;
    e.index = (uint32_t)k;
    e.pad = 0;
    entries[k] = e;
}
// Replaced slots: the record, identity flag, status and table of compact key j go to slot idx[j] (a table of zeros for
// keys registered without one).  One 16-byte word per thread.
static constexpr size_t KT_KEY_U128 = KT_KEY_U64 / 2;
__global__ void __launch_bounds__(256) k_keyset_scatter(size_t m, const uint32_t* __restrict__ idx,
                                                        const uint64_t* __restrict__ src_pk12, const uint8_t* __restrict__ src_inf,
                                                        const uint8_t* __restrict__ src_status,
                                                        const ulonglong2* __restrict__ src_tab, uint64_t* __restrict__ pk12,
                                                        uint8_t* __restrict__ pk_inf, uint8_t* __restrict__ status,
                                                        ulonglong2* __restrict__ tab) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m * (KT_KEY_U128 + 13)) return;
    if (t < m * KT_KEY_U128) {
        size_t j = t / KT_KEY_U128, w = t % KT_KEY_U128;
        tab[(size_t)idx[j] * KT_KEY_U128 + w] = src_tab[t];
        return;
    }
    t -= m * KT_KEY_U128;
    size_t j = t / 13, c = t % 13;
    size_t k = idx[j];
    if (c < 12) {
        pk12[12 * k + c] = src_pk12[12 * j + c];
    } else {
        pk_inf[k] = src_inf[j];
        status[k] = src_status[j];
    }
}
// 49-byte compressed keys -> index of the registered key with exactly that encoding, or KEYSET_MISS
__global__ void __launch_bounds__(128) k_keyset_lookup(size_t n, const uint8_t* __restrict__ keys49,
                                                       const keyset_entry* __restrict__ lut, uint32_t n_lut,
                                                       uint32_t* __restrict__ key_idx) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* rec = keys49 + 49 * i;
    uint64_t x[6];
#pragma unroll
    for (int k = 0; k < 6; k++) x[k] = load_u64_le(rec + 8 * k);
    key_idx[i] = keyset_lookup(lut, n_lut, x, rec[48]);
}
// Front end of a keyed call against a registered set (KeyedSignature records, src/signature.rs:237-271): the
// signature bytes, then the key searched in the set.  A hit writes the registered record (as k_keyset_gather) and the
// key index; a miss decompresses the key as k_split_keyed does and writes KEYSET_MISS.  *miss_count += the misses.
__global__ void __launch_bounds__(128) k_keyed_split_lookup(size_t n, const uint8_t* __restrict__ keyed130,
                                                            const keyset_entry* __restrict__ lut, uint32_t n_lut,
                                                            const uint64_t* __restrict__ ks_pk12,
                                                            const uint8_t* __restrict__ ks_inf, uint8_t* __restrict__ pk96,
                                                            uint8_t* __restrict__ pk_inf, uint8_t* __restrict__ ok,
                                                            uint8_t* __restrict__ sigs81, uint32_t* __restrict__ key_idx,
                                                            uint32_t* __restrict__ miss_count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool miss = false;
    if (i < n) {
        const uint8_t* rec = keyed130 + 130 * i;
        fp6 x;
#pragma unroll
        for (int k = 0; k < 6; k++) x.c[k] = load_u64_le(rec + 8 * k);
        uint32_t k = keyset_lookup(lut, n_lut, x.c, rec[48]);
        miss = k == KEYSET_MISS;
        if (!miss) {
            uint64_t* o = reinterpret_cast<uint64_t*>(pk96 + 96 * i);
#pragma unroll
            for (int c = 0; c < 12; c++) o[c] = ks_pk12[12 * (size_t)k + c];
            pk_inf[i] = ks_inf[k];
            ok[i] = 1;
        } else {
            fp6 ox, oy;
            bool inf;
            bool good = decompress_point(x, rec[48], ox, oy, inf);
            store_point96(pk96 + 96 * i, ox, oy);
            pk_inf[i] = inf ? 1 : 0;
            ok[i] = good ? 1 : 0;
        }
        key_idx[i] = k;
        for (int c = 0; c < 81; c++) sigs81[81 * i + c] = rec[49 + c];
    }
    unsigned m = __ballot_sync(0xffffffffu, miss);   // every launch is a whole number of warps
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(miss_count, (unsigned)__popc(m));
}

// Signature::verify against registered keys: the shape of k_verify_fast (block-agreed challenge hash, stand-in inputs
// for threads without work, the same verdicts and hand-back list), with h*P from the key's table instead of the
// doubling chain and no subgroup check (the key's status).  Items handed back are finished by k_verify, which reads
// the key k_keyset_gather placed in the planes.
// LOOKUP: the items of a keyed call (k_keyed_split_lookup), where key_idx[i] == KEYSET_MISS marks a record whose key
// is not in the set: it is handed to k_verify, which reads the key decompressed into the planes.
template <bool LOOKUP>
__global__ void __launch_bounds__(VERIFY_THREADS) k_verify_reg(soa_batch in, const uint32_t* __restrict__ key_idx,
                                                               const uint8_t* __restrict__ key_status,
                                                               const uint64_t* __restrict__ ktab,
                                                               const uint8_t* __restrict__ msgs,
                                                               const uint64_t* __restrict__ msg_off,
                                                               const uint64_t* __restrict__ gtab,
                                                               uint8_t* __restrict__ verdicts,
                                                               uint32_t* __restrict__ work_list,
                                                               uint32_t* __restrict__ work_count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool live = i < in.n;
    uint8_t fl = live ? in.flags[i] : FL_MALFORMED;
    // a record that is not malformed has an index inside the set (k_keyset_gather)
    bool keyed = !(fl & (FL_MALFORMED | FL_PK_INF));
    uint32_t k = keyed ? key_idx[i] : 0;
    bool miss = LOOKUP && k == KEYSET_MISS;
    if (miss) {
        keyed = false;
        k = 0;
    }
    uint8_t st = keyed ? key_status[k] : KEY_OK;
    bool work = keyed && st == KEY_OK;
    uint64_t off = work ? msg_off[i] : 0, len = work ? msg_off[i + 1] - off : 0;
    hash_vote hv = block_hash_vote(work ? hash_message_permutations(len) : -1, off, len);
    fp6 sx = fp6_zero(), px, py;
    scalar e = sc_zero();
    if (work) {
        sx = load_fp6_planes(in.planes, 0, in.n, i);
        e = load_scalar_planes(in.planes, 3, in.n, i);
        px = load_fp6_planes(in.planes, 5, in.n, i);
        py = load_fp6_planes(in.planes, 8, in.n, i);
    } else {  // 1 * G, the first entry of the fixed-base table
        const uint64_t* g = gtab + (size_t)1 * GTAB_ENTRY_U64;
#pragma unroll
        for (int c = 0; c < 6; c++) {
            px.c[c] = g[c];
            py.c[c] = g[6 + c];
        }
    }
    bool x_ok = !(fl & FL_X_BAD);
    scalar h = sc_zero();
    if (hv.any) {  // block-uniform
        h = challenge_scalar(sx, px, py, false, msgs + off, len, hv.sync);
        if (!x_ok || !work) h = sc_zero();
    }
    jf_pt r;
    int fr = verify_core_reg(h, e, ktab + (size_t)k * KT_KEY_U64, gtab, &r);
    if (!live) return;
    uint8_t v;
    if (fl & FL_MALFORMED) v = VERDICT_MALFORMED;
    else if (fl & FL_PK_INF) v = VERDICT_NEEDS_EXACT;   // the identity key is the exact kernel's business
    else if (miss) v = VERDICT_NEEDS_EXACT;
    else v = reg_verdict(st, x_ok, fr, r, sx);
    verdicts[i] = v;
    if (v == VERDICT_NEEDS_EXACT) work_list[atomicAdd(work_count, 1u)] = (uint32_t)i;
}

// ------------------------------------------------------------------------------------------------
// test hook: raw field operations on the device (the PTX paths cannot be exercised on a CPU box)
//   out[i] = { fp6_mul(a,b) (6) | fp6_sqr(a) (6) | a+b (6) | a-b (6) | limb-wise fp_mul (6) | limb-wise fp_sqr(a) (6) |
//              fp6_inv(a) (6) | limb-wise rescue x^(1/7) of a (6) }
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_debug_field(size_t n, const uint64_t* __restrict__ a6, const uint64_t* __restrict__ b6,
                                                     uint64_t* __restrict__ out48) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp6 a, b;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        a.c[k] = a6[i * 6 + k];
        b.c[k] = b6[i * 6 + k];
    }
    fp6 m = fp6_mul(a, b), q = fp6_sqr(a), ad = fp6_add(a, b), su = fp6_sub(a, b), iv = fp6_inv(a);
    uint64_t* o = out48 + i * 48;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        o[k] = m.c[k];
        o[6 + k] = q.c[k];
        o[12 + k] = ad.c[k];
        o[18 + k] = su.c[k];
        o[24 + k] = fp_mul(a.c[k], b.c[k]);
        o[30 + k] = fp_sqr(a.c[k]);
        o[36 + k] = iv.c[k];
        o[42 + k] = rescue_inv_sbox(a.c[k]);
    }
}

// test hook for the lazily reduced forms of the fast path (debug_ops.cuh): out[i] = 8 x 6 limbs
__global__ void __launch_bounds__(128) k_debug_lazy(size_t n, const uint64_t* __restrict__ a6, const uint64_t* __restrict__ b6,
                                                    uint64_t* __restrict__ out48) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp6 a, b, r[8];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        a.c[k] = a6[i * 6 + k];
        b.c[k] = b6[i * 6 + k];
    }
    debug_lazy_ops(a, b, r);
    for (int j = 0; j < 8; j++)
        for (int k = 0; k < 6; k++) out48[i * 48 + 6 * j + k] = r[j].c[k];
}

// ------------------------------------------------------------------------------------------------
// K6: integer-multiply roofline calibration.  8 independent accumulator chains per thread of
// 32x32+64 -> 64 multiply-adds (IMAD.WIDE.U32), no memory traffic.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_imad_peak(int iters, uint64_t* sink) {
    uint32_t a = threadIdx.x * 2654435761u + 12345u, b = blockIdx.x * 40503u + 977u;
    uint64_t acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = k;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[k]) : "r"(a + k), "r"(b));
        }
        b += 3;
    }
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= acc[k];
    if (s == 0x123456789abcdefULL) sink[0] = s;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static inline unsigned grid_for(size_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// tables of n_pts base points (k_tab_bases / k_tab_fill); bases: n_pts * windows Jacobian points of scratch
static int build_tables(schnorr_b200_ctx* ctx, size_t n_pts, const uint64_t* pts12, const uint8_t* skip, int w, int windows,
                        jac_pt* bases, uint64_t* tab) {
    size_t threads = n_pts * (size_t)windows * (((size_t)1 << (w - 1)) + 1);
    k_tab_bases<<<grid_for(n_pts, 128), 128, 0, ctx->stream>>>(n_pts, pts12, skip, w, windows, bases);
    k_tab_fill<<<grid_for(threads, 128), 128, 0, ctx->stream>>>(n_pts, skip, w, windows, bases, tab);
    ctx->launches += 2;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

static int alloc_soa(schnorr_b200_ctx* ctx, size_t n, soa_batch* b) {
    void *p, *f, *sf;
    if (int rc = ensure_scratch(ctx, SL_A, sizeof(ulonglong2) * SOA_PLANES * n, &p)) return rc;
    if (int rc = ensure_scratch(ctx, SL_B, n, &f)) return rc;
    if (int rc = ensure_scratch(ctx, SL_C, n, &sf)) return rc;
    b->planes = (ulonglong2*)p;
    b->flags = (uint8_t*)f;
    b->sig_flag = (uint8_t*)sf;
    b->n = n;
    return 0;
}

// The offset table of a HOST call must start at 0 and be non-decreasing (the reference's `&[&[u8]]` cannot express
// anything else); a bad table would otherwise turn into out-of-bounds device reads.  O(n) on the host.
static bool msg_off_valid(size_t n, const uint64_t* msg_off) {
    if (msg_off[0] != 0) return false;
    for (size_t i = 0; i < n; i++)
        if (msg_off[i + 1] < msg_off[i]) return false;
    return true;
}
#define CHECK_MSG_OFF(ctx, n, msg_off)                                                            \
    do {                                                                                          \
        if (!msg_off_valid((n), (msg_off))) {                                                     \
            (ctx)->err = "message offsets must start at 0 and be non-decreasing";                 \
            return SCHNORR_B200_EARG;                                                             \
        }                                                                                         \
    } while (0)

// host -> device staging helper
static int stage_in(schnorr_b200_ctx* ctx, int slot, const void* host, size_t bytes, void** dev) {
    if (int rc = ensure_scratch(ctx, slot, bytes, dev)) return rc;
    if (host && bytes) CUDA_TRY(ctx, cudaMemcpyAsync(*dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

// Several regions in one scratch slot, each starting on a 256-byte boundary: *dev receives the region's device
// address, and `host` (when not null) is copied there.  A null `host` only reserves the region.
struct stage_region {
    const void* host;
    size_t bytes;
    uint8_t** dev;
};
static int stage_in(schnorr_b200_ctx* ctx, int slot, std::initializer_list<stage_region> regions) {
    auto padded = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t total = 0;
    for (const stage_region& r : regions) total += padded(r.bytes);
    void* blob;
    if (int rc = ensure_scratch(ctx, slot, total, &blob)) return rc;
    uint8_t* p = (uint8_t*)blob;
    for (const stage_region& r : regions) {
        *r.dev = p;
        if (r.host && r.bytes) CUDA_TRY(ctx, cudaMemcpyAsync(p, r.host, r.bytes, cudaMemcpyHostToDevice, ctx->stream));
        p += padded(r.bytes);
    }
    return 0;
}

// the single-device context of device k of a context: the context itself unless it has shards
static schnorr_b200_ctx* device_ctx(schnorr_b200_ctx* ctx, size_t k) { return ctx->shards.empty() ? ctx : ctx->shards[k]; }

#define MULTI_DISPATCH(ctx, call)                                  \
    do {                                                           \
        if ((ctx) && !(ctx)->shards.empty()) return call;          \
    } while (0)
#define NOT_ON_MULTI(ctx)                                                                                          \
    do {                                                                                                           \
        if ((ctx) && !(ctx)->shards.empty()) {                                                                     \
            (ctx)->err = "device-pointer entry points need a single-device context (buffers live on one device)"; \
            return SCHNORR_B200_EARG;                                                                              \
        }                                                                                                          \
    } while (0)

static int verify_many_host(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96, const uint8_t* pk_inf,
                            const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts, bool validate_offsets);
#include "batch.cuh"
#include "multi.cuh"
// K2 for the smallest calls: one thread block per signature (uses the six-lane primitives of dist.cuh and the 24-lane
// Jacobian toolkit of batch.cuh)
#include "one.cuh"
// registration of a few keys: one thread block per key (the phases of k_verify_one)
#include "keyset_block.cuh"


// Signature::verify over an ingested SoA batch: fast path (per-thread or warp-cooperative by call size), then the exact kernel over the handful of
// items it handed back.  `list_base` = first element of this batch in the per-call work list (pipelined chunks
// use disjoint regions), `counter` = index of its counter.
static int launch_verify(schnorr_b200_ctx* ctx, const soa_batch& soa, const uint8_t* msgs, const uint64_t* msg_off,
                         uint8_t* verdicts, size_t list_base, int counter, size_t list_total, cudaStream_t st) {
    unsigned grid = grid_for(soa.n, VERIFY_THREADS);
    if (counter == 0) ctx->exact_counters_used = 0;
    if (ctx->exact_only) {
        k_verify<<<grid, VERIFY_THREADS, 0, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, nullptr, nullptr);
        ctx->launches += 1;
        return 0;
    }
    void* wl;
    if (int rc = ensure_scratch(ctx, SL_M, 4 * (list_total + schnorr_b200_ctx::MAX_CHUNKS), &wl)) return rc;
    uint32_t* counters = (uint32_t*)wl;
    uint32_t* list = counters + schnorr_b200_ctx::MAX_CHUNKS + list_base;
    CUDA_TRY(ctx, cudaMemsetAsync(counters + counter, 0, 4, st));
    if (counter + 1 > ctx->exact_counters_used) ctx->exact_counters_used = counter + 1;
    if (soa.n <= ctx->one_max)
        if (soa.n <= (size_t)2 * ctx->sm_count)   // every block resident at two per SM: the full register budget
            k_verify_one<2><<<(unsigned)soa.n, ONE_THREADS, 0, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, list, counters + counter);
        else
            k_verify_one<4><<<(unsigned)soa.n, ONE_THREADS, 0, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, list, counters + counter);
    else if (soa.n <= ctx->dist_max)
        k_verify_dist<<<grid_for(soa.n, DIST_SIGS_PER_BLOCK), DIST_THREADS, 0, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, list,
                                                                                   counters + counter);
    else
        k_verify_fast<<<grid, VERIFY_THREADS, VERIFY_FAST_SMEM, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, list, counters + counter);
    // the exact kernel sizes itself from the device-side counter: blocks beyond it exit at once
    k_verify<<<grid, VERIFY_THREADS, 0, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, list, counters + counter);
    ctx->launches += 2;
    return 0;
}

extern "C" {

int schnorr_b200_params_pinned(void) { return CHEETAH_PARAMS_PINNED; }
const char* schnorr_b200_params_provenance(void) { return CHEETAH_PARAMS_PROVENANCE; }

int schnorr_b200_create(int device, schnorr_b200_ctx** out) {
    if (!out) return SCHNORR_B200_EARG;
    *out = nullptr;
#if !CHEETAH_PARAMS_PINNED
    {   // once per process: results are bit-exact against the RESTATED oracle only (DESIGN.md 3, INTEGRATION.md 5)
        static bool warned = false;
        if (!warned) {
            warned = true;
            fprintf(stderr, "schnorr_b200: curve / hash parameters are NOT pinned to the upstream cheetah / hash crates (%s). "
                            "Keys and signatures interoperate with the real schnorr-sig crate only after "
                            "rust/dump_params has been run and include/cheetah_params.h regenerated.\n",
                    CHEETAH_PARAMS_PROVENANCE);
        }
    }
#endif
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        (void)cudaGetLastError();
        return SCHNORR_B200_ENODEV;
    }
    schnorr_b200_ctx* ctx = new schnorr_b200_ctx();
    ctx->device = device;
    auto fail = [&](int rc) {
        fprintf(stderr, "schnorr_b200_create: %s\n", ctx->err.c_str());
        schnorr_b200_destroy(ctx);
        return rc;
    };
#define CREATE_TRY(expr)                                                          \
    do {                                                                          \
        cudaError_t e_ = (expr);                                                  \
        if (e_ != cudaSuccess) {                                                  \
            ctx->err = std::string(#expr) + ": " + cudaGetErrorString(e_);        \
            return fail(SCHNORR_B200_ECUDA);                                      \
        }                                                                         \
    } while (0)
    CREATE_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CREATE_TRY(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    CREATE_TRY(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    {
        int per_sm = 0;
        CREATE_TRY(cudaFuncSetAttribute(k_verify_fast, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VERIFY_FAST_SMEM));
        CREATE_TRY(cudaFuncSetAttribute(k_verify_fast, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CREATE_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_verify_fast, VERIFY_THREADS, VERIFY_FAST_SMEM));
        if (per_sm < 1) per_sm = 1;
        ctx->verify_wave = (size_t)ctx->sm_count * per_sm * VERIFY_THREADS;
    }
    CREATE_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CREATE_TRY(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
    CREATE_TRY(cudaEventCreateWithFlags(&ctx->ev_aux, cudaEventDisableTiming));
    for (int c = 0; c < schnorr_b200_ctx::MAX_CHUNKS; c++) CREATE_TRY(cudaEventCreateWithFlags(&ctx->ev_chunk[c], cudaEventDisableTiming));
    CREATE_TRY(cudaEventCreate(&ctx->ev_k0));
    CREATE_TRY(cudaEventCreate(&ctx->ev_k1));
    CREATE_TRY(cudaMemcpyToSymbol(c_ark, RESCUE_ARK, sizeof(uint64_t) * 2 * RESCUE_ROUNDS * 12));
    CREATE_TRY(cudaMemcpyToSymbol(c_q_wnaf5, CHEETAH_Q_WNAF5, sizeof(CHEETAH_Q_WNAF5)));  // the tail of the symbol stays zero
    CREATE_TRY(cudaMemcpyToSymbol(c_q_wnaf4, CHEETAH_Q_WNAF4, 256));
    CREATE_TRY(cudaMalloc(&ctx->gtab, GTAB_U64 * sizeof(uint64_t)));
    jac_pt* bases = nullptr;  // the GTAB_WINDOWS bases, then G itself (12 limbs)
    CREATE_TRY(cudaMalloc(&bases, sizeof(jac_pt) * GTAB_WINDOWS + 96));
    uint64_t* g12 = reinterpret_cast<uint64_t*>(bases + GTAB_WINDOWS);
    CREATE_TRY(cudaMemcpyAsync(g12, CHEETAH_GX, 48, cudaMemcpyHostToDevice, ctx->stream));
    CREATE_TRY(cudaMemcpyAsync(g12 + 6, CHEETAH_GY, 48, cudaMemcpyHostToDevice, ctx->stream));
    if (build_tables(ctx, 1, g12, nullptr, GTAB_W, GTAB_WINDOWS, bases, ctx->gtab)) {
        cudaFree(bases);
        return fail(SCHNORR_B200_ECUDA);
    }
    CREATE_TRY(cudaStreamSynchronize(ctx->stream));
    cudaFree(bases);
#undef CREATE_TRY
    *out = ctx;
    return SCHNORR_B200_OK;
}

int schnorr_b200_create_multi(const int* devices, int n_devices, schnorr_b200_ctx** out) {
    if (!out) return SCHNORR_B200_EARG;
    *out = nullptr;
    if (!devices || n_devices <= 0 || n_devices > 64) return SCHNORR_B200_EARG;
    if (n_devices == 1) return schnorr_b200_create(devices[0], out);
    schnorr_b200_ctx* ctx = new schnorr_b200_ctx();
    ctx->device = devices[0];
    for (int k = 0; k < n_devices; k++) {
        schnorr_b200_ctx* sh = nullptr;
        int rc = schnorr_b200_create(devices[k], &sh);
        if (rc != SCHNORR_B200_OK) {
            schnorr_b200_destroy(ctx);
            return rc;
        }
        ctx->shards.push_back(sh);
    }
    ctx->sm_count = ctx->shards[0]->sm_count;
    ctx->verify_wave = ctx->shards[0]->verify_wave;
    *out = ctx;
    return SCHNORR_B200_OK;
}
int schnorr_b200_device_count(const schnorr_b200_ctx* ctx) { return !ctx ? 0 : (ctx->shards.empty() ? 1 : (int)ctx->shards.size()); }

void schnorr_b200_destroy(schnorr_b200_ctx* ctx) {
    if (!ctx) return;
    if (!ctx->shards.empty()) {
        for (schnorr_b200_ctx* sh : ctx->shards) schnorr_b200_destroy(sh);
        delete ctx;
        return;
    }
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    for (int s = 0; s < SL_COUNT; s++)
        if (ctx->scratch[s]) cudaFree(ctx->scratch[s]);
    if (ctx->gtab) cudaFree(ctx->gtab);
    for (int c = 0; c < schnorr_b200_ctx::MAX_CHUNKS; c++)
        if (ctx->ev_chunk[c]) cudaEventDestroy(ctx->ev_chunk[c]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->ev_aux) cudaEventDestroy(ctx->ev_aux);
    if (ctx->ev_k0) cudaEventDestroy(ctx->ev_k0);
    if (ctx->ev_k1) cudaEventDestroy(ctx->ev_k1);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char* schnorr_b200_last_error(const schnorr_b200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int schnorr_b200_set_stream(schnorr_b200_ctx* ctx, void* stream) {
    if (!ctx) return SCHNORR_B200_EARG;
    NOT_ON_MULTI(ctx);
    ctx->stream = stream ? (cudaStream_t)stream : ctx->own_stream;
    return SCHNORR_B200_OK;
}
int schnorr_b200_synchronize(schnorr_b200_ctx* ctx) {
    if (!ctx) return SCHNORR_B200_EARG;
    for (schnorr_b200_ctx* sh : ctx->shards)
        if (int rc = schnorr_b200_synchronize(sh)) return rc;
    if (!ctx->shards.empty()) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}
uint64_t schnorr_b200_launch_count(const schnorr_b200_ctx* ctx) {
    if (!ctx) return 0;
    uint64_t total = ctx->launches;
    for (const schnorr_b200_ctx* sh : ctx->shards) total += sh->launches;
    return total;
}
int schnorr_b200_last_kernel_ms(schnorr_b200_ctx* ctx, float* ms) {
    if (!ctx || !ms) return SCHNORR_B200_EARG;
    if (!ctx->shards.empty()) {  // the slowest device
        *ms = 0;
        for (schnorr_b200_ctx* sh : ctx->shards) {
            float m = 0;
            if (int rc = schnorr_b200_last_kernel_ms(sh, &m)) return rc;
            if (m > *ms) *ms = m;
        }
        return SCHNORR_B200_OK;
    }
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_k1));
    CUDA_TRY(ctx, cudaEventElapsedTime(ms, ctx->ev_k0, ctx->ev_k1));
    return SCHNORR_B200_OK;
}

int schnorr_b200_set_exact_only(schnorr_b200_ctx* ctx, int exact_only) {
    if (!ctx) return SCHNORR_B200_EARG;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->exact_only = exact_only != 0;
    ctx->exact_only = exact_only != 0;
    return SCHNORR_B200_OK;
}
int schnorr_b200_set_dist_threshold(schnorr_b200_ctx* ctx, size_t max_signatures) {
    if (!ctx) return SCHNORR_B200_EARG;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->dist_max = max_signatures;
    ctx->dist_max = max_signatures;
    return SCHNORR_B200_OK;
}
int schnorr_b200_set_one_threshold(schnorr_b200_ctx* ctx, size_t max_signatures) {
    if (!ctx) return SCHNORR_B200_EARG;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->one_max = max_signatures;
    ctx->one_max = max_signatures;
    return SCHNORR_B200_OK;
}
int schnorr_b200_set_batch_small_threshold(schnorr_b200_ctx* ctx, size_t max_signatures) {
    if (!ctx) return SCHNORR_B200_EARG;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->batch_small_max = max_signatures;
    ctx->batch_small_max = max_signatures;
    return SCHNORR_B200_OK;
}
int schnorr_b200_set_batch_dist_threshold(schnorr_b200_ctx* ctx, size_t max_signatures) {
    if (!ctx) return SCHNORR_B200_EARG;
    ctx->batch_dist_max = max_signatures;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->batch_dist_max = max_signatures;
    return SCHNORR_B200_OK;
}
int schnorr_b200_set_msm_geometry(schnorr_b200_ctx* ctx, int window_bits, unsigned segment_len) {
    if (!ctx || (window_bits != 0 && (window_bits < 4 || window_bits > 16)) || (segment_len != 0 && segment_len < 8))
        return SCHNORR_B200_EARG;
    ctx->msm_c_override = window_bits;
    ctx->msm_t_override = segment_len;
    for (schnorr_b200_ctx* sh : ctx->shards) {
        sh->msm_c_override = window_bits;
        sh->msm_t_override = segment_len;
    }
    return SCHNORR_B200_OK;
}
int schnorr_b200_last_batch_plan(const schnorr_b200_ctx* ctx, int* window_bits, int* windows, unsigned* segment_len) {
    if (!ctx) return SCHNORR_B200_EARG;
    const schnorr_b200_ctx* c = ctx->shards.empty() ? ctx : ctx->shards[0];
    if (window_bits) *window_bits = c->last_msm_c;
    if (windows) *windows = c->last_msm_K;
    if (segment_len) *segment_len = c->last_msm_T;
    return SCHNORR_B200_OK;
}
int schnorr_b200_last_batch_points(const schnorr_b200_ctx* ctx, uint64_t* points) {
    if (!ctx || !points) return SCHNORR_B200_EARG;
    *points = ctx->last_batch_points;
    return SCHNORR_B200_OK;
}
int schnorr_b200_set_registered_batch_threshold(schnorr_b200_ctx* ctx, size_t min_signatures_per_key) {
    if (!ctx) return SCHNORR_B200_EARG;
    ctx->reg_batch_min_per_key = min_signatures_per_key;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->reg_batch_min_per_key = min_signatures_per_key;
    return SCHNORR_B200_OK;
}
int schnorr_b200_last_exact_count(schnorr_b200_ctx* ctx, uint64_t* count) {
    if (!ctx || !count) return SCHNORR_B200_EARG;
    *count = 0;
    if (!ctx->shards.empty()) {
        for (schnorr_b200_ctx* sh : ctx->shards) {
            uint64_t c = 0;
            if (int rc = schnorr_b200_last_exact_count(sh, &c)) return rc;
            *count += c;
        }
        return SCHNORR_B200_OK;
    }
    if (ctx->exact_counters_used == 0 || !ctx->scratch[SL_M]) return SCHNORR_B200_OK;
    uint32_t c[schnorr_b200_ctx::MAX_CHUNKS] = {};
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(ctx, cudaMemcpy(c, ctx->scratch[SL_M], 4 * ctx->exact_counters_used, cudaMemcpyDeviceToHost));
    for (int i = 0; i < ctx->exact_counters_used; i++) *count += c[i];
    return SCHNORR_B200_OK;
}

// ---- hash_messages ---------------------------------------------------------------------------
int schnorr_b200_hash_messages_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* rx48, const uint8_t* pk96,
                                   const uint8_t* msgs, const uint64_t* msg_off, uint8_t* digests) {
    NOT_ON_MULTI(ctx);
    if (!ctx || (n && (!rx48 || !pk96 || !msg_off || !digests))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaEventRecord(ctx->ev_k0, ctx->stream);
    if (n <= ctx->dist_max)
        k_hash_dist<<<grid_for(n, DIST_SIGS_PER_BLOCK), DIST_THREADS, 0, ctx->stream>>>(n, rx48, pk96, msgs, msg_off, digests);
    else
        k_hash<<<grid_for(n, HASH_THREADS), HASH_THREADS, 0, ctx->stream>>>(n, rx48, pk96, msgs, msg_off, digests);
    cudaEventRecord(ctx->ev_k1, ctx->stream);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

int schnorr_b200_hash_messages(schnorr_b200_ctx* ctx, size_t n, const uint8_t* rx48, const uint8_t* pk96,
                               const uint8_t* msgs, const uint64_t* msg_off, uint8_t* digests) {
    MULTI_DISPATCH(ctx, multi_hash_messages(ctx, n, rx48, pk96, msgs, msg_off, digests));
    if (!ctx || (n && (!rx48 || !pk96 || !msg_off || !digests))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CHECK_MSG_OFF(ctx, n, msg_off);
    size_t mb = msg_off[n];
    if (mb && !msgs) return SCHNORR_B200_EARG;
    void *d_rx, *d_pk, *d_m, *d_off, *d_out;
    if (int rc = stage_in(ctx, SL_D, rx48, n * 48, &d_rx)) return rc;
    if (int rc = stage_in(ctx, SL_E, pk96, n * 96, &d_pk)) return rc;
    if (int rc = stage_in(ctx, SL_F, msgs, mb, &d_m)) return rc;
    if (int rc = stage_in(ctx, SL_G, msg_off, (n + 1) * 8, &d_off)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n * 32, &d_out)) return rc;
    if (int rc = schnorr_b200_hash_messages_dev(ctx, n, (uint8_t*)d_rx, (uint8_t*)d_pk, (uint8_t*)d_m, (uint64_t*)d_off,
                                                (uint8_t*)d_out))
        return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(digests, d_out, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

// ---- verify_many -----------------------------------------------------------------------------
int schnorr_b200_verify_many_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                 const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                                 uint8_t* verdicts) {
    NOT_ON_MULTI(ctx);
    if (!ctx || (n && (!sigs81 || !pk96 || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    soa_batch soa;
    if (int rc = alloc_soa(ctx, n, &soa)) return rc;
    k_ingest<<<grid_for(n, INGEST_THREADS), INGEST_THREADS, 0, ctx->stream>>>(n, sigs81, pk96, pk_inf, soa);
    cudaEventRecord(ctx->ev_k0, ctx->stream);
    if (int rc = launch_verify(ctx, soa, msgs, msg_off, verdicts, 0, 0, n, ctx->stream)) return rc;
    cudaEventRecord(ctx->ev_k1, ctx->stream);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

// Host entry point.  Large calls are pipelined: the batch is cut into up to 8 chunks; chunk c+1 is copied
// host->device on a second stream while chunk c is being verified, and each chunk's verdicts are copied
// back as soon as its kernel ends, so the PCIe time hides behind the kernels.
int schnorr_b200_verify_many(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                             const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    MULTI_DISPATCH(ctx, multi_verify_many(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, verdicts));
    if (!ctx || (n && (!sigs81 || !pk96 || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    if (msg_off[0] != 0 || msg_off[n] < msg_off[0]) {
        ctx->err = "message offsets must start at 0 and be non-decreasing";
        return SCHNORR_B200_EARG;
    }
    // the rest of the table is validated chunk by chunk inside the pipeline, behind the kernels of the chunks before
    // (one pass over 2^20 offsets on the calling thread, in front of the first copy, was 1 % of the call)
    return verify_many_host(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, verdicts, true);
}
} // extern "C" (the internal host pipeline below has C++ linkage; it is declared before multi.cuh)

// The pipelined host path on ONE device.  `msg_off` is a table of n + 1 offsets into `msgs` whose first entry may be
// non-zero (the multi-device layer hands every shard its slice of the caller's table as it is) and whose END POINTS the
// caller has checked (msg_off[0] <= msg_off[n] <= size of the blob).  With `validate_offsets` every chunk's part of the
// table is checked right before that chunk is enqueued -- non-decreasing and not beyond msg_off[n], so that no copy and
// no kernel of the chunk leaves the blob -- while the GPU is busy with the chunks before; a bad table ends the call with
// EARG after the work already enqueued has drained.
static int verify_many_host(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                            const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts,
                            bool validate_offsets) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t base = msg_off[0];
    size_t mb = msg_off[n] - base;
    if (mb && !msgs) return SCHNORR_B200_EARG;
    void *d_sig, *d_pk, *d_inf = nullptr, *d_m, *d_off, *d_out;
    if (int rc = ensure_scratch(ctx, SL_D, n * 81, &d_sig)) return rc;
    if (int rc = ensure_scratch(ctx, SL_E, n * 96, &d_pk)) return rc;
    if (int rc = ensure_scratch(ctx, SL_F, mb, &d_m)) return rc;
    if (int rc = ensure_scratch(ctx, SL_G, (n + 1) * 8, &d_off)) return rc;
    if (pk_inf)
        if (int rc = ensure_scratch(ctx, SL_I, n, &d_inf)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n, &d_out)) return rc;
    soa_batch soa;
    if (int rc = alloc_soa(ctx, n, &soa)) return rc;
    // chunk plan in whole kernel waves (no partial-wave tail between chunks): 1, 3, 8 waves, then the rest.
    // Every chunk's copy hides behind the kernels of the chunks before it as long as the host link sustains
    // ~6 GB/s (a wave of 37 888 signatures = 7 MB of input takes ~3.5 ms to verify).
    size_t bounds[5] = {0, n, n, n, n};
    int chunks = 1;
    {
        const size_t w = ctx->verify_wave;
        const size_t cum[3] = {w, 4 * w, 12 * w};
        int k = 0;
        while (k < 3 && n > cum[k] + 2 * w) {
            bounds[k + 1] = cum[k];
            k++;
        }
        bounds[k + 1] = n;
        chunks = k + 1;
    }
    cudaStream_t cs = ctx->copy_stream, ks = ctx->stream, ks2 = ctx->aux_stream;
    // neither the copy stream nor the second compute stream may overtake work of a previous call that still reads the
    // scratch buffers
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_chunk[0], ks));
    CUDA_TRY(ctx, cudaStreamWaitEvent(cs, ctx->ev_chunk[0], 0));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ks2, ctx->ev_chunk[0], 0));
    CUDA_TRY(ctx, cudaMemcpyAsync(d_off, msg_off, (n + 1) * 8, cudaMemcpyHostToDevice, cs));
    for (int c = 0; c < chunks; c++) {
        size_t lo = bounds[c], hi = bounds[c + 1], cn = hi - lo;
        if (validate_offsets) {
            uint64_t bad = msg_off[hi] > msg_off[n];
            for (size_t i = lo; i < hi; i++) bad |= msg_off[i + 1] < msg_off[i];   // branch-free: vectorises
            if (bad) {
                cudaStreamSynchronize(cs);
                cudaStreamSynchronize(ks2);
                cudaStreamSynchronize(ks);
                ctx->err = "message offsets must start at 0 and be non-decreasing";
                return SCHNORR_B200_EARG;
            }
        }
        CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)d_sig + 81 * lo, sigs81 + 81 * lo, cn * 81, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)d_pk + 96 * lo, pk96 + 96 * lo, cn * 96, cudaMemcpyHostToDevice, cs));
        if (pk_inf) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)d_inf + lo, pk_inf + lo, cn, cudaMemcpyHostToDevice, cs));
        size_t b0 = msg_off[lo], b1 = msg_off[hi];
        if (b1 > b0) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)d_m + (b0 - base), msgs + b0, b1 - b0, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_chunk[c], cs));
        // consecutive chunks run on alternating compute streams: the blocks of chunk c + 1 start on the SMs that chunk c
        // is draining instead of waiting for its last block (chunks touch disjoint regions of every buffer)
        cudaStream_t st = (c & 1) ? ks2 : ks;
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_chunk[c], 0));
        soa_batch sc;
        sc.planes = soa.planes + (size_t)SOA_PLANES * lo;   // a private [11][cn] region per chunk
        sc.flags = soa.flags + lo;
        sc.sig_flag = soa.sig_flag + lo;
        sc.n = cn;
        k_ingest<<<grid_for(cn, INGEST_THREADS), INGEST_THREADS, 0, st>>>(cn, (uint8_t*)d_sig + 81 * lo, (uint8_t*)d_pk + 96 * lo,
                                                                         pk_inf ? (uint8_t*)d_inf + lo : nullptr, sc);
        if (st == ks) cudaEventRecord(ctx->ev_k0, ks);
        // the kernels index the message blob with the caller's absolute offsets: shift the device base accordingly
        if (int rc = launch_verify(ctx, sc, (uint8_t*)d_m - base, (uint64_t*)d_off + lo, (uint8_t*)d_out + lo, lo, c, n, st)) return rc;
        if (st == ks) cudaEventRecord(ctx->ev_k1, ks);
        ctx->launches += 1;
    }
    if (chunks > 1) {  // the main stream continues after the second one
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_aux, ks2));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ks, ctx->ev_aux, 0));
    }
    // verdicts come back after EVERY chunk has been enqueued: a device-to-host copy into pageable memory blocks the
    // host until the kernels before it have finished, which would serialise the pipeline above (1 byte per signature:
    // nothing to overlap anyway)
    CUDA_TRY(ctx, cudaMemcpyAsync(verdicts, d_out, n, cudaMemcpyDeviceToHost, ks));
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaStreamSynchronize(ks));
    return SCHNORR_B200_OK;
}
extern "C" {

// ---- KeyedSignature::verify over wire records -------------------------------------------------
int schnorr_b200_verify_keyed_many_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* keyed130, const uint8_t* msgs,
                                       const uint64_t* msg_off, uint8_t* verdicts) {
    NOT_ON_MULTI(ctx);
    if (!ctx || (n && (!keyed130 || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_pk, *d_inf, *d_ok, *d_sig;
    if (int rc = ensure_scratch(ctx, SL_J, n * 96, &d_pk)) return rc;
    if (int rc = ensure_scratch(ctx, SL_K, n * 2, &d_inf)) return rc;
    if (int rc = ensure_scratch(ctx, SL_L, n * 81 + 256, &d_sig)) return rc;
    d_ok = (uint8_t*)d_inf + n;
    k_split_keyed<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, keyed130, (uint8_t*)d_pk, (uint8_t*)d_inf, (uint8_t*)d_ok,
                                                           (uint8_t*)d_sig);
    ctx->launches += 1;
    if (int rc = schnorr_b200_verify_many_dev(ctx, n, (uint8_t*)d_sig, (uint8_t*)d_pk, (uint8_t*)d_inf, msgs, msg_off, verdicts))
        return rc;
    k_mask_verdicts<<<grid_for(n, 256), 256, 0, ctx->stream>>>(n, (uint8_t*)d_ok, verdicts);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}
int schnorr_b200_verify_keyed_many(schnorr_b200_ctx* ctx, size_t n, const uint8_t* keyed130, const uint8_t* msgs,
                                   const uint64_t* msg_off, uint8_t* verdicts) {
    MULTI_DISPATCH(ctx, multi_verify_keyed_many(ctx, n, keyed130, msgs, msg_off, verdicts));
    if (!ctx || (n && (!keyed130 || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CHECK_MSG_OFF(ctx, n, msg_off);
    size_t mb = msg_off[n];
    if (mb && !msgs) return SCHNORR_B200_EARG;
    void *d_rec, *d_m, *d_off, *d_out;
    if (int rc = stage_in(ctx, SL_D, keyed130, n * 130, &d_rec)) return rc;
    if (int rc = stage_in(ctx, SL_F, msgs, mb, &d_m)) return rc;
    if (int rc = stage_in(ctx, SL_G, msg_off, (n + 1) * 8, &d_off)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n, &d_out)) return rc;
    if (int rc = schnorr_b200_verify_keyed_many_dev(ctx, n, (uint8_t*)d_rec, (uint8_t*)d_m, (uint64_t*)d_off, (uint8_t*)d_out))
        return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(verdicts, d_out, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

} // extern "C"

// ---- registered key sets (keyset.cuh) ---------------------------------------------------------
// what one device of the context holds of a set (every device holds the same)
struct keyset_dev {
    int device = 0;
    size_t cap = 0;             // slots allocated (append grows records, status and tables geometrically)
    uint64_t* pk12 = nullptr;   // [cap][12] the registered records, gathered per item ahead of k_ingest
    uint8_t* pk_inf = nullptr;  // [cap]
    uint8_t* status = nullptr;  // [cap] KEY_OK / KEY_NOT_TORSION_FREE / KEY_MALFORMED
    uint64_t* ktab = nullptr;   // [cap][KT_KEY_U64]; zeros for keys without a table and for unused slots
    keyset_entry* lut = nullptr;  // [n_lut] the findable encodings, sorted (keyset.cuh: keyset_lookup)
    uint32_t n_lut = 0;
    size_t lut_cap = 0;
};

struct schnorr_b200_keyset {
    schnorr_b200_ctx* ctx = nullptr;  // the context the set was created on
    size_t n_keys = 0;                // slots, removed ones included
    bool any_not_torsion_free = false;  // a key of status KEY_NOT_TORSION_FREE: batches use the per-signature points
    // host model: the status of every slot, the lookup entry of every slot and whether it is findable, and every
    // findable entry sorted with duplicates (keyset_update_entries)
    std::vector<uint8_t> h_status;
    std::vector<keyset_entry> h_entry;
    std::vector<uint8_t> h_findable;
    std::vector<keyset_entry> h_all;
    std::vector<keyset_dev> devs;     // devs[k] on device_ctx(ctx, k)
};

static void keyset_free(schnorr_b200_keyset* ks) {
    for (keyset_dev& d : ks->devs)
        if (d.pk12 || d.ktab || d.lut) {
            cudaSetDevice(d.device);
            cudaFree(d.pk12);   // pk_inf and status live in the same allocation
            cudaFree(d.ktab);
            cudaFree(d.lut);
        }
    delete ks;
}

// records of `cap` slots: pk12 [cap][12] | pk_inf [cap] | status [cap]
static int keyset_alloc_records(schnorr_b200_ctx* ctx, size_t cap, uint64_t** pk12, uint8_t** pk_inf, uint8_t** status) {
    void* rec;
    CUDA_TRY(ctx, cudaMalloc(&rec, cap * 96 + 2 * cap));
    *pk12 = (uint64_t*)rec;
    *pk_inf = (uint8_t*)rec + cap * 96;
    *status = *pk_inf + cap;
    return 0;
}

// Scratch of a registration of m keys (keyset_register): SL_D skip flags, then the table bases
static size_t keyset_skip_bytes(size_t m) { return (m + 15) / 16 * 16; }
static int keyset_register_scratch(schnorr_b200_ctx* ctx, size_t m, void** tmp) {
    return ensure_scratch(ctx, SL_D, keyset_skip_bytes(m) + m * KT_WINDOWS * sizeof(jac_pt), tmp);
}

// Registration of m keys on one device, the one routine of create, append and replace: status[j] of record j
// (keyset_key_status) and, for keys of status 0 other than the identity, the table at tab + j KT_KEY_U64 (left as it
// is for the others).  Up to ctx->keyset_block_max keys run one block per key (k_keyset_register_block), more one
// thread per key (k_keyset_register, k_tab_bases); k_tab_fill builds the tables.  Scratch: keyset_register_scratch.
static int keyset_register(schnorr_b200_ctx* ctx, size_t m, const uint64_t* pk12, const uint8_t* pk_inf, uint8_t* status,
                           uint64_t* tab) {
    void* tmp;
    if (int rc = keyset_register_scratch(ctx, m, &tmp)) return rc;
    uint8_t* skip = (uint8_t*)tmp;
    jac_pt* bases = (jac_pt*)((uint8_t*)tmp + keyset_skip_bytes(m));
    if (m <= ctx->keyset_block_max) {
        k_keyset_register_block<<<(unsigned)m, ONE_THREADS, 0, ctx->stream>>>(m, pk12, pk_inf, status, skip, bases);
        size_t threads = m * (size_t)KT_WINDOWS * KT_ENTRIES;
        k_tab_fill<<<grid_for(threads, 128), 128, 0, ctx->stream>>>(m, skip, KT_W, KT_WINDOWS, bases, tab);
        ctx->launches += 2;
        CUDA_TRY(ctx, cudaGetLastError());
        return 0;
    }
    k_keyset_register<<<grid_for(m, 128), 128, 0, ctx->stream>>>(m, pk12, pk_inf, status, skip);
    ctx->launches += 1;
    return build_tables(ctx, m, pk12, skip, KT_W, KT_WINDOWS, bases, tab);
}

// Encodings of m records (k_keyset_encode), enqueued with their copies into `entries` / `findable` (host, m each);
// the host may read them after ctx->ev_aux.  Scratch: SL_E.
static int keyset_encode_async(schnorr_b200_ctx* ctx, size_t m, const uint64_t* pk12, const uint8_t* pk_inf,
                               keyset_entry* entries, uint8_t* findable) {
    void* enc;  // lookup entries, then the findable flags
    if (int rc = ensure_scratch(ctx, SL_E, m * (sizeof(keyset_entry) + 1), &enc)) return rc;
    k_keyset_encode<<<grid_for(m, 128), 128, 0, ctx->stream>>>(m, pk12, pk_inf, (keyset_entry*)enc,
                                                              (uint8_t*)enc + m * sizeof(keyset_entry));
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaMemcpyAsync(entries, enc, m * sizeof(keyset_entry), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(findable, (uint8_t*)enc + m * sizeof(keyset_entry), m, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_aux, ctx->stream));
    return 0;
}

// the lookup table `lut` uploaded to one device (the buffer was sized by the caller: lut_cap >= lut.size())
static int keyset_upload_lut(schnorr_b200_ctx* ctx, keyset_dev& kd, const std::vector<keyset_entry>& lut) {
    kd.n_lut = (uint32_t)lut.size();
    if (!lut.empty())
        CUDA_TRY(ctx, cudaMemcpyAsync(kd.lut, lut.data(), lut.size() * sizeof(keyset_entry), cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

// registration of the set's n_keys records on device k (context ctx): copies the records, registers them
// (keyset_register), and builds the lookup table of the encodings (k_keyset_encode; sorted on the host while the key
// tables are built).  Device 0 also fills the host model.
static int keyset_build(schnorr_b200_ctx* ctx, schnorr_b200_keyset* ks, size_t k, const uint8_t* pk96, const uint8_t* pk_inf) {
    const size_t n = ks->n_keys;
    keyset_dev& kd = ks->devs[k];
    kd.device = ctx->device;
    kd.cap = n;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (int rc = keyset_alloc_records(ctx, n, &kd.pk12, &kd.pk_inf, &kd.status)) return rc;
    CUDA_TRY(ctx, cudaMalloc(&kd.ktab, n * KT_KEY_U64 * sizeof(uint64_t)));
    CUDA_TRY(ctx, cudaMemsetAsync(kd.ktab, 0, n * KT_KEY_U64 * sizeof(uint64_t), ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(kd.pk12, pk96, n * 96, cudaMemcpyHostToDevice, ctx->stream));
    if (pk_inf) CUDA_TRY(ctx, cudaMemcpyAsync(kd.pk_inf, pk_inf, n, cudaMemcpyHostToDevice, ctx->stream));
    else CUDA_TRY(ctx, cudaMemsetAsync(kd.pk_inf, 0, n, ctx->stream));
    std::vector<keyset_entry> entries(n);
    std::vector<uint8_t> findable(n);
    if (int rc = keyset_encode_async(ctx, n, kd.pk12, kd.pk_inf, entries.data(), findable.data())) return rc;
    if (int rc = keyset_register(ctx, n, kd.pk12, kd.pk_inf, kd.status, kd.ktab)) return rc;
    if (k == 0) {
        ks->h_status.resize(n);
        CUDA_TRY(ctx, cudaMemcpyAsync(ks->h_status.data(), kd.status, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_aux));
    std::vector<keyset_entry> added, all, lut;
    for (size_t j = 0; j < n; j++)
        if (findable[j]) added.push_back(entries[j]);
    keyset_update_entries(all, nullptr, 0, std::move(added), lut);
    kd.lut_cap = lut.size() ? lut.size() : 1;
    CUDA_TRY(ctx, cudaMalloc(&kd.lut, kd.lut_cap * sizeof(keyset_entry)));
    if (int rc = keyset_upload_lut(ctx, kd, lut)) return rc;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (k == 0) {
        ks->h_entry.swap(entries);
        ks->h_findable.swap(findable);
        ks->h_all.swap(all);
    }
    return 0;
}

// Calls of at most this many items run verify_many's kernels (launch_verify) on the gathered records: at these sizes
// its block-per-signature kernel wins on latency.  Measured on a B200 (1000 W, 1965 MHz; profiles/r3_registered.md):
// 1 / 128 / 384 signatures 0.47 / 0.47 / 0.58 ms there against 0.59 / 0.60 / 0.60 ms in k_verify_reg, 512 signatures
// 0.61 against 0.60 ms.
static constexpr size_t REG_SMALL_MAX = 384;

// the fast kernel over an ingested batch of registered items, then the exact kernel over the items it handed back;
// exact_only and small calls go through launch_verify (same verdicts: the planes hold each item's key record).
// LOOKUP: key_idx may hold KEYSET_MISS (k_keyed_split_lookup); those items are finished by k_verify.
template <bool LOOKUP>
static int launch_verify_registered(schnorr_b200_ctx* ctx, const keyset_dev& kd, const soa_batch& soa,
                                    const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    cudaStream_t st = ctx->stream;
    if (ctx->exact_only || soa.n <= REG_SMALL_MAX) return launch_verify(ctx, soa, msgs, msg_off, verdicts, 0, 0, soa.n, st);
    void* wl;
    if (int rc = ensure_scratch(ctx, SL_M, 4 * (soa.n + schnorr_b200_ctx::MAX_CHUNKS), &wl)) return rc;
    uint32_t* counter = (uint32_t*)wl;
    uint32_t* list = counter + schnorr_b200_ctx::MAX_CHUNKS;
    CUDA_TRY(ctx, cudaMemsetAsync(counter, 0, 4, st));
    ctx->exact_counters_used = 1;
    unsigned grid = grid_for(soa.n, VERIFY_THREADS);
    k_verify_reg<LOOKUP><<<grid, VERIFY_THREADS, 0, st>>>(soa, key_idx, kd.status, kd.ktab, msgs, msg_off, ctx->gtab, verdicts, list, counter);
    k_verify<<<grid, VERIFY_THREADS, 0, st>>>(soa, msgs, msg_off, ctx->gtab, verdicts, list, counter);
    ctx->launches += 2;
    return 0;
}

// device buffers on device k of the set (context ctx), arguments checked by the caller
static int verify_registered_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n, const uint8_t* sigs81,
                                 const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    const keyset_dev& kd = ks->devs[k];
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_pk, *d_inf;
    if (int rc = ensure_scratch(ctx, SL_E, n * 96, &d_pk)) return rc;
    if (int rc = ensure_scratch(ctx, SL_I, n, &d_inf)) return rc;
    soa_batch soa;
    if (int rc = alloc_soa(ctx, n, &soa)) return rc;
    k_keyset_gather<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, key_idx, ks->n_keys, kd.pk12, kd.pk_inf, (uint64_t*)d_pk,
                                                              (uint8_t*)d_inf);
    k_ingest<<<grid_for(n, INGEST_THREADS), INGEST_THREADS, 0, ctx->stream>>>(n, sigs81, (uint8_t*)d_pk, (uint8_t*)d_inf, soa);
    ctx->launches += 2;
    cudaEventRecord(ctx->ev_k0, ctx->stream);
    if (int rc = launch_verify_registered<false>(ctx, kd, soa, key_idx, msgs, msg_off, verdicts)) return rc;
    cudaEventRecord(ctx->ev_k1, ctx->stream);
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// host buffers on device k of the set: staged with cudaMemcpyAsync, verdicts copied back, synchronised
static int verify_registered_host(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n, const uint8_t* sigs81,
                                  const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    size_t mb = msg_off[n];
    void *d_sig, *d_idx, *d_m, *d_off, *d_out;
    if (int rc = stage_in(ctx, SL_D, sigs81, n * 81, &d_sig)) return rc;
    if (int rc = stage_in(ctx, SL_J, key_idx, n * 4, &d_idx)) return rc;
    if (int rc = stage_in(ctx, SL_F, msgs, mb, &d_m)) return rc;
    if (int rc = stage_in(ctx, SL_G, msg_off, (n + 1) * 8, &d_off)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n, &d_out)) return rc;
    if (int rc = verify_registered_dev(ctx, ks, k, n, (uint8_t*)d_sig, (uint32_t*)d_idx, (uint8_t*)d_m, (uint64_t*)d_off,
                                       (uint8_t*)d_out))
        return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(verdicts, d_out, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

#define CHECK_KEYSET(ctx, ks)                                                   \
    do {                                                                        \
        if ((ks)->ctx != (ctx)) {                                               \
            (ctx)->err = "the key set was created on another context";          \
            return SCHNORR_B200_EARG;                                           \
        }                                                                       \
    } while (0)

// whether the host model holds a key of status KEY_NOT_TORSION_FREE
static bool keyset_any_not_torsion_free(const schnorr_b200_keyset* ks) {
    return std::find(ks->h_status.begin(), ks->h_status.end(), KEY_NOT_TORSION_FREE) != ks->h_status.end();
}

// buffers of one device's set that an update allocates before it writes anything
struct keyset_grow {
    uint64_t* pk12 = nullptr;
    uint8_t *pk_inf = nullptr, *status = nullptr;
    uint64_t* ktab = nullptr;
    size_t cap = 0;
    keyset_entry* lut = nullptr;
    size_t lut_cap = 0;
    void *stage = nullptr, *ctab = nullptr;
};
static void keyset_grow_free(int device, keyset_grow& g) {
    cudaSetDevice(device);
    cudaFree(g.pk12);
    cudaFree(g.ktab);
    cudaFree(g.lut);
    g.pk12 = nullptr;
    g.ktab = nullptr;
    g.lut = nullptr;
}

// append (key_idx == NULL: slots n_keys ... n_keys + m - 1) or replace (slots key_idx[j], distinct and inside the set)
// of m keys, on every device; arguments checked by the caller.  The set ends exactly as keyset_create would build it
// from the updated list of records.  Every allocation comes first, so a failure there leaves the set unchanged.  On
// each device: the records are staged (SL_F); an append registers them into its new slots, a replace into a compact
// table (SL_G) that k_keyset_scatter copies to the slots, zeros included.  The first device encodes them; the host
// merges the new lookup entries into its model (keyset_update_entries) and uploads the table to every device.
static int keyset_update(schnorr_b200_ctx* ctx, schnorr_b200_keyset* ks, size_t m, const uint32_t* key_idx,
                         const uint8_t* pk96, const uint8_t* pk_inf, uint8_t* status) {
    const size_t n = ks->n_keys, new_n = key_idx ? n : n + m;
    const size_t lut_need = ks->h_all.size() + m;  // distinct findable encodings after the update, at most
    const size_t stage_bytes = m * 96 + (m + 15) / 16 * 16 + m * 4;
    std::vector<keyset_grow> gr(ks->devs.size());
    auto fail = [&](int rc, size_t d) {
        schnorr_b200_ctx* c = device_ctx(ctx, d);
        if (c != ctx) ctx->err = "device " + std::to_string(c->device) + ": " + c->err;
        for (size_t e = 0; e < gr.size(); e++) keyset_grow_free(ks->devs[e].device, gr[e]);
        return rc;
    };
    // ---- allocations
    for (size_t d = 0; d < ks->devs.size(); d++) {
        schnorr_b200_ctx* c = device_ctx(ctx, d);
        const keyset_dev& s = ks->devs[d];
        keyset_grow& g = gr[d];
        int rc = 0;
        if (cudaSetDevice(c->device) != cudaSuccess) {
            c->err = "cudaSetDevice failed";
            return fail(SCHNORR_B200_ECUDA, d);
        }
        if (new_n > s.cap) {  // geometric growth: repeated appends copy the tables O(log n) times
            g.cap = std::max(new_n, s.cap + s.cap / 2);
            if ((rc = keyset_alloc_records(c, g.cap, &g.pk12, &g.pk_inf, &g.status))) return fail(rc, d);
            if (cudaMalloc(&g.ktab, g.cap * KT_KEY_U64 * sizeof(uint64_t)) != cudaSuccess) {
                c->err = "cudaMalloc of the grown key tables failed";
                return fail(SCHNORR_B200_ECUDA, d);
            }
        }
        if (lut_need > s.lut_cap) {
            g.lut_cap = std::max(lut_need, s.lut_cap + s.lut_cap / 2);
            if (cudaMalloc(&g.lut, g.lut_cap * sizeof(keyset_entry)) != cudaSuccess) {
                c->err = "cudaMalloc of the lookup table failed";
                return fail(SCHNORR_B200_ECUDA, d);
            }
        }
        void* enc;
        if ((rc = ensure_scratch(c, SL_F, stage_bytes, &g.stage))) return fail(rc, d);
        if ((rc = keyset_register_scratch(c, m, &enc))) return fail(rc, d);
        if (d == 0 && (rc = ensure_scratch(c, SL_E, m * (sizeof(keyset_entry) + 1), &enc))) return fail(rc, d);
        if (key_idx && (rc = ensure_scratch(c, SL_G, m * KT_KEY_U64 * sizeof(uint64_t) + m, &g.ctab))) return fail(rc, d);
    }
    // ---- the set is written from here on
    std::vector<keyset_entry> entries(m);
    std::vector<uint8_t> findable(m), st(m);
    std::vector<std::pair<int, void*>> old;  // replaced buffers, freed once every device has synchronised
    for (size_t d = 0; d < ks->devs.size(); d++) {
        schnorr_b200_ctx* c = device_ctx(ctx, d);
        keyset_dev& s = ks->devs[d];
        keyset_grow& g = gr[d];
        cudaStream_t sm = c->stream;
        int rc = 0;
        CUDA_TRY(c, cudaSetDevice(c->device));
        if (g.pk12) {  // one device-to-device copy per buffer; the new tail of the tables is zeros
            CUDA_TRY(c, cudaMemcpyAsync(g.pk12, s.pk12, n * 96, cudaMemcpyDeviceToDevice, sm));
            CUDA_TRY(c, cudaMemcpyAsync(g.pk_inf, s.pk_inf, n, cudaMemcpyDeviceToDevice, sm));
            CUDA_TRY(c, cudaMemcpyAsync(g.status, s.status, n, cudaMemcpyDeviceToDevice, sm));
            CUDA_TRY(c, cudaMemcpyAsync(g.ktab, s.ktab, n * KT_KEY_U64 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, sm));
            CUDA_TRY(c, cudaMemsetAsync(g.ktab + n * KT_KEY_U64, 0, (g.cap - n) * KT_KEY_U64 * sizeof(uint64_t), sm));
            old.emplace_back(c->device, s.pk12);
            old.emplace_back(c->device, s.ktab);
            s.pk12 = g.pk12;
            s.pk_inf = g.pk_inf;
            s.status = g.status;
            s.ktab = g.ktab;
            s.cap = g.cap;
            g.pk12 = nullptr;
            g.ktab = nullptr;
        }
        if (g.lut) {
            old.emplace_back(c->device, s.lut);
            s.lut = g.lut;
            s.lut_cap = g.lut_cap;
            g.lut = nullptr;
        }
        uint64_t* spk = (uint64_t*)g.stage;
        uint8_t* sinf = (uint8_t*)g.stage + m * 96;
        uint32_t* sidx = (uint32_t*)(sinf + (m + 15) / 16 * 16);
        CUDA_TRY(c, cudaMemcpyAsync(spk, pk96, m * 96, cudaMemcpyHostToDevice, sm));
        if (pk_inf) CUDA_TRY(c, cudaMemcpyAsync(sinf, pk_inf, m, cudaMemcpyHostToDevice, sm));
        else CUDA_TRY(c, cudaMemsetAsync(sinf, 0, m, sm));
        if (d == 0 && (rc = keyset_encode_async(c, m, spk, sinf, entries.data(), findable.data()))) return rc;
        uint8_t* new_status;
        if (!key_idx) {
            CUDA_TRY(c, cudaMemcpyAsync(s.pk12 + 12 * n, spk, m * 96, cudaMemcpyDeviceToDevice, sm));
            CUDA_TRY(c, cudaMemcpyAsync(s.pk_inf + n, sinf, m, cudaMemcpyDeviceToDevice, sm));
            new_status = s.status + n;
            if ((rc = keyset_register(c, m, s.pk12 + 12 * n, s.pk_inf + n, new_status, s.ktab + n * KT_KEY_U64))) return rc;
        } else {
            uint64_t* ctab = (uint64_t*)g.ctab;
            new_status = (uint8_t*)(ctab + m * KT_KEY_U64);
            CUDA_TRY(c, cudaMemcpyAsync(sidx, key_idx, m * 4, cudaMemcpyHostToDevice, sm));
            CUDA_TRY(c, cudaMemsetAsync(ctab, 0, m * KT_KEY_U64 * sizeof(uint64_t), sm));
            if ((rc = keyset_register(c, m, spk, sinf, new_status, ctab))) return rc;
            k_keyset_scatter<<<grid_for(m * (KT_KEY_U128 + 13), 256), 256, 0, sm>>>(
                m, sidx, spk, sinf, new_status, (const ulonglong2*)ctab, s.pk12, s.pk_inf, s.status, (ulonglong2*)s.ktab);
            c->launches += 1;
            CUDA_TRY(c, cudaGetLastError());
        }
        if (d == 0) CUDA_TRY(c, cudaMemcpyAsync(st.data(), new_status, m, cudaMemcpyDeviceToHost, sm));
    }
    // ---- the host model and the lookup table
    schnorr_b200_ctx* c0 = device_ctx(ctx, 0);
    CUDA_TRY(c0, cudaSetDevice(c0->device));
    CUDA_TRY(c0, cudaStreamSynchronize(c0->stream));
    std::vector<uint8_t> changed(new_n, 0);
    std::vector<keyset_entry> added, lut;
    ks->h_status.resize(new_n);
    ks->h_entry.resize(new_n);
    ks->h_findable.resize(new_n);
    for (size_t j = 0; j < m; j++) {
        size_t k = key_idx ? key_idx[j] : n + j;
        changed[k] = 1;
        entries[j].index = (uint32_t)k;
        ks->h_status[k] = st[j];
        ks->h_entry[k] = entries[j];
        ks->h_findable[k] = findable[j];
        if (findable[j]) added.push_back(entries[j]);
    }
    keyset_update_entries(ks->h_all, changed.data(), new_n, std::move(added), lut);
    for (size_t d = 0; d < ks->devs.size(); d++) {
        schnorr_b200_ctx* c = device_ctx(ctx, d);
        CUDA_TRY(c, cudaSetDevice(c->device));
        if (int rc = keyset_upload_lut(c, ks->devs[d], lut)) return rc;
    }
    // every device synchronised: work enqueued before the update has finished with the old buffers
    for (size_t d = 0; d < ks->devs.size(); d++) {
        schnorr_b200_ctx* c = device_ctx(ctx, d);
        CUDA_TRY(c, cudaSetDevice(c->device));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    for (auto& o : old) {
        cudaSetDevice(o.first);
        cudaFree(o.second);
    }
    ks->any_not_torsion_free = keyset_any_not_torsion_free(ks);
    ks->n_keys = new_n;
    if (status) memcpy(status, st.data(), m);
    return SCHNORR_B200_OK;
}

extern "C" {

int schnorr_b200_keyset_create(schnorr_b200_ctx* ctx, size_t n_keys, const uint8_t* pk96, const uint8_t* pk_inf,
                               uint8_t* status, schnorr_b200_keyset** out) {
    if (!out) return SCHNORR_B200_EARG;
    *out = nullptr;
    if (!ctx || !pk96 || n_keys == 0 || (uint64_t)n_keys >= ((uint64_t)1 << 32)) return SCHNORR_B200_EARG;
    schnorr_b200_keyset* ks = new schnorr_b200_keyset();
    ks->ctx = ctx;
    ks->n_keys = n_keys;
    ks->devs.resize(schnorr_b200_device_count(ctx));
    // one table per device; the host model and the status come from the first (every device computes the same)
    for (size_t k = 0; k < ks->devs.size(); k++) {
        schnorr_b200_ctx* c = device_ctx(ctx, k);
        if (int rc = keyset_build(c, ks, k, pk96, pk_inf)) {
            if (c != ctx) ctx->err = "device " + std::to_string(c->device) + ": " + c->err;
            keyset_free(ks);
            return rc;
        }
    }
    ks->any_not_torsion_free = keyset_any_not_torsion_free(ks);
    if (status) memcpy(status, ks->h_status.data(), n_keys);
    *out = ks;
    return SCHNORR_B200_OK;
}

void schnorr_b200_keyset_destroy(schnorr_b200_keyset* ks) {
    if (ks) keyset_free(ks);
}

int schnorr_b200_keyset_append(schnorr_b200_ctx* ctx, schnorr_b200_keyset* ks, size_t n, const uint8_t* pk96,
                               const uint8_t* pk_inf, uint8_t* status) {
    if (!ctx || !ks || (n && !pk96)) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n == 0) return SCHNORR_B200_OK;
    if ((uint64_t)ks->n_keys + n >= ((uint64_t)1 << 32)) {
        ctx->err = "a key set holds fewer than 2^32 slots";
        return SCHNORR_B200_EARG;
    }
    return keyset_update(ctx, ks, n, nullptr, pk96, pk_inf, status);
}

int schnorr_b200_keyset_replace(schnorr_b200_ctx* ctx, schnorr_b200_keyset* ks, size_t n, const uint32_t* key_idx,
                                const uint8_t* pk96, const uint8_t* pk_inf, uint8_t* status) {
    if (!ctx || !ks || (n && (!key_idx || !pk96))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n == 0) return SCHNORR_B200_OK;
    std::vector<uint32_t> sorted(key_idx, key_idx + n);
    std::sort(sorted.begin(), sorted.end());
    if (sorted.back() >= ks->n_keys) {
        ctx->err = "a key index is outside the set";
        return SCHNORR_B200_EARG;
    }
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end()) {
        ctx->err = "a key index is repeated in one replace call";
        return SCHNORR_B200_EARG;
    }
    return keyset_update(ctx, ks, n, key_idx, pk96, pk_inf, status);
}

int schnorr_b200_keyset_remove(schnorr_b200_ctx* ctx, schnorr_b200_keyset* ks, size_t n, const uint32_t* key_idx) {
    if (!ctx || !ks || (n && !key_idx)) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n == 0) return SCHNORR_B200_OK;
    std::vector<uint32_t> idx(key_idx, key_idx + n);
    std::sort(idx.begin(), idx.end());
    idx.erase(std::unique(idx.begin(), idx.end()), idx.end());
    if (idx.back() >= ks->n_keys) {
        ctx->err = "a key index is outside the set";
        return SCHNORR_B200_EARG;
    }
    // the removed record: what k_keyset_gather writes for an index outside the set
    std::vector<uint8_t> rec(idx.size() * 96, 0xFF), inf(idx.size(), 0);
    return keyset_update(ctx, ks, idx.size(), idx.data(), rec.data(), inf.data(), nullptr);
}

int schnorr_b200_keyset_debug_export(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, int device_index, size_t first,
                                     size_t count, uint8_t* pk96, uint8_t* pk_inf, uint8_t* status, uint64_t* tables,
                                     uint8_t* lut64, uint32_t* n_lut) {
    if (!ctx || !ks || device_index < 0 || first > ks->n_keys || count > ks->n_keys - first) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (device_index >= (int)ks->devs.size()) return SCHNORR_B200_EARG;
    schnorr_b200_ctx* c = device_ctx(ctx, device_index);
    const keyset_dev& s = ks->devs[device_index];
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (count) {
        if (pk96) CUDA_TRY(c, cudaMemcpyAsync(pk96, s.pk12 + 12 * first, count * 96, cudaMemcpyDeviceToHost, c->stream));
        if (pk_inf) CUDA_TRY(c, cudaMemcpyAsync(pk_inf, s.pk_inf + first, count, cudaMemcpyDeviceToHost, c->stream));
        if (status) CUDA_TRY(c, cudaMemcpyAsync(status, s.status + first, count, cudaMemcpyDeviceToHost, c->stream));
        if (tables)
            CUDA_TRY(c, cudaMemcpyAsync(tables, s.ktab + first * KT_KEY_U64, count * KT_KEY_U64 * sizeof(uint64_t),
                                        cudaMemcpyDeviceToHost, c->stream));
    }
    if (lut64 && s.n_lut)
        CUDA_TRY(c, cudaMemcpyAsync(lut64, s.lut, s.n_lut * sizeof(keyset_entry), cudaMemcpyDeviceToHost, c->stream));
    if (n_lut) *n_lut = s.n_lut;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return SCHNORR_B200_OK;
}

int schnorr_b200_set_keyset_block_threshold(schnorr_b200_ctx* ctx, size_t max_keys) {
    if (!ctx) return SCHNORR_B200_EARG;
    ctx->keyset_block_max = max_keys;
    for (schnorr_b200_ctx* sh : ctx->shards) sh->keyset_block_max = max_keys;
    return SCHNORR_B200_OK;
}

int schnorr_b200_verify_registered_many(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* sigs81,
                                        const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    if (!ctx || !ks || (n && (!sigs81 || !key_idx || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n == 0) return SCHNORR_B200_OK;
    CHECK_MSG_OFF(ctx, n, msg_off);
    if (msg_off[n] && !msgs) return SCHNORR_B200_EARG;
    if (ctx->shards.empty()) return verify_registered_host(ctx, ks, 0, n, sigs81, key_idx, msgs, msg_off, verdicts);
    auto sl = multi_slices(ctx, n);
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        auto off = rebase_offsets(msg_off, s.lo, s.hi);
        return verify_registered_host(ctx->shards[k], ks, k, s.hi - s.lo, sigs81 + 81 * s.lo, key_idx + s.lo,
                                      msgs ? msgs + msg_off[s.lo] : nullptr, off.data(), verdicts + s.lo);
    });
}

int schnorr_b200_verify_registered_many_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                            const uint8_t* sigs81, const uint32_t* key_idx, const uint8_t* msgs,
                                            const uint64_t* msg_off, uint8_t* verdicts) {
    // msgs is required too: the offset table lives on the device, so whether every message is empty is not known here
    if (!ctx || !ks || (n && (!sigs81 || !key_idx || !msgs || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    NOT_ON_MULTI(ctx);
    if (n == 0) return SCHNORR_B200_OK;
    return verify_registered_dev(ctx, ks, 0, n, sigs81, key_idx, msgs, msg_off, verdicts);
}

}  // extern "C"

// ---- KeyedSignature records against a registered key set ----------------------------------------------------------
// A record whose key is in the set takes k_verify_reg with the registered record; every other record (a miss) is
// decompressed and finished by k_verify, the exact kernel, at about 1.8x the cost of k_verify_fast per item.  Host
// calls whose miss fraction is above this run verify_many on the decoded records instead (the verdicts are the same).
// Measured on a B200 (1000 W, 1965 MHz; profiles/r5_keyed_registered.md), 2^20 records, for 1 to 16 384 keys: the
// lookup path takes 21.6-22.0 / 32.2-32.6 / 88.9-89.1 ms at 0 / 1/16 / 1/2 misses against 76.6-76.9 ms for
// verify_keyed_many; the line between the last two points crosses it at 0.41.
static constexpr double KEYED_REG_MAX_MISS_FRACTION = 0.4;

// device buffers, single-device context, arguments checked by the caller.  `select`: read the miss count of the front
// end (synchronises) and take verify_many above KEYED_REG_MAX_MISS_FRACTION.
// Scratch: J decoded keys, K identity / ok flags | key indices | miss counter, L signatures (the slots of
// verify_keyed_many_dev, which small calls run); the kernels after them use A-C and M.
static int verify_keyed_registered_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n,
                                       const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts,
                                       bool select) {
    if (n <= REG_SMALL_MAX) return schnorr_b200_verify_keyed_many_dev(ctx, n, keyed130, msgs, msg_off, verdicts);
    const keyset_dev& kd = ks->devs[k];
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    void *d_pk, *d_sig;
    uint8_t *d_inf, *d_idx, *d_miss;
    if (int rc = ensure_scratch(ctx, SL_J, n * 96, &d_pk)) return rc;
    if (int rc = stage_in(ctx, SL_K, {{nullptr, 2 * n, &d_inf}, {nullptr, 4 * n, &d_idx}, {nullptr, 4, &d_miss}})) return rc;
    if (int rc = ensure_scratch(ctx, SL_L, n * 81 + 256, &d_sig)) return rc;
    uint8_t* d_ok = d_inf + n;
    CUDA_TRY(ctx, cudaMemsetAsync(d_miss, 0, 4, st));
    k_keyed_split_lookup<<<grid_for(n, 128), 128, 0, st>>>(n, keyed130, kd.lut, kd.n_lut, kd.pk12, kd.pk_inf, (uint8_t*)d_pk,
                                                          d_inf, d_ok, (uint8_t*)d_sig, (uint32_t*)d_idx, (uint32_t*)d_miss);
    ctx->launches += 1;
    bool lookup_path = true;
    if (select) {
        uint32_t misses = 0;
        CUDA_TRY(ctx, cudaMemcpyAsync(&misses, d_miss, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(ctx, cudaStreamSynchronize(st));
        lookup_path = misses <= KEYED_REG_MAX_MISS_FRACTION * (double)n;
    }
    if (lookup_path) {
        soa_batch soa;
        if (int rc = alloc_soa(ctx, n, &soa)) return rc;
        k_ingest<<<grid_for(n, INGEST_THREADS), INGEST_THREADS, 0, st>>>(n, (uint8_t*)d_sig, (uint8_t*)d_pk, d_inf, soa);
        ctx->launches += 1;
        cudaEventRecord(ctx->ev_k0, st);
        if (int rc = launch_verify_registered<true>(ctx, kd, soa, (uint32_t*)d_idx, msgs, msg_off, verdicts)) return rc;
        cudaEventRecord(ctx->ev_k1, st);
    } else if (int rc = schnorr_b200_verify_many_dev(ctx, n, (uint8_t*)d_sig, (uint8_t*)d_pk, d_inf, msgs, msg_off, verdicts)) {
        return rc;
    }
    k_mask_verdicts<<<grid_for(n, 256), 256, 0, st>>>(n, d_ok, verdicts);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// host buffers on device k of the set: staged in D, F, G, verdicts in H, synchronised
static int verify_keyed_registered_host(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n,
                                        const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    size_t mb = msg_off[n];
    void *d_rec, *d_m, *d_off, *d_out;
    if (int rc = stage_in(ctx, SL_D, keyed130, n * 130, &d_rec)) return rc;
    if (int rc = stage_in(ctx, SL_F, msgs, mb, &d_m)) return rc;
    if (int rc = stage_in(ctx, SL_G, msg_off, (n + 1) * 8, &d_off)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n, &d_out)) return rc;
    if (int rc = verify_keyed_registered_dev(ctx, ks, k, n, (uint8_t*)d_rec, (uint8_t*)d_m, (uint64_t*)d_off, (uint8_t*)d_out, true))
        return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(verdicts, d_out, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" {

int schnorr_b200_keyset_lookup(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* keys49,
                               uint32_t* key_idx) {
    if (!ctx || !ks || (n && (!keys49 || !key_idx))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n == 0) return SCHNORR_B200_OK;
    schnorr_b200_ctx* c = device_ctx(ctx, 0);
    const keyset_dev& kd = ks->devs[0];
    CUDA_TRY(c, cudaSetDevice(c->device));
    void *d_in, *d_out;
    if (int rc = stage_in(c, SL_D, keys49, n * 49, &d_in)) return rc;
    if (int rc = ensure_scratch(c, SL_H, n * 4, &d_out)) return rc;
    k_keyset_lookup<<<grid_for(n, 128), 128, 0, c->stream>>>(n, (uint8_t*)d_in, kd.lut, kd.n_lut, (uint32_t*)d_out);
    c->launches += 1;
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(key_idx, d_out, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return SCHNORR_B200_OK;
}

int schnorr_b200_keyset_lookup_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* keys49,
                                   uint32_t* key_idx) {
    if (!ctx || !ks || (n && (!keys49 || !key_idx))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    NOT_ON_MULTI(ctx);
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    k_keyset_lookup<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, keys49, ks->devs[0].lut, ks->devs[0].n_lut, key_idx);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

int schnorr_b200_verify_keyed_registered_many(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                              const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off,
                                              uint8_t* verdicts) {
    if (!ctx || !ks || (n && (!keyed130 || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n == 0) return SCHNORR_B200_OK;
    CHECK_MSG_OFF(ctx, n, msg_off);
    if (msg_off[n] && !msgs) return SCHNORR_B200_EARG;
    if (ctx->shards.empty()) return verify_keyed_registered_host(ctx, ks, 0, n, keyed130, msgs, msg_off, verdicts);
    auto sl = multi_slices(ctx, n);
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        auto off = rebase_offsets(msg_off, s.lo, s.hi);
        return verify_keyed_registered_host(ctx->shards[k], ks, k, s.hi - s.lo, keyed130 + 130 * s.lo,
                                            msgs ? msgs + msg_off[s.lo] : nullptr, off.data(), verdicts + s.lo);
    });
}

int schnorr_b200_verify_keyed_registered_many_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                                  const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off,
                                                  uint8_t* verdicts) {
    // msgs is required too: the offset table lives on the device, so whether every message is empty is not known here
    if (!ctx || !ks || (n && (!keyed130 || !msgs || !msg_off || !verdicts))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    NOT_ON_MULTI(ctx);
    if (n == 0) return SCHNORR_B200_OK;
    return verify_keyed_registered_dev(ctx, ks, 0, n, keyed130, msgs, msg_off, verdicts, false);
}

}  // extern "C"

// ---- batch verification against a registered key set (src/batch.rs:84-130) -------------------------------------------
// The key side aggregated per key (batch.cuh: k_keyset_scalar_sum, k_keyset_batch_term, keyset.cuh) needs [q]P_k = O for
// every key, and pays up to one table product per key of the set for the n MSM points it saves.  Otherwise the items'
// key records are gathered and the batch runs the per-signature pipeline unchanged, as do batches small enough for
// the block-per-signature kernel (k_batch_small, the latency form).
static bool reg_batch_aggregates(const schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n) {
    return n > ctx->batch_small_max && !ks->any_not_torsion_free && n / ks->n_keys >= ctx->reg_batch_min_per_key;
}

// The key side of an aggregated batch on device k of the set, in slot O: per-block key terms | column sums, key partial,
// MSM partial, 64 zero bytes | for keyed records (miss_count != null) the route buffers of k_keyed_route.  The MSM is
// planned for msm_points points.
static int reg_batch_setup(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n, const uint32_t* key_idx,
                           const uint32_t* miss_count, size_t msm_points, reg_batch* rb) {
    size_t max_blocks = (size_t)2 * ctx->sm_count, want = (ks->n_keys + KEYTERM_THREADS / 32 - 1) / (KEYTERM_THREADS / 32);
    unsigned blocks = (unsigned)(want < max_blocks ? want : max_blocks);
    const size_t sz_cols = ks->n_keys * 8 * sizeof(unsigned long long);
    size_t r = miss_count ? n : 0;   // route buffers
    uint8_t *d_terms, *d_cols, *d_miss, *d_pos, *d_tiles, *d_tk, *d_mpts, *d_msc;
    if (int rc = stage_in(ctx, SL_O, {{nullptr, (size_t)blocks * sizeof(jac_pt), &d_terms},
                                      {nullptr, sz_cols + 192 + 192 + 64, &d_cols},
                                      {nullptr, r * 4, &d_miss},
                                      {nullptr, r * 4, &d_pos},
                                      {nullptr, (r + SCAN_TILE - 1) / SCAN_TILE * 4, &d_tiles},
                                      {nullptr, r * 32, &d_tk},
                                      {nullptr, r * 96, &d_mpts},
                                      {nullptr, r * 32, &d_msc}}))
        return rc;
    rb->key_idx = key_idx;
    rb->n_keys = ks->n_keys;
    rb->ktab = ks->devs[k].ktab;
    rb->cols = (unsigned long long*)d_cols;
    rb->terms = (uint64_t*)d_terms;
    rb->term_blocks = blocks;
    rb->key_partial = (uint64_t*)(d_cols + sz_cols);
    rb->msm_partial = rb->key_partial + 24;
    rb->zero = (const uint32_t*)(rb->msm_partial + 24);
    rb->msm_points = msm_points;
    rb->miss_count = miss_count;
    rb->miss = (uint32_t*)d_miss;
    rb->pos = (uint32_t*)d_pos;
    rb->tile_total = (uint32_t*)d_tiles;
    rb->tk = (uint32_t*)d_tk;
    rb->mpts = (uint64_t*)d_mpts;
    rb->msc = (uint32_t*)d_msc;
    CUDA_TRY(ctx, cudaMemsetAsync((void*)rb->zero, 0, 64, ctx->stream));
    return SCHNORR_B200_OK;
}

// one 192-byte partial of a registered batch of n > 0 signatures on device buffers of device k of the set (arguments
// checked)
static int batch_partial_registered(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n, const uint8_t* sigs81,
                                    const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32,
                                    uint8_t* partial192, uint64_t* rhs_pre) {
    const keyset_dev& kd = ks->devs[k];
    cudaStream_t st = ctx->stream;
    uint8_t *d_pk, *d_inf;
    if (int rc = stage_in(ctx, SL_N, {{nullptr, n * 96, &d_pk}, {nullptr, n, &d_inf}})) return rc;
    k_keyset_gather<<<grid_for(n, 128), 128, 0, st>>>(n, key_idx, ks->n_keys, kd.pk12, kd.pk_inf, (uint64_t*)d_pk, d_inf);
    ctx->launches += 1;
    if (!reg_batch_aggregates(ctx, ks, n))
        return batch_partial_impl(ctx, n, sigs81, d_pk, d_inf, msgs, msg_off, rand32, partial192, rhs_pre);
    reg_batch rb;
    if (int rc = reg_batch_setup(ctx, ks, k, n, key_idx, nullptr, n, &rb)) return rc;
    return batch_partial_impl(ctx, n, sigs81, d_pk, d_inf, msgs, msg_off, rand32, partial192, rhs_pre, &rb);
}

// host inputs (n > 0, offsets checked) -> staged in slot H -> one partial at `partial` (device memory of this context)
static int batch_partial_registered_host(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n,
                                         const uint8_t* sigs81, const uint32_t* key_idx, const uint8_t* msgs,
                                         const uint64_t* msg_off, const uint8_t* rand32, uint8_t* partial, uint64_t* rhs_pre) {
    uint8_t *d_sig, *d_idx, *d_m, *d_off, *d_rand;
    if (int rc = stage_in(ctx, SL_H, {{sigs81, n * 81, &d_sig}, {key_idx, n * 4, &d_idx}, {msgs, msg_off[n], &d_m},
                                      {msg_off, (n + 1) * 8, &d_off}, {rand32, n * 32, &d_rand}}))
        return rc;
    return batch_partial_registered(ctx, ks, k, n, d_sig, (uint32_t*)d_idx, d_m, (uint64_t*)d_off, d_rand, partial, rhs_pre);
}

extern "C" {

int schnorr_b200_verify_batch_registered(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* sigs81,
                                         const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off,
                                         const uint8_t* rand32, int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    if (!ctx || !ks || !verdict || (n && (!sigs81 || !key_idx || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n) {
        CHECK_MSG_OFF(ctx, n, msg_off);
        if (msg_off[n] && !msgs) return SCHNORR_B200_EARG;
    }
    if (!ctx->shards.empty())
        return multi_verify_batch(ctx, n, msg_off, verdict, lhs97, rhs97, [&](int k, auto s, const uint64_t* off, uint8_t* partial) {
            return batch_partial_registered_host(ctx->shards[k], ks, k, s.hi - s.lo, sigs81 + 81 * s.lo, key_idx + s.lo,
                                                 msgs ? msgs + msg_off[s.lo] : nullptr, off, rand32 + 32 * s.lo, partial, nullptr);
        });
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    uint8_t* res = nullptr;
    if (int rc = batch_whole(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
            return batch_partial_registered_host(ctx, ks, 0, n, sigs81, key_idx, msgs, msg_off, rand32, partial, rhs_pre);
        }, res))
        return rc;
    return read_result(ctx, res, verdict, lhs97, rhs97);
}

int schnorr_b200_verify_batch_registered_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                             const uint8_t* sigs81, const uint32_t* key_idx, const uint8_t* msgs,
                                             const uint64_t* msg_off, const uint8_t* rand32, uint8_t* result216) {
    if (!ctx || !ks || !result216 || (n && (!sigs81 || !key_idx || !msgs || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    NOT_ON_MULTI(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return batch_whole(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
        return batch_partial_registered(ctx, ks, 0, n, sigs81, key_idx, msgs, msg_off, rand32, partial, rhs_pre);
    }, result216);
}

// localisation on the first device: the inputs staged in slot M, the items' key records gathered into slot N, then the
// per-signature bisection of schnorr_b200_locate_invalid_dev (which uses neither slot)
int schnorr_b200_locate_invalid_registered(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* sigs81,
                                           const uint32_t* key_idx, const uint8_t* msgs, const uint64_t* msg_off,
                                           const uint8_t* rand32, uint8_t* flags, uint64_t* n_bad) {
    if (!ctx || !ks || (n && (!sigs81 || !key_idx || !msg_off || !rand32 || !flags))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    if (n_bad) *n_bad = 0;
    if (n == 0) return SCHNORR_B200_OK;
    CHECK_MSG_OFF(ctx, n, msg_off);
    size_t mb = msg_off[n];
    if (mb && !msgs) return SCHNORR_B200_EARG;
    schnorr_b200_ctx* c = device_ctx(ctx, 0);
    const keyset_dev& kd = ks->devs[0];
    CUDA_TRY(c, cudaSetDevice(c->device));
    uint8_t *d_sig, *d_idx, *d_m, *d_off, *d_rand, *d_flags, *d_pk, *d_inf;
    if (int rc = stage_in(c, SL_M, {{sigs81, n * 81, &d_sig}, {key_idx, n * 4, &d_idx}, {msgs, mb, &d_m}, {msg_off, (n + 1) * 8, &d_off},
                                    {rand32, n * 32, &d_rand}, {nullptr, n, &d_flags}}))
        return rc;
    if (int rc = stage_in(c, SL_N, {{nullptr, n * 96, &d_pk}, {nullptr, n, &d_inf}})) return rc;
    k_keyset_gather<<<grid_for(n, 128), 128, 0, c->stream>>>(n, (uint32_t*)d_idx, ks->n_keys, kd.pk12, kd.pk_inf, (uint64_t*)d_pk,
                                                            d_inf);
    c->launches += 1;
    return locate_invalid_staged(ctx, n, d_sig, d_pk, d_inf, d_m, (const uint64_t*)d_off, d_rand, d_flags, flags, n_bad);
}

}  // extern "C"

// ---- batch verification over KeyedSignature records (src/signature.rs:237-271, src/batch.rs:31-130) -----------------
// The front end writes, in slot N, the records verify_batch sees: the signature bytes and the decoded key -- key k's
// registered record where the key bytes are the encoding of a findable key k of `ks` (the same bytes decompression
// gives) -- or, where the key does not decode, the record of an index outside a set, which makes the batch malformed.
// With a set, idx holds each record's key index or KEYSET_MISS, and *miss the number of misses.
struct keyed_front {
    uint8_t *pk, *inf, *sig, *idx, *miss;
};
static int keyed_front_end(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n, const uint8_t* keyed130,
                           keyed_front* f) {
    cudaStream_t st = ctx->stream;
    uint8_t* ok;
    if (int rc = stage_in(ctx, SL_N, {{nullptr, n * 96, &f->pk}, {nullptr, n, &f->inf}, {nullptr, n, &ok}, {nullptr, n * 81, &f->sig},
                                      {nullptr, ks ? n * 4 : 0, &f->idx}, {nullptr, 4, &f->miss}}))
        return rc;
    if (ks) {
        const keyset_dev& kd = ks->devs[k];
        CUDA_TRY(ctx, cudaMemsetAsync(f->miss, 0, 4, st));
        k_keyed_split_lookup<<<grid_for(n, 128), 128, 0, st>>>(n, keyed130, kd.lut, kd.n_lut, kd.pk12, kd.pk_inf, f->pk, f->inf,
                                                              ok, f->sig, (uint32_t*)f->idx, (uint32_t*)f->miss);
    } else {
        k_split_keyed<<<grid_for(n, 128), 128, 0, st>>>(n, keyed130, f->pk, f->inf, ok, f->sig);
    }
    k_keyed_bad_records<<<grid_for(n, 128), 128, 0, st>>>(n, ok, (uint64_t*)f->pk, f->inf);
    ctx->launches += 2;
    return SCHNORR_B200_OK;
}

// One 192-byte partial of a batch over n > 0 keyed records on device buffers (arguments checked), against device k's
// copy of `ks` when a set is given.  Under the rules of reg_batch_aggregates the hits' key side is summed per key and
// the MSM runs over the n points R_i and the misses' -P_i (k_keyed_route); otherwise the front-end records take the
// per-signature pipeline.  read_misses (host forms): read the miss count, which synchronises, and plan the MSM for
// n + m points; the _dev forms plan for 2n.
static int batch_partial_keyed(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n, const uint8_t* keyed130,
                               const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32, uint8_t* partial192,
                               uint64_t* rhs_pre, bool read_misses) {
    keyed_front f;
    if (int rc = keyed_front_end(ctx, ks, k, n, keyed130, &f)) return rc;
    if (!ks || !reg_batch_aggregates(ctx, ks, n))
        return batch_partial_impl(ctx, n, f.sig, f.pk, f.inf, msgs, msg_off, rand32, partial192, rhs_pre);
    size_t points = 2 * n;
    if (read_misses) {
        uint32_t m = 0;
        CUDA_TRY(ctx, cudaMemcpyAsync(&m, f.miss, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        points = n + m;
    }
    reg_batch rb;
    if (int rc = reg_batch_setup(ctx, ks, k, n, (const uint32_t*)f.idx, (const uint32_t*)f.miss, points, &rb)) return rc;
    return batch_partial_impl(ctx, n, f.sig, f.pk, f.inf, msgs, msg_off, rand32, partial192, rhs_pre, &rb);
}

// host inputs (n > 0, offsets checked) -> staged in slot H -> one partial at `partial` (device memory of this context)
static int batch_partial_keyed_host(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t k, size_t n,
                                    const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32,
                                    uint8_t* partial, uint64_t* rhs_pre) {
    uint8_t *d_rec, *d_m, *d_off, *d_rand;
    if (int rc = stage_in(ctx, SL_H, {{keyed130, n * 130, &d_rec}, {msgs, msg_off[n], &d_m}, {msg_off, (n + 1) * 8, &d_off},
                                      {rand32, n * 32, &d_rand}}))
        return rc;
    return batch_partial_keyed(ctx, ks, k, n, d_rec, d_m, (uint64_t*)d_off, d_rand, partial, rhs_pre, true);
}

// the host forms, with or without a set (ks checked by the caller)
static int verify_batch_keyed_host(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* keyed130,
                                   const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32, int* verdict,
                                   uint8_t* lhs97, uint8_t* rhs97) {
    if (n) {
        CHECK_MSG_OFF(ctx, n, msg_off);
        if (msg_off[n] && !msgs) return SCHNORR_B200_EARG;
    }
    if (!ctx->shards.empty())
        return multi_verify_batch(ctx, n, msg_off, verdict, lhs97, rhs97, [&](int k, auto s, const uint64_t* off, uint8_t* partial) {
            return batch_partial_keyed_host(ctx->shards[k], ks, k, s.hi - s.lo, keyed130 + 130 * s.lo,
                                            msgs ? msgs + msg_off[s.lo] : nullptr, off, rand32 + 32 * s.lo, partial, nullptr);
        });
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    uint8_t* res = nullptr;
    if (int rc = batch_whole(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
            return batch_partial_keyed_host(ctx, ks, 0, n, keyed130, msgs, msg_off, rand32, partial, rhs_pre);
        }, res))
        return rc;
    return read_result(ctx, res, verdict, lhs97, rhs97);
}

// localisation on the first device: the inputs staged in slot M, the front-end records in slot N, then the bisection of
// schnorr_b200_locate_invalid_dev (which uses neither slot)
static int locate_invalid_keyed_host(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n, const uint8_t* keyed130,
                                     const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32, uint8_t* flags,
                                     uint64_t* n_bad) {
    if (n_bad) *n_bad = 0;
    if (n == 0) return SCHNORR_B200_OK;
    CHECK_MSG_OFF(ctx, n, msg_off);
    size_t mb = msg_off[n];
    if (mb && !msgs) return SCHNORR_B200_EARG;
    schnorr_b200_ctx* c = device_ctx(ctx, 0);
    CUDA_TRY(c, cudaSetDevice(c->device));
    uint8_t *d_rec, *d_m, *d_off, *d_rand, *d_flags;
    if (int rc = stage_in(c, SL_M, {{keyed130, n * 130, &d_rec}, {msgs, mb, &d_m}, {msg_off, (n + 1) * 8, &d_off},
                                    {rand32, n * 32, &d_rand}, {nullptr, n, &d_flags}}))
        return rc;
    keyed_front f;
    if (int rc = keyed_front_end(c, ks, 0, n, d_rec, &f)) {
        if (c != ctx) ctx->err = c->err;
        return rc;
    }
    return locate_invalid_staged(ctx, n, f.sig, f.pk, f.inf, d_m, (const uint64_t*)d_off, d_rand, d_flags, flags, n_bad);
}

extern "C" {

int schnorr_b200_verify_batch_keyed(schnorr_b200_ctx* ctx, size_t n, const uint8_t* keyed130, const uint8_t* msgs,
                                    const uint64_t* msg_off, const uint8_t* rand32, int* verdict, uint8_t* lhs97,
                                    uint8_t* rhs97) {
    if (!ctx || !verdict || (n && (!keyed130 || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    return verify_batch_keyed_host(ctx, nullptr, n, keyed130, msgs, msg_off, rand32, verdict, lhs97, rhs97);
}

int schnorr_b200_verify_batch_keyed_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* keyed130, const uint8_t* msgs,
                                        const uint64_t* msg_off, const uint8_t* rand32, uint8_t* result216) {
    if (!ctx || !result216 || (n && (!keyed130 || !msgs || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    NOT_ON_MULTI(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return batch_whole(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
        return batch_partial_keyed(ctx, nullptr, 0, n, keyed130, msgs, msg_off, rand32, partial, rhs_pre, false);
    }, result216);
}

int schnorr_b200_verify_batch_keyed_registered(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                               const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off,
                                               const uint8_t* rand32, int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    if (!ctx || !ks || !verdict || (n && (!keyed130 || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    return verify_batch_keyed_host(ctx, ks, n, keyed130, msgs, msg_off, rand32, verdict, lhs97, rhs97);
}

int schnorr_b200_verify_batch_keyed_registered_dev(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                                   const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off,
                                                   const uint8_t* rand32, uint8_t* result216) {
    if (!ctx || !ks || !result216 || (n && (!keyed130 || !msgs || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    NOT_ON_MULTI(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return batch_whole(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
        return batch_partial_keyed(ctx, ks, 0, n, keyed130, msgs, msg_off, rand32, partial, rhs_pre, false);
    }, result216);
}

int schnorr_b200_locate_invalid_keyed(schnorr_b200_ctx* ctx, size_t n, const uint8_t* keyed130, const uint8_t* msgs,
                                      const uint64_t* msg_off, const uint8_t* rand32, uint8_t* flags, uint64_t* n_bad) {
    if (!ctx || (n && (!keyed130 || !msg_off || !rand32 || !flags))) return SCHNORR_B200_EARG;
    return locate_invalid_keyed_host(ctx, nullptr, n, keyed130, msgs, msg_off, rand32, flags, n_bad);
}

int schnorr_b200_locate_invalid_keyed_registered(schnorr_b200_ctx* ctx, const schnorr_b200_keyset* ks, size_t n,
                                                 const uint8_t* keyed130, const uint8_t* msgs, const uint64_t* msg_off,
                                                 const uint8_t* rand32, uint8_t* flags, uint64_t* n_bad) {
    if (!ctx || !ks || (n && (!keyed130 || !msg_off || !rand32 || !flags))) return SCHNORR_B200_EARG;
    CHECK_KEYSET(ctx, ks);
    return locate_invalid_keyed_host(ctx, ks, n, keyed130, msgs, msg_off, rand32, flags, n_bad);
}

// ---- keygen / sign ---------------------------------------------------------------------------
int schnorr_b200_keygen_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sk32, uint8_t* pk96, uint8_t* pk_inf) {
    NOT_ON_MULTI(ctx);
    if (!ctx || (n && (!sk32 || !pk96))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    k_keygen<<<grid_for(n, SIGN_THREADS), SIGN_THREADS, 0, ctx->stream>>>(n, sk32, ctx->gtab, pk96, pk_inf);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}
int schnorr_b200_keygen(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sk32, uint8_t* pk96, uint8_t* pk_inf) {
    MULTI_DISPATCH(ctx, multi_keygen(ctx, n, sk32, pk96, pk_inf));
    if (!ctx || (n && (!sk32 || !pk96))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_sk, *d_pk, *d_inf;
    if (int rc = stage_in(ctx, SL_D, sk32, n * 32, &d_sk)) return rc;
    if (int rc = ensure_scratch(ctx, SL_E, n * 96, &d_pk)) return rc;
    if (int rc = ensure_scratch(ctx, SL_I, n, &d_inf)) return rc;
    if (int rc = schnorr_b200_keygen_dev(ctx, n, (uint8_t*)d_sk, (uint8_t*)d_pk, (uint8_t*)d_inf)) return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(d_sk, 0, n * 32, ctx->stream));  // the staging arena is reused: do not keep secret keys in it
    CUDA_TRY(ctx, cudaMemcpyAsync(pk96, d_pk, n * 96, cudaMemcpyDeviceToHost, ctx->stream));
    if (pk_inf) CUDA_TRY(ctx, cudaMemcpyAsync(pk_inf, d_inf, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}
int schnorr_b200_sign_many_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sk32, const uint8_t* pk96,
                               const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                               const uint8_t* nonce32, uint8_t* sigs81) {
    NOT_ON_MULTI(ctx);
    if (!ctx || (n && (!sk32 || !pk96 || !msg_off || !nonce32 || !sigs81))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    k_sign<<<grid_for(n, SIGN_THREADS), SIGN_THREADS, 0, ctx->stream>>>(n, sk32, pk96, pk_inf, msgs, msg_off, nonce32,
                                                                        ctx->gtab, sigs81);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}
int schnorr_b200_sign_many(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sk32, const uint8_t* pk96,
                           const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* nonce32,
                           uint8_t* sigs81) {
    MULTI_DISPATCH(ctx, multi_sign_many(ctx, n, sk32, pk96, pk_inf, msgs, msg_off, nonce32, sigs81));
    if (!ctx || (n && (!sk32 || !pk96 || !msg_off || !nonce32 || !sigs81))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CHECK_MSG_OFF(ctx, n, msg_off);
    size_t mb = msg_off[n];
    if (mb && !msgs) return SCHNORR_B200_EARG;
    void *d_sk, *d_pk, *d_inf = nullptr, *d_m, *d_off, *d_nonce, *d_out;
    if (int rc = stage_in(ctx, SL_D, sk32, n * 32, &d_sk)) return rc;
    if (int rc = stage_in(ctx, SL_E, pk96, n * 96, &d_pk)) return rc;
    if (int rc = stage_in(ctx, SL_F, msgs, mb, &d_m)) return rc;
    if (int rc = stage_in(ctx, SL_G, msg_off, (n + 1) * 8, &d_off)) return rc;
    if (pk_inf)
        if (int rc = stage_in(ctx, SL_I, pk_inf, n, &d_inf)) return rc;
    if (int rc = stage_in(ctx, SL_J, nonce32, n * 32, &d_nonce)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n * 81, &d_out)) return rc;
    if (int rc = schnorr_b200_sign_many_dev(ctx, n, (uint8_t*)d_sk, (uint8_t*)d_pk, (uint8_t*)d_inf, (uint8_t*)d_m,
                                            (uint64_t*)d_off, (uint8_t*)d_nonce, (uint8_t*)d_out))
        return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(d_sk, 0, n * 32, ctx->stream));      // secret keys and nonces do not stay in the
    CUDA_TRY(ctx, cudaMemsetAsync(d_nonce, 0, n * 32, ctx->stream));   // reusable staging arena
    CUDA_TRY(ctx, cudaMemcpyAsync(sigs81, d_out, n * 81, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

// ---- f4: hierarchical deterministic derivation ---------------------------------------------------------------
int schnorr_b200_derive_master_keys(schnorr_b200_ctx* ctx, size_t n, const uint8_t* seeds32, uint8_t* xsk64, uint8_t* ok) {
    if (!ctx || (n && (!seeds32 || !xsk64 || !ok))) return SCHNORR_B200_EARG;
    MULTI_DISPATCH(ctx, schnorr_b200_derive_master_keys(ctx->shards[0], n, seeds32, xsk64, ok));
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_in, *d_out, *d_ok;
    if (int rc = stage_in(ctx, SL_D, seeds32, n * 32, &d_in)) return rc;
    if (int rc = ensure_scratch(ctx, SL_E, n * 64, &d_out)) return rc;
    if (int rc = ensure_scratch(ctx, SL_I, n, &d_ok)) return rc;
    k_derive_master<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, (uint8_t*)d_in, (uint8_t*)d_out, (uint8_t*)d_ok);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemsetAsync(d_in, 0, n * 32, ctx->stream));   // seeds are secrets
    CUDA_TRY(ctx, cudaMemcpyAsync(xsk64, d_out, n * 64, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ok, d_ok, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(d_out, 0, n * 64, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}
int schnorr_b200_derive_private_children(schnorr_b200_ctx* ctx, size_t n, const uint8_t* parent_xsk64, const uint32_t* indices,
                                         uint8_t* children_xsk64, uint8_t* ok) {
    if (!ctx || !parent_xsk64 || (n && (!indices || !children_xsk64 || !ok))) return SCHNORR_B200_EARG;
    MULTI_DISPATCH(ctx, schnorr_b200_derive_private_children(ctx->shards[0], n, parent_xsk64, indices, children_xsk64, ok));
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_par, *d_idx, *d_out, *d_ok;
    if (int rc = ensure_scratch(ctx, SL_D, 128, &d_par)) return rc;          // [0,64) parent, [64,128) its public key bytes
    CUDA_TRY(ctx, cudaMemcpyAsync(d_par, parent_xsk64, 64, cudaMemcpyHostToDevice, ctx->stream));
    if (int rc = stage_in(ctx, SL_F, indices, n * 4, &d_idx)) return rc;
    if (int rc = ensure_scratch(ctx, SL_E, n * 64, &d_out)) return rc;
    if (int rc = ensure_scratch(ctx, SL_I, n, &d_ok)) return rc;
    uint8_t* d_pk49 = (uint8_t*)d_par + 64;
    k_parent_public<<<1, 32, 0, ctx->stream>>>((uint8_t*)d_par, ctx->gtab, d_pk49);
    k_derive_private<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, (uint8_t*)d_par, d_pk49, (uint32_t*)d_idx, (uint8_t*)d_out,
                                                               (uint8_t*)d_ok);
    ctx->launches += 2;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(children_xsk64, d_out, n * 64, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ok, d_ok, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(d_par, 0, 128, ctx->stream));              // secrets do not stay in the arena
    CUDA_TRY(ctx, cudaMemsetAsync(d_out, 0, n * 64, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}
int schnorr_b200_derive_public_children(schnorr_b200_ctx* ctx, size_t n, const uint8_t* parent_xpk81, const uint32_t* indices,
                                        uint8_t* children_xpk81, uint8_t* ok) {
    if (!ctx || !parent_xpk81 || (n && (!indices || !children_xpk81 || !ok))) return SCHNORR_B200_EARG;
    MULTI_DISPATCH(ctx, schnorr_b200_derive_public_children(ctx->shards[0], n, parent_xpk81, indices, children_xpk81, ok));
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_par, *d_idx, *d_out, *d_ok;
    // parent record (81) | decompressed key (96) | identity flag (1) | decode flag (1), 16-byte aligned pieces
    if (int rc = ensure_scratch(ctx, SL_D, 96 + 96 + 16 + 16, &d_par)) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(d_par, parent_xpk81, 81, cudaMemcpyHostToDevice, ctx->stream));
    if (int rc = stage_in(ctx, SL_F, indices, n * 4, &d_idx)) return rc;
    if (int rc = ensure_scratch(ctx, SL_E, n * 81, &d_out)) return rc;
    if (int rc = ensure_scratch(ctx, SL_I, n, &d_ok)) return rc;
    uint8_t *d_pk96 = (uint8_t*)d_par + 96, *d_inf = d_pk96 + 96, *d_dec = d_inf + 16;
    k_decompress<<<1, 128, 0, ctx->stream>>>(1, (uint8_t*)d_par, d_pk96, d_inf, d_dec);   // ExtendedPublicKey::from_bytes (:295-311)
    k_derive_public<<<grid_for(n, SIGN_THREADS), SIGN_THREADS, 0, ctx->stream>>>(n, (uint8_t*)d_par, d_pk96, d_inf, (uint32_t*)d_idx,
                                                                                ctx->gtab, (uint8_t*)d_out, (uint8_t*)d_ok);
    ctx->launches += 2;
    CUDA_TRY(ctx, cudaGetLastError());
    uint8_t dec = 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(&dec, d_dec, 1, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(children_xpk81, d_out, n * 81, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ok, d_ok, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (!dec) {  // the parent key does not decode: no child exists
        ctx->err = "parent extended public key does not decode";
        return SCHNORR_B200_EARG;
    }
    return SCHNORR_B200_OK;
}

// ---- codecs ----------------------------------------------------------------------------------
int schnorr_b200_decompress(schnorr_b200_ctx* ctx, size_t n, const uint8_t* in49, uint8_t* pk96, uint8_t* pk_inf,
                            uint8_t* ok) {
    MULTI_DISPATCH(ctx, schnorr_b200_decompress(ctx->shards[0], n, in49, pk96, pk_inf, ok));
    if (!ctx || (n && (!in49 || !pk96 || !pk_inf || !ok))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_in, *d_pk, *d_inf, *d_ok;
    if (int rc = stage_in(ctx, SL_D, in49, n * 49, &d_in)) return rc;
    if (int rc = ensure_scratch(ctx, SL_E, n * 96, &d_pk)) return rc;
    if (int rc = ensure_scratch(ctx, SL_I, n, &d_inf)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n, &d_ok)) return rc;
    k_decompress<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, (uint8_t*)d_in, (uint8_t*)d_pk, (uint8_t*)d_inf,
                                                            (uint8_t*)d_ok);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(pk96, d_pk, n * 96, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(pk_inf, d_inf, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ok, d_ok, n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}
int schnorr_b200_compress(schnorr_b200_ctx* ctx, size_t n, const uint8_t* pk96, const uint8_t* pk_inf, uint8_t* out49) {
    MULTI_DISPATCH(ctx, schnorr_b200_compress(ctx->shards[0], n, pk96, pk_inf, out49));
    if (!ctx || (n && (!pk96 || !out49))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_pk, *d_inf = nullptr, *d_out;
    if (int rc = stage_in(ctx, SL_E, pk96, n * 96, &d_pk)) return rc;
    if (pk_inf)
        if (int rc = stage_in(ctx, SL_I, pk_inf, n, &d_inf)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n * 49, &d_out)) return rc;
    k_compress<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, (uint8_t*)d_pk, (uint8_t*)d_inf, (uint8_t*)d_out);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(out49, d_out, n * 49, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

// ---- test hook -------------------------------------------------------------------------------
int schnorr_b200_debug_field_ops(schnorr_b200_ctx* ctx, size_t n, const uint64_t* a6, const uint64_t* b6, uint64_t* out48) {
    MULTI_DISPATCH(ctx, schnorr_b200_debug_field_ops(ctx->shards[0], n, a6, b6, out48));
    if (!ctx || (n && (!a6 || !b6 || !out48))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_a, *d_b, *d_o;
    if (int rc = stage_in(ctx, SL_D, a6, n * 48, &d_a)) return rc;
    if (int rc = stage_in(ctx, SL_E, b6, n * 48, &d_b)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n * 48 * 8, &d_o)) return rc;
    k_debug_field<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, (uint64_t*)d_a, (uint64_t*)d_b, (uint64_t*)d_o);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(out48, d_o, n * 48 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

int schnorr_b200_debug_lazy_ops(schnorr_b200_ctx* ctx, size_t n, const uint64_t* a6, const uint64_t* b6, uint64_t* out48) {
    MULTI_DISPATCH(ctx, schnorr_b200_debug_lazy_ops(ctx->shards[0], n, a6, b6, out48));
    if (!ctx || (n && (!a6 || !b6 || !out48))) return SCHNORR_B200_EARG;
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void *d_a, *d_b, *d_o;
    if (int rc = stage_in(ctx, SL_D, a6, n * 48, &d_a)) return rc;
    if (int rc = stage_in(ctx, SL_E, b6, n * 48, &d_b)) return rc;
    if (int rc = ensure_scratch(ctx, SL_H, n * 48 * 8, &d_o)) return rc;
    k_debug_lazy<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, (uint64_t*)d_a, (uint64_t*)d_b, (uint64_t*)d_o);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(out48, d_o, n * 48 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

// ---- roofline calibration --------------------------------------------------------------------
int schnorr_b200_imad_peak(schnorr_b200_ctx* ctx, int iters, double* wide_mul_per_s, double* elapsed_ms) {
    MULTI_DISPATCH(ctx, schnorr_b200_imad_peak(ctx->shards[0], iters, wide_mul_per_s, elapsed_ms));
    if (!ctx || iters <= 0 || !wide_mul_per_s) return SCHNORR_B200_EARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void* sink;
    if (int rc = ensure_scratch(ctx, SL_H, 64, &sink)) return rc;
    int blocks = ctx->sm_count * 8;
    cudaEvent_t a, b;
    CUDA_TRY(ctx, cudaEventCreate(&a));
    CUDA_TRY(ctx, cudaEventCreate(&b));
    k_imad_peak<<<blocks, 256, 0, ctx->stream>>>(iters / 8 + 1, (uint64_t*)sink);  // warm-up
    CUDA_TRY(ctx, cudaEventRecord(a, ctx->stream));
    k_imad_peak<<<blocks, 256, 0, ctx->stream>>>(iters, (uint64_t*)sink);
    CUDA_TRY(ctx, cudaEventRecord(b, ctx->stream));
    ctx->launches += 2;
    CUDA_TRY(ctx, cudaEventSynchronize(b));
    float ms = 0;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    double total = (double)blocks * 256.0 * (double)iters * 8.0;
    *wide_mul_per_s = total / (ms * 1e-3);
    if (elapsed_ms) *elapsed_ms = ms;
    return SCHNORR_B200_OK;
}

}  // extern "C"
