// Multi-device contexts behind the C ABI (schnorr_b200_create_multi, SURVEY.md §8(b)/(e)).
//
// A multi-device context owns one ordinary single-device context ("shard") per entry of the device list: its own
// stream, scratch arena and fixed-base table on that GPU.  The HOST entry points cut the call into contiguous slices,
// one per shard, and run the slices concurrently -- one host thread per device drives the existing single-device
// pipeline (copy / ingest / verify overlapped per device), so there is no data-path exchange at all for independent
// verification (signatures are independent, `src/signature.rs:181-205`).  Batch verification (`src/batch.rs:31-130`)
// has exactly one exchange step: every shard reduces its slice to a 192-byte partial (Jacobian point + partial
// scalar), the partials travel to the first device with cudaMemcpyPeerAsync (NVLink / NVSwitch between B200s) and
// k_batch_finish adds them there.  Randomisers are indexed by signature, so the result does not depend on the
// sharding.  The same device may be listed more than once (used by the tests to exercise the sharded code paths on a
// single-GPU box).  Included by schnorr_b200.cu (single translation unit).
#pragma once
#include <thread>

// calls smaller than this stay on the first shard: below it the per-call latency dominates and a second device
// cannot shorten it
static constexpr size_t MULTI_MIN_PER_SHARD = 4096;

struct shard_slice {
    size_t lo, hi;
};
static std::vector<shard_slice> multi_slices(const schnorr_b200_ctx* ctx, size_t n) {
    size_t g = ctx->shards.size();
    if (n < MULTI_MIN_PER_SHARD * 2) g = 1;
    else if (n / g < MULTI_MIN_PER_SHARD) g = n / MULTI_MIN_PER_SHARD;
    std::vector<shard_slice> out;
    size_t per = (n + g - 1) / g;
    per = (per + 127) / 128 * 128;  // whole 128-signature thread blocks per shard
    for (size_t lo = 0; lo < n; lo += per) out.push_back({lo, lo + per < n ? lo + per : n});
    if (out.empty()) out.push_back({0, 0});
    return out;
}
// offsets of a slice rebased to 0 (the single-device entry points expect a table that starts at 0)
static std::vector<uint64_t> rebase_offsets(const uint64_t* msg_off, size_t lo, size_t hi) {
    std::vector<uint64_t> o(hi - lo + 1);
    uint64_t base = msg_off[lo];
    for (size_t i = lo; i <= hi; i++) o[i - lo] = msg_off[i] - base;
    return o;
}
// runs fn(shard index, slice) on one host thread per slice; returns the first non-zero code and copies that shard's
// error text into the parent context
template <typename F>
static int multi_run(schnorr_b200_ctx* ctx, const std::vector<shard_slice>& sl, F fn) {
    std::vector<int> rc(sl.size(), 0);
    if (sl.size() == 1) {
        rc[0] = fn(0, sl[0]);
    } else {
        std::vector<std::thread> th;
        th.reserve(sl.size());
        for (size_t k = 0; k < sl.size(); k++) th.emplace_back([&, k] { rc[k] = fn((int)k, sl[k]); });
        for (auto& t : th) t.join();
    }
    for (size_t k = 0; k < sl.size(); k++)
        if (rc[k] != 0) {
            ctx->err = "device " + std::to_string(ctx->shards[k]->device) + ": " + ctx->shards[k]->err;
            return rc[k];
        }
    return SCHNORR_B200_OK;
}

static int multi_verify_many(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96, const uint8_t* pk_inf,
                             const uint8_t* msgs, const uint64_t* msg_off, uint8_t* verdicts) {
    auto sl = multi_slices(ctx, n);
    // the hot entry point: every shard gets its slice of the caller's offset table as it is (no rebasing pass) and
    // validates it chunk by chunk inside its own pipeline, on its own host thread; here only the slice boundaries are
    // checked, which bounds every shard's view of the blob by msg_off[n]
    bool ok = n == 0 || msg_off[0] == 0;
    for (const shard_slice& s : sl) ok = ok && msg_off[s.lo] <= msg_off[s.hi] && msg_off[s.hi] <= msg_off[n];
    if (!ok) {
        ctx->err = "message offsets must start at 0 and be non-decreasing";
        return SCHNORR_B200_EARG;
    }
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        return verify_many_host(ctx->shards[k], s.hi - s.lo, sigs81 + 81 * s.lo, pk96 + 96 * s.lo,
                                pk_inf ? pk_inf + s.lo : nullptr, msgs, msg_off + s.lo, verdicts + s.lo, true);
    });
}
static int multi_verify_keyed_many(schnorr_b200_ctx* ctx, size_t n, const uint8_t* keyed130, const uint8_t* msgs,
                                   const uint64_t* msg_off, uint8_t* verdicts) {
    CHECK_MSG_OFF(ctx, n, msg_off);
    auto sl = multi_slices(ctx, n);
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        auto off = rebase_offsets(msg_off, s.lo, s.hi);
        return schnorr_b200_verify_keyed_many(ctx->shards[k], s.hi - s.lo, keyed130 + 130 * s.lo,
                                              msgs ? msgs + msg_off[s.lo] : nullptr, off.data(), verdicts + s.lo);
    });
}
static int multi_hash_messages(schnorr_b200_ctx* ctx, size_t n, const uint8_t* rx48, const uint8_t* pk96, const uint8_t* msgs,
                               const uint64_t* msg_off, uint8_t* digests) {
    CHECK_MSG_OFF(ctx, n, msg_off);
    auto sl = multi_slices(ctx, n);
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        auto off = rebase_offsets(msg_off, s.lo, s.hi);
        return schnorr_b200_hash_messages(ctx->shards[k], s.hi - s.lo, rx48 + 48 * s.lo, pk96 + 96 * s.lo,
                                          msgs ? msgs + msg_off[s.lo] : nullptr, off.data(), digests + 32 * s.lo);
    });
}
static int multi_keygen(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sk32, uint8_t* pk96, uint8_t* pk_inf) {
    auto sl = multi_slices(ctx, n);
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        return schnorr_b200_keygen(ctx->shards[k], s.hi - s.lo, sk32 + 32 * s.lo, pk96 + 96 * s.lo,
                                   pk_inf ? pk_inf + s.lo : nullptr);
    });
}
static int multi_sign_many(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sk32, const uint8_t* pk96, const uint8_t* pk_inf,
                           const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* nonce32, uint8_t* sigs81) {
    CHECK_MSG_OFF(ctx, n, msg_off);
    auto sl = multi_slices(ctx, n);
    return multi_run(ctx, sl, [&](int k, shard_slice s) {
        auto off = rebase_offsets(msg_off, s.lo, s.hi);
        return schnorr_b200_sign_many(ctx->shards[k], s.hi - s.lo, sk32 + 32 * s.lo, pk96 + 96 * s.lo,
                                      pk_inf ? pk_inf + s.lo : nullptr, msgs ? msgs + msg_off[s.lo] : nullptr, off.data(),
                                      nonce32 + 32 * s.lo, sigs81 + 81 * s.lo);
    });
}

// verify_batch (and its registered-key-set form) over all devices: per-shard partials from `partial_fn`, one peer copy
// each, finish on the first device.  A batch always uses every shard slice it is given (an empty slice contributes the
// identity).
template <typename F>
static int multi_verify_batch(schnorr_b200_ctx* ctx, size_t n, const uint64_t* msg_off, int* verdict, uint8_t* lhs97,
                              uint8_t* rhs97, F partial_fn) {
    if (n) CHECK_MSG_OFF(ctx, n, msg_off);
    auto sl = multi_slices(ctx, n);
    size_t g = sl.size();
    schnorr_b200_ctx* root = ctx->shards[0];
    CUDA_TRY(root, cudaSetDevice(root->device));
    // root buffer: [64 B flags of batch_partial_impl | result | g partials]
    void* d_res;
    if (int rc = ensure_scratch(root, SL_L, 64 + RESULT_BYTES + 192 * (g + 1), &d_res)) {
        ctx->err = root->err;
        return rc;
    }
    uint8_t* res = (uint8_t*)d_res + 64;
    uint8_t* gathered = res + RESULT_BYTES;  // g x 192 B on the root device
    int rc = multi_run(ctx, sl, [&](int k, shard_slice s) {
        schnorr_b200_ctx* sh = ctx->shards[k];
        if (cudaSetDevice(sh->device) != cudaSuccess) return (int)SCHNORR_B200_ECUDA;
        uint8_t* partial;
        if (k == 0) {
            partial = gathered;  // the root writes its partial in place
        } else {
            void* d_loc;
            if (int r2 = ensure_scratch(sh, SL_L, 64 + RESULT_BYTES + 192, &d_loc)) return r2;
            partial = (uint8_t*)d_loc + 64 + RESULT_BYTES;
        }
        size_t cn = s.hi - s.lo;
        int r;
        if (cn == 0) {
            r = batch_partial_empty(sh, partial);
        } else {
            auto off = rebase_offsets(msg_off, s.lo, s.hi);
            r = partial_fn(k, s, off.data(), partial);
            // `off` must outlive the asynchronous copy that reads it: synchronise before it goes out of scope
            if (r == 0 && cudaStreamSynchronize(sh->stream) != cudaSuccess) r = SCHNORR_B200_ECUDA;
        }
        if (r) return r;
        if (k != 0) {  // the ONE exchange step of the batch path: 192 bytes over NVLink to the root device
            if (cudaMemcpyPeerAsync(gathered + 192 * (size_t)k, root->device, partial, sh->device, 192, sh->stream) != cudaSuccess) {
                sh->err = "cudaMemcpyPeerAsync of the batch partial failed";
                return (int)SCHNORR_B200_ECUDA;
            }
        }
        if (cudaStreamSynchronize(sh->stream) != cudaSuccess) {
            sh->err = "stream synchronisation failed";
            return (int)SCHNORR_B200_ECUDA;
        }
        return (int)SCHNORR_B200_OK;
    });
    if (rc) return rc;
    ctx->last_batch_points = 0;
    for (size_t k = 0; k < g; k++)
        if (sl[k].hi > sl[k].lo) ctx->last_batch_points += ctx->shards[k]->last_batch_points;
    CUDA_TRY(root, cudaSetDevice(root->device));
    if (int r = schnorr_b200_batch_finish_dev(root, g, gathered, res)) {
        ctx->err = root->err;
        return r;
    }
    int r = read_result(root, res, verdict, lhs97, rhs97);
    if (r) ctx->err = root->err;
    return r;
}
