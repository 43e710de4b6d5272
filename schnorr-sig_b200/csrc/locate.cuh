// Failed-batch localisation (SURVEY.md 8(f) f3) on one device or over the devices of a multi-device context.
//
// A range whose own random linear combination
//     sum_{i in range} s_i R_i - s_i h_i P_i  ==  (sum_{i in range} s_i e_i) G
// holds is clean (up to the 2^-255 soundness error of the batch itself).  The tree of ranges (locate_plan.h) is defined
// by n alone: each node is checked by its own partial MSM, and the leaves -- ranges of at most LOCATE_LEAF signatures,
// or everything that is left once the suspects stop shrinking -- go through k_batch_item_check.  One bad signature
// among 2^20 costs about two batch verifications; a batch riddled with bad signatures degrades to one per-item pass.
//
// On a multi-device context each device owns a contiguous block of the level-2 parts (locate_owned) and every node
// below them, and holds the records of its owned range only, staged once.  The whole batch is one partial per device,
// finished on the first (multi_batch_partials); every later level is checked by the owners of its parts, each in tree
// order, and the calling thread joins the verdicts before it cuts the next level.  So the tree, the cap and the flags
// are those of one device, byte for byte.  Included by schnorr_b200.cu after multi.cuh.
#pragma once
#include <memory>

#include "locate_plan.h"

// The records one device localises: its owned range [lo, hi) of the batch, on that device, with the offsets rebased to
// lo (a null `inf`: no identity keys), and its hi - lo flags.
struct locate_shard {
    size_t lo, hi;
    const uint8_t *sig, *pk, *inf, *msgs;
    const uint64_t* off;
    const uint8_t* rand;
    uint8_t* flags;
};

// the leaves of one device through k_batch_item_check (ranges relative to the records passed)
static int locate_items(schnorr_b200_ctx* ctx, const std::vector<locate_range>& ranges, const uint8_t* sigs81,
                        const uint8_t* pk96, const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                        const uint8_t* rand32, uint8_t* flags) {
    for (const locate_range& r : ranges) {
        size_t cn = r.hi - r.lo;
        if (cn == 0) continue;
        scratch_scope scope(ctx->scratch, ctx->stream);
        soa_batch soa;
        if (int rc = alloc_soa(ctx, cn, &soa)) return rc;
        k_ingest<<<grid_for(cn, INGEST_THREADS), INGEST_THREADS, 0, ctx->stream>>>(cn, sigs81 + 81 * r.lo, pk96 + 96 * r.lo,
                                                                                   pk_inf ? pk_inf + r.lo : nullptr, soa);
        k_batch_item_check<<<grid_for(cn, VERIFY_THREADS), VERIFY_THREADS, 0, ctx->stream>>>(soa, msgs, msg_off + r.lo,
                                                                                           rand32 + 32 * r.lo, ctx->gtab,
                                                                                           flags + r.lo);
        ctx->launches += 2;
        CUDA_TRY(ctx, cudaGetLastError());
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SCHNORR_B200_OK;
}

// parts[idx[0]], parts[idx[1]], ... (all inside s) on device context c, each through its own partial MSM and
// k_batch_finish; ok[idx[i]] = 1 where the part verifies
static int locate_check_parts(schnorr_b200_ctx* c, const locate_shard& s, const std::vector<locate_range>& parts,
                              const std::vector<size_t>& idx, uint8_t* ok) {
    if (idx.empty()) return SCHNORR_B200_OK;
    CUDA_TRY(c, cudaSetDevice(c->device));
    scratch_scope scope(c->scratch, c->stream);
    const size_t slot = RESULT_BYTES + 192 + 40;   // result | partial, per part
    uint8_t* base;
    if (int rc = stage_in(c, {{nullptr, slot * idx.size(), &base}})) return rc;
    for (size_t i = 0; i < idx.size(); i++) {
        const locate_range& r = parts[idx[i]];
        size_t o = r.lo - s.lo;
        uint8_t* res = base + i * slot;
        uint8_t* partial = res + RESULT_BYTES;
        if (int rc = batch_partial_impl(c, r.hi - r.lo, s.sig + 81 * o, s.pk + 96 * o, s.inf ? s.inf + o : nullptr, s.msgs,
                                        s.off + o, s.rand + 32 * o, partial))
            return rc;
        k_batch_finish<<<1, 32, 0, c->stream>>>(1, (const uint64_t*)partial, c->gtab, res, nullptr);
        c->launches += 1;
    }
    std::vector<uint8_t> host(idx.size() * slot);
    CUDA_TRY(c, cudaMemcpyAsync(host.data(), base, host.size(), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < idx.size(); i++) ok[idx[i]] = host[i * slot] == VERDICT_OK;
    return SCHNORR_B200_OK;
}

// The bisection of n items, device k of ctx holding sh[k] (one entry: the context's own device).  Each device zeroes
// and writes its flags in place, and copies them to host_flags + lo when host_flags is not null.
static int locate_run(schnorr_b200_ctx* ctx, size_t n, const std::vector<locate_shard>& sh, uint8_t* host_flags) {
    std::vector<shard_slice> sl;
    std::vector<locate_range> owned;
    for (const locate_shard& s : sh) {
        sl.push_back({s.lo, s.hi});
        owned.push_back({s.lo, s.hi});
    }
    auto check = [&](const std::vector<locate_range>& parts, uint8_t* ok) -> int {
        if (locate_owner(owned, parts[0]) < 0) {   // the whole batch over several devices
            int verdict = 0;
            int rc = multi_batch_partials(ctx, sl, &verdict, nullptr, nullptr, [&](int k, shard_slice, uint8_t* partial) {
                const locate_shard& s = sh[k];
                return batch_partial_impl(ctx->shards[k], s.hi - s.lo, s.sig, s.pk, s.inf, s.msgs, s.off, s.rand, partial);
            });
            ok[0] = verdict == VERDICT_OK;
            return rc;
        }
        std::vector<std::vector<size_t>> mine(sh.size());
        for (size_t j = 0; j < parts.size(); j++) mine[locate_owner(owned, parts[j])].push_back(j);
        return multi_run(ctx, sl, [&](int k, shard_slice) {
            return locate_check_parts(device_ctx(ctx, k), sh[k], parts, mine[k], ok);
        });
    };
    auto items = [&](const std::vector<locate_range>& leaves) -> int {
        std::vector<std::vector<locate_range>> mine(sh.size());
        for (const locate_range& r : leaves) {
            int k = locate_owner(owned, r);
            mine[k].push_back({r.lo - sh[k].lo, r.hi - sh[k].lo});
        }
        return multi_run(ctx, sl, [&](int k, shard_slice) -> int {
            schnorr_b200_ctx* c = device_ctx(ctx, k);
            const locate_shard& s = sh[k];
            CUDA_TRY(c, cudaSetDevice(c->device));
            CUDA_TRY(c, cudaMemsetAsync(s.flags, 0, s.hi - s.lo, c->stream));
            if (int rc = locate_items(c, mine[k], s.sig, s.pk, s.inf, s.msgs, s.off, s.rand, s.flags)) return rc;
            if (host_flags) {
                CUDA_TRY(c, cudaMemcpyAsync(host_flags + s.lo, s.flags, s.hi - s.lo, cudaMemcpyDeviceToHost, c->stream));
                CUDA_TRY(c, cudaStreamSynchronize(c->stream));
            }
            return SCHNORR_B200_OK;
        });
    };
    return locate_bisect(n, check, items);
}

// The host forms of localisation (argument pointers checked by the caller).  Each device's owned range is staged there
// once, in a scope of its arena held for the whole call: the message bytes with rebased offsets, the randomisers (or
// the seed, generated there from rs.from(lo)), a flag region, and the form's records, which records(c, k, lo, hi, &shard)
// builds on device k (context c) and sets in the shard.  Then locate_run, the flags copied back and counted.
template <typename F>
static int locate_invalid_host(schnorr_b200_ctx* ctx, size_t n, const uint8_t* msgs, const uint64_t* msg_off,
                               const rand_source& rs, uint8_t* flags, uint64_t* n_bad, F records) {
    if (n_bad) *n_bad = 0;
    if (n == 0) return SCHNORR_B200_OK;
    CHECK_MSG_OFF(ctx, n, msg_off);
    if (msg_off[n] && !msgs) return SCHNORR_B200_EARG;
    std::vector<locate_range> owned =
        locate_owned(n, ctx->shards.empty() ? 1 : locate_devices(ctx->shards.size(), n, MULTI_MIN_PER_SHARD));
    std::vector<shard_slice> sl;
    std::vector<locate_shard> sh(owned.size());
    std::vector<std::unique_ptr<scratch_scope>> scopes;   // the staged records, until the call returns
    for (size_t k = 0; k < owned.size(); k++) {
        schnorr_b200_ctx* c = device_ctx(ctx, k);
        CUDA_TRY(ctx, cudaSetDevice(c->device));
        scopes.emplace_back(new scratch_scope(c->scratch, c->stream));
        sl.push_back({owned[k].lo, owned[k].hi});
    }
    int rc = multi_run(ctx, sl, [&](int k, shard_slice s) -> int {
        schnorr_b200_ctx* c = device_ctx(ctx, k);
        CUDA_TRY(c, cudaSetDevice(c->device));
        size_t len = s.hi - s.lo;
        std::vector<uint64_t> off = rebase_offsets(msg_off, s.lo, s.hi);
        rand_source r = rs.from(s.lo);
        uint8_t *d_m, *d_off, *d_rand, *d_seed, *d_flags;
        if (int e = stage_in(c, {{msgs ? msgs + msg_off[s.lo] : nullptr, off[len], &d_m}, {off.data(), (len + 1) * 8, &d_off},
                                 r.rand_region(len, &d_rand), r.seed_region(&d_seed), {nullptr, len, &d_flags}}))
            return e;
        if (int e = rand_generate(c, len, r, d_seed, d_rand)) return e;
        sh[k] = {s.lo, s.hi, nullptr, nullptr, nullptr, d_m, (const uint64_t*)d_off, d_rand, d_flags};
        if (int e = records(c, (size_t)k, s.lo, s.hi, &sh[k])) return e;
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));   // `off` is read by an asynchronous copy
        return SCHNORR_B200_OK;
    });
    if (rc) return rc;
    if (int e = locate_run(ctx, n, sh, flags)) return e;
    if (n_bad)
        for (size_t i = 0; i < n; i++) *n_bad += flags[i] != 0;
    return SCHNORR_B200_OK;
}

// signatures and keys as the caller gives them
static int locate_invalid_plain(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const rand_source& rs,
                                uint8_t* flags, uint64_t* n_bad) {
    return locate_invalid_host(ctx, n, msgs, msg_off, rs, flags, n_bad,
                               [&](schnorr_b200_ctx* c, size_t, size_t lo, size_t hi, locate_shard* s) {
        size_t len = hi - lo;
        uint8_t *d_sig, *d_pk, *d_inf;
        if (int rc = stage_in(c, {{sigs81 + 81 * lo, len * 81, &d_sig}, {pk96 + 96 * lo, len * 96, &d_pk},
                                  {pk_inf ? pk_inf + lo : nullptr, len, &d_inf}}))
            return rc;
        s->sig = d_sig;
        s->pk = d_pk;
        s->inf = pk_inf ? d_inf : nullptr;
        return 0;
    });
}

extern "C" {

int schnorr_b200_locate_invalid_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                    const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                                    const uint8_t* rand32, uint8_t* flags) {
    if (!ctx || (n && (!sigs81 || !pk96 || !msg_off || !rand32 || !flags))) return SCHNORR_B200_EARG;
    NOT_ON_MULTI(ctx);
    if (n == 0) return SCHNORR_B200_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return locate_run(ctx, n, {{0, n, sigs81, pk96, pk_inf, msgs, msg_off, rand32, flags}}, nullptr);
}

int schnorr_b200_locate_invalid(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32,
                                uint8_t* flags, uint64_t* n_bad) {
    if (!ctx || (n && (!sigs81 || !pk96 || !msg_off || !rand32 || !flags))) return SCHNORR_B200_EARG;
    return locate_invalid_plain(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rand_from_host(rand32), flags, n_bad);
}

int schnorr_b200_locate_invalid_seeded(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                       const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                                       const uint8_t* seed32, uint8_t* flags, uint64_t* n_bad) {
    if (!ctx || !seed32 || (n && (!sigs81 || !pk96 || !msg_off || !flags))) return SCHNORR_B200_EARG;
    return locate_invalid_plain(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rand_from_seed(seed32), flags, n_bad);
}

}  // extern "C"
