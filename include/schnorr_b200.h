/* schnorr_b200 -- C ABI of the B200-native Schnorr verification engine (Cheetah curve / Rescue hash).
 *
 * This is the drop-in boundary for the hot path of toposware/schnorr-sig.  The reference has no FFI
 * (`#![deny(unsafe_code)]`, src/lib.rs:152); the entry points below are what a `schnorr-sig-sys`
 * layer under the reference's public API would bind (INTEGRATION.md shows the Rust side).  Each
 * function cites the reference interface it replaces.
 *
 * Conventions
 *  - plain pointers and sizes, no CUDA/torch types; `void *stream` is a cudaStream_t.
 *  - record layouts are the reference's own byte encodings:
 *      signature  81 B  = CompressedPoint (48 B little-endian limbs c0..c5 of R.x, 1 flag byte:
 *                         bit 7 infinity, bit 6 y-sign) || Scalar e (32 B LE)    src/signature.rs:208-214
 *      public key 96 B  = affine x (48 B) || y (48 B), the in-memory `PublicKey(AffinePoint)`
 *                         (src/public.rs:24) + one byte per key: 1 = identity
 *      scalar     32 B  little-endian                                            src/constants.rs:12
 *      messages   one byte blob + uint64 offsets[n+1]  (the reference's `&[&[u8]]`)
 *  - verdict bytes: 0 = Ok(()), 1 = Err(InvalidPublicKey), 2 = Err(InvalidSignature)
 *    (src/error.rs:13-18), 3 = malformed input on which the reference panics or which its types
 *    cannot represent (non-canonical limb / scalar >= q; src/signature.rs:186, src/batch.rs:67,104).
 *  - return value: 0 on success, negative SCHNORR_B200_E* on argument / CUDA failure.  An invalid
 *    signature is data (a verdict), never an error code.
 *  - `*_dev` variants take DEVICE pointers for every buffer, enqueue on the context stream and do
 *    not synchronise; the host variants copy in, run the same kernels, copy out and synchronise.
 *  - a context is single-owner: one in-flight call per context; create several for concurrency.  The same holds for
 *    a registered key set: an update (keyset_append / _replace / _remove) synchronises every device of the context,
 *    so *_dev calls enqueued before it see the old set and calls made after it the new one.
 *  - there is NO CPU fallback: without a CUDA device `schnorr_b200_create` fails.
 */
#ifndef SCHNORR_B200_H
#define SCHNORR_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCHNORR_B200_OK 0
#define SCHNORR_B200_EARG (-1)    /* bad argument */
#define SCHNORR_B200_ECUDA (-2)   /* CUDA runtime failure, see schnorr_b200_last_error */
#define SCHNORR_B200_ENODEV (-3)  /* no usable CUDA device */

#define SCHNORR_B200_SIGNATURE_BYTES 81   /* SIGNATURE_LENGTH   src/constants.rs:30 */
#define SCHNORR_B200_POINT_BYTES 96       /* affine x||y */
#define SCHNORR_B200_COMPRESSED_BYTES 49  /* PUBLIC_KEY_LENGTH  src/constants.rs:24 */
#define SCHNORR_B200_SCALAR_BYTES 32      /* SCALAR_LENGTH      src/constants.rs:12 */
#define SCHNORR_B200_DIGEST_BYTES 32
#define SCHNORR_B200_PARTIAL_BYTES 192    /* Jacobian point 144 B || partial scalar 32 B || flags 16 B */

typedef struct schnorr_b200_ctx schnorr_b200_ctx;

/* Value-level provenance of the curve / hash constants compiled into the library (include/cheetah_params.h).
 * 0 = NOT pinned to the upstream `cheetah` / `hash` crates: the reference's tests hold no generator, digest or signature
 * known answers and its dependencies are un-vendored git crates, so the generator is a placeholder and the Rescue
 * instance is recalled / spec-derived; every result is bit-exact against the restated oracle (oracle/), and keys /
 * signatures interoperate with the real crate only after rust/dump_params has been run on a machine with cargo and the
 * header regenerated (INTEGRATION.md 5).  schnorr_b200_create prints this once per process while it is 0. */
int schnorr_b200_params_pinned(void);
const char *schnorr_b200_params_provenance(void);

/* Creates a context on CUDA device `device`: stream, scratch arena and the fixed-base table of G
 * (the reference's `cheetah::BASEPOINT_TABLE`, src/signature.rs:19) built on the device. */
int schnorr_b200_create(int device, schnorr_b200_ctx **out);
/* Multi-device context (SURVEY.md 8(b)/(e)): one stream, scratch arena and fixed-base table per listed CUDA device.
 * The HOST entry points (verify_many, verify_keyed_many, hash_messages, verify_batch, keygen, sign_many) then shard
 * every call over the devices in contiguous slices -- independent verification without any exchange, batch
 * verification with ONE 192-byte peer copy per device (partial MSM point + partial scalar) to the first device, where
 * the batch is finished.  This is what `verify_batch(&[Signature], &[PublicKey], &[&[u8]], rng)` (src/batch.rs:31-36)
 * and a loop over `Signature::verify` bind to on an 8-GPU box.  The *_dev entry points and set_stream need a
 * single-device context (device buffers live on one GPU) and return SCHNORR_B200_EARG here.  A device may be listed
 * more than once (independent contexts on the same GPU).  n_devices == 1 is schnorr_b200_create. */
int schnorr_b200_create_multi(const int *devices, int n_devices, schnorr_b200_ctx **out);
/* number of device contexts behind `ctx` (1 for schnorr_b200_create) */
int schnorr_b200_device_count(const schnorr_b200_ctx *ctx);
void schnorr_b200_destroy(schnorr_b200_ctx *ctx);
const char *schnorr_b200_last_error(const schnorr_b200_ctx *ctx);
/* Use an external stream (e.g. the caller's current stream) for all subsequent work. NULL = own stream. */
int schnorr_b200_set_stream(schnorr_b200_ctx *ctx, void *stream);
int schnorr_b200_synchronize(schnorr_b200_ctx *ctx);
/* Number of kernel launches issued by this context since creation (bench `gpu_launches`). */
uint64_t schnorr_b200_launch_count(const schnorr_b200_ctx *ctx);
/* Device time (CUDA events on the context stream) of the dominant kernel of the last *_dev call:
 * k_verify (verify_many), k_hash (hash_messages), k_msm_segment_sum (batch).  Synchronises on it. */
int schnorr_b200_last_kernel_ms(schnorr_b200_ctx *ctx, float *ms);
/* Single verification runs a fast path (inversion-free affine formulas, denominators kept in Fp) and re-runs the items
 * that hit one of its exceptional cases (identity / small-order keys, colliding partial sums) through the exact Jacobian kernel.
 * exact_only = 1 sends everything through the exact kernel (A/B measurements, tests).
 * last_exact_count: how many items of the last verify_many* call took the exact kernel (synchronises). */
int schnorr_b200_set_exact_only(schnorr_b200_ctx *ctx, int exact_only);
int schnorr_b200_last_exact_count(schnorr_b200_ctx *ctx, uint64_t *count);
/* Calls of at most `max_signatures` signatures (per pipeline chunk) run the warp-cooperative kernel (one signature per
 * six lanes: ~4x lower latency, 6x more parallelism per signature, ~1.5x the work); larger calls the one-signature-per-
 * thread kernel.  0 disables it, SIZE_MAX forces it (tests).  Default 10240 (measured crossover ~12 k). */
int schnorr_b200_set_dist_threshold(schnorr_b200_ctx *ctx, size_t max_signatures);
/* Calls of at most `max_signatures` signatures (per pipeline chunk) run one thread BLOCK per signature: the doubling
 * chain, the challenge hash, e*G and then the sixteen bucket accumulations of one verification proceed side by side on
 * the block's warps (lowest latency for the reference's own Criterion case, a single Signature::verify,
 * benches/schnorr.rs:22-66).  0 disables it.  Default 512 (measured: 0.50-0.65 ms for 1..512 signatures against
 * 0.98-1.08 ms on six lanes; beyond ~1000 blocks the six-lane kernel is faster).  The same threshold selects the
 * block-per-signature form of calls against a registered key set (verify_registered_many, the host form of
 * verify_keyed_registered_many): the challenge hash, e*G and a tree of the key's 32 table terms on the block's warps,
 * with no doubling chain; larger registered calls run one signature per thread.  SIZE_MAX forces the block form, 0 the
 * per-thread one (tests). */
int schnorr_b200_set_one_threshold(schnorr_b200_ctx *ctx, size_t max_signatures);
/* Batches of at most `max_signatures` compute their challenges with one signature per six lanes ahead of the (then
 * hash-free) prepare kernel; larger ones hash one signature per thread.  Default 2^18 (measured crossover). */
int schnorr_b200_set_batch_dist_threshold(schnorr_b200_ctx *ctx, size_t max_signatures);
/* Batches (per device) of at most `max_signatures` signatures run one thread block per signature: block i evaluates its
 * own term s_i R_i - s_i h_i P_i of the batch equation (src/batch.rs:102-123) with the two doubling chains, the challenge
 * hash and the bucket accumulations side by side on its warps, and one more block adds the terms -- the latency form for
 * the reference's Criterion cases of 4 ... 128 signatures (benches/schnorr.rs:67-96).  Larger batches take the Pippenger
 * pipeline.  0 disables it.  Default 256. */
int schnorr_b200_set_batch_small_threshold(schnorr_b200_ctx *ctx, size_t max_signatures);
/* Test hook: force the Pippenger window width (4..16, 0 = planner's choice) and the segment length of the bucket
 * accumulation (>= 8, 0 = automatic) of the batch path, to exercise the skewed-bucket code paths. */
int schnorr_b200_set_msm_geometry(schnorr_b200_ctx *ctx, int window_bits, unsigned segment_len);
/* Pippenger geometry of the last batch call on this context (window width c, number of windows K, entries per
 * accumulation segment): the unit count of the batch roofline is computed from the plan actually used (cost_model.py). */
int schnorr_b200_last_batch_plan(const schnorr_b200_ctx *ctx, int *window_bits, int *windows, unsigned *segment_len);

/* hash_message(&Fp6, &PublicKey, &[u8]) -> [u8; 32]            src/signature.rs:274-306
 * rx48: n x 48 B (R.x limbs), pk96: n x 96 B, digests: n x 32 B.  */
int schnorr_b200_hash_messages(schnorr_b200_ctx *ctx, size_t n, const uint8_t *rx48, const uint8_t *pk96,
                               const uint8_t *msgs, const uint64_t *msg_off, uint8_t *digests);
int schnorr_b200_hash_messages_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *rx48, const uint8_t *pk96,
                                   const uint8_t *msgs, const uint64_t *msg_off, uint8_t *digests);

/* Signature::verify(self, message, &PublicKey) for n independent triples  src/signature.rs:181-205
 * (also PublicKey::verify_signature :170-176, KeyPair::verify_signature :159-165,
 *  KeyedSignature::verify :232-234).  pk_inf may be NULL (no identity keys). */
int schnorr_b200_verify_many(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                             const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                             uint8_t *verdicts);
int schnorr_b200_verify_many_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                 const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                 uint8_t *verdicts);

/* Registered key sets: Signature::verify (src/signature.rs:181-205, also PublicKey::verify_signature :170-176) for many
 * signatures under a small, recurring set of public keys.  Registration does once per key what every verification
 * otherwise repeats: the subgroup check [q]P == O and the doubling chain of h*P, kept as a table of 32 x 129 affine
 * multiples of P (396 KB per key, on every device of the context).  A verification is then the challenge hash and about
 * 52 table additions.
 * Keys are public data: the tables are indexed by challenge digits and are not constant-time (DESIGN.md §7).
 *
 * keyset_create registers n_keys public keys (pk96 / pk_inf as in verify_many; pk_inf may be NULL) on every device of
 * ctx.  status (optional, n_keys bytes): 0 = in the prime-order subgroup (the identity included), 1 = not (verify gives
 * InvalidPublicKey), 3 = non-canonical limb (verify gives 3).  EARG for n_keys == 0 or n_keys >= 2^32.  Duplicate keys
 * are allowed.  A set belongs to the context it was created on and must be destroyed before it. */
typedef struct schnorr_b200_keyset schnorr_b200_keyset;
int schnorr_b200_keyset_create(schnorr_b200_ctx *ctx, size_t n_keys, const uint8_t *pk96, const uint8_t *pk_inf,
                               uint8_t *status, schnorr_b200_keyset **out);
void schnorr_b200_keyset_destroy(schnorr_b200_keyset *ks);
/* Signature::verify for n (signature, key, message) triples, key = key_idx[i] into the set: verdicts[i] is, byte for
 * byte, what verify_many returns for sigs81[i], message i and that key.  An index outside the set gives verdict 3
 * (indexing past the end of a slice panics in the reference).  A set from another context returns EARG.
 * last_exact_count, last_kernel_ms and set_exact_only apply as for verify_many.  Calls (per device) of at most
 * set_one_threshold signatures run one thread block per signature from the key's table, the latency form for a node
 * that sees one vote or certificate at a time; larger calls one thread per signature.  The host form shards a
 * multi-device context in contiguous slices, and each device picks its form by the size of its own slice; the _dev form
 * (device buffers, no synchronisation) needs a single-device context and a non-NULL msgs even when every message is
 * empty. */
int schnorr_b200_verify_registered_many(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                        const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                        const uint64_t *msg_off, uint8_t *verdicts);
int schnorr_b200_verify_registered_many_dev(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                            const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                            const uint64_t *msg_off, uint8_t *verdicts);

/* Updating a registered key set in place (a validator or committee set: a key joins, rotates, leaves).  After every
 * update the set is exactly, byte for byte on every device, what keyset_create builds from the current list of slot
 * records: records, identity flags, status bytes, tables (zeros for slots without one) and the lookup table (smallest
 * findable index per encoding), and whether batches may sum the key side per key.
 *  - keyset_append registers n keys in the next slots (indices n_keys ... n_keys + n - 1); EARG when the set would
 *    reach 2^32 slots.  Records, status bytes and tables grow geometrically, so repeated appends copy the tables only
 *    O(log n) times; while a buffer grows, the device holds the old and the new one (old plus new slots' tables).
 *  - keyset_replace registers pk96[j] / pk_inf[j] in slot key_idx[j]; the slot keeps its index.  EARG for an index at
 *    or beyond n_keys and for an index repeated in one call.
 *  - keyset_remove writes the record of an index outside the set (96 bytes of 0xFF, identity flag 0) into the listed
 *    slots: status 3, no table, not findable, so a removed index behaves like an index outside the set everywhere
 *    (verdict 3, a malformed batch, flag 3 in locate_invalid_registered, a miss in keyset_lookup).  Repeated and
 *    already removed indices are accepted.  Removed slots keep their index and memory and still count in n_keys
 *    (and in the batch rule of set_registered_batch_threshold); keyset_replace reuses them.
 * pk_inf may be NULL; status (optional, n bytes) as in keyset_create; n == 0 returns OK.  Argument checks and every
 * allocation come before the set is written: an update that returns EARG, or fails to allocate, leaves it unchanged.
 * An update synchronises every device of the context before it returns: *_dev calls enqueued before it see the old
 * set, calls made after it the new one, and grown buffers are freed only after the work that may read them.  Registrations
 * of up to set_keyset_block_threshold keys run one thread block per key (lowest latency), larger ones one thread per key.
 * (No reference counterpart: the reference verifies each signature from scratch, src/signature.rs:181-205.) */
int schnorr_b200_keyset_append(schnorr_b200_ctx *ctx, schnorr_b200_keyset *ks, size_t n, const uint8_t *pk96,
                               const uint8_t *pk_inf, uint8_t *status);
int schnorr_b200_keyset_replace(schnorr_b200_ctx *ctx, schnorr_b200_keyset *ks, size_t n, const uint32_t *key_idx,
                                const uint8_t *pk96, const uint8_t *pk_inf, uint8_t *status);
int schnorr_b200_keyset_remove(schnorr_b200_ctx *ctx, schnorr_b200_keyset *ks, size_t n, const uint32_t *key_idx);
/* Registrations (keyset_create, _append, _replace) of at most `max_keys` keys run one thread block per key, larger ones
 * one thread per key; the results are identical.  0 = never, SIZE_MAX = always (tests).  Default 512 (measured: one
 * key 0.64 against 3.5 ms per replace call, 512 keys 10.3 against 12.8 ms, 4096 keys 81.5 against 79.5 ms). */
int schnorr_b200_set_keyset_block_threshold(schnorr_b200_ctx *ctx, size_t max_keys);
/* Test hook (no reference counterpart): copies to the host, from device `device_index` of the context (0 for a
 * single-device context), slots first ... first + count - 1 of the set -- pk96 (count x 96 B), pk_inf (count),
 * status (count), tables (count x 32 x 129 x 12 u64) -- and the lookup table: lut64 (room for n_keys entries of 64 B:
 * 6 x-limbs, flag u32, index u32, pad u64) and *n_lut.  Any output may be NULL.  Synchronises. */
int schnorr_b200_keyset_debug_export(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, int device_index, size_t first,
                                     size_t count, uint8_t *pk96, uint8_t *pk_inf, uint8_t *status, uint64_t *tables,
                                     uint8_t *lut64, uint32_t *n_lut);

/* Compressed keys against a registered key set.  Registration also builds a sorted table of the set's encodings
 * (PublicKey::to_bytes of key k, src/public.rs:49-51, exactly as schnorr_b200_compress writes it), searched on the device
 * by binary search: at most log2(n_keys) + 1 probes whatever keys were registered.  Key k is FINDABLE when decompressing
 * its encoding (PublicKey::from_bytes, src/public.rs:54-56) gives back its registered record byte for byte (the same 96
 * bytes, the same identity flag).  Keys of status 3, points off the curve and an identity registered with non-zero
 * coordinates are therefore not findable; keys of status 1 are.
 *
 * keyset_lookup: key_idx[i] = the smallest findable index whose encoding equals keys49[i] exactly, or 0xFFFFFFFF (any
 * other 49 bytes miss, including undecodable encodings, flag bytes with bits 0x3f set and non-canonical limbs).  The
 * indices feed verify_registered_many and verify_batch_registered.  The host form runs on the first device of a
 * multi-device context; the _dev form (device buffers, no synchronisation) needs a single-device context. */
int schnorr_b200_keyset_lookup(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n, const uint8_t *keys49,
                               uint32_t *key_idx);
int schnorr_b200_keyset_lookup_dev(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n, const uint8_t *keys49,
                                   uint32_t *key_idx);
/* KeyedSignature::from_bytes + KeyedSignature::verify (src/signature.rs:232-271) over n 130-byte wire records, against
 * a registered key set: verdicts[i] is, byte for byte, what verify_keyed_many returns for record i.  A record whose key
 * bytes are the encoding of a findable key k takes the registered path of verify_registered_many with key k (the
 * decompressed key IS key k's record, so the verdict is verify_many's); every other record is decompressed and verified
 * as verify_keyed_many does (verdict 3 where the key does not decode).  Records whose key is not in the set cost more
 * than in verify_keyed_many (the exact kernel): the host form reads the miss count and runs verify_many on the decoded
 * records when more than 40 % of them miss; the _dev form does not synchronise and always takes the lookup path.  Calls
 * (per device) of at most set_one_threshold records: the host form takes the lookup path with the block-per-signature
 * kernel of verify_registered_many when every key was found and verify_many on the decoded records when any missed;
 * the _dev form runs verify_keyed_many.  last_exact_count (misses count as exact items),
 * last_kernel_ms and set_exact_only apply.  The host form shards a multi-device context in contiguous slices, each with
 * that device's copy of the set; the _dev form needs a single-device context and a non-NULL msgs. */
int schnorr_b200_verify_keyed_registered_many(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                              const uint8_t *keyed130, const uint8_t *msgs, const uint64_t *msg_off,
                                              uint8_t *verdicts);
int schnorr_b200_verify_keyed_registered_many_dev(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                  const uint8_t *keyed130, const uint8_t *msgs, const uint64_t *msg_off,
                                                  uint8_t *verdicts);

/* KeyedSignature::from_bytes + KeyedSignature::verify over n 130-byte wire records
 * (49-byte compressed public key || 81-byte signature)   src/signature.rs:232-271, src/constants.rs:33
 * The key is decompressed on the device; a record whose key does not decode gets verdict 3. */
int schnorr_b200_verify_keyed_many(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                   const uint64_t *msg_off, uint8_t *verdicts);
int schnorr_b200_verify_keyed_many_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                       const uint64_t *msg_off, uint8_t *verdicts);

/* verify_batch(&[Signature], &[PublicKey], &[&[u8]], rng)                  src/batch.rs:31-50
 * = generate_batch_coefficients (:56-81) + verify_prepared_batch (:84-130).
 * rand32: n x 32 B caller-supplied randomisers s_i (reduced mod q) -- the seam the reference has at
 * verify_prepared_batch.  *verdict: 0 / 2 / 3.  lhs97 / rhs97 (optional): affine x||y||inf of
 * sum s_i R_i - sum s_i h_i P_i  and of (sum s_i e_i) G  for bit-exact comparison. */
int schnorr_b200_verify_batch(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                              const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                              const uint8_t *rand32, int *verdict, uint8_t *lhs97, uint8_t *rhs97);
/* Same on DEVICE buffers (single-device context): enqueues the whole batch -- partial MSM, (sum s_i e_i) G on a second
 * stream beside it, finish -- and does not synchronise.  result216 (device): verdict(1) pad(7) lhs97 pad(7) rhs97 pad(7). */
int schnorr_b200_verify_batch_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                  const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                  const uint8_t *rand32, uint8_t *result216);
/* Multi-GPU form: each rank reduces its slice to one 192-byte partial (device buffer), the caller
 * gathers the partials (one small NCCL gather) and any rank finishes.  */
int schnorr_b200_batch_partial_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                   const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                   const uint8_t *rand32, uint8_t *partial192);
int schnorr_b200_batch_finish_dev(schnorr_b200_ctx *ctx, size_t n_partials, const uint8_t *partials192,
                                  uint8_t *result216 /* device, 216 B: verdict(1) pad(7) lhs97 pad(7) rhs97 pad(7) */);
int schnorr_b200_batch_finish(schnorr_b200_ctx *ctx, size_t n_partials, const uint8_t *partials192_host,
                              int *verdict, uint8_t *lhs97, uint8_t *rhs97);

/* Failed-batch localisation (SURVEY.md 8(f) f3).  The reference answers a bad batch with ONE Err for the lot
 * (src/batch.rs:125-129); this names the culprits, in BATCH semantics: item i is bad when its own term of the batch
 * equation, s_i D_i with D_i = R_i - h_i P_i - e_i G, R_i = from_compressed(sig_i.x) INCLUDING the flag byte and no
 * subgroup check on P_i (src/batch.rs:102-106), is not the identity -- e.g. a signature whose y-sign flag is flipped fails
 * the batch although Signature::verify (x-only, src/signature.rs:186,200) accepts it, while an item with s_i = 0, or with
 * a D_i of small order that its randomiser kills, cannot fail the batch and is not flagged, whichever items surround it.
 * Bisection over partial MSMs (a range whose own random linear combination holds is clean), exact per-item check on the
 * failing slices: only items inside a failing slice can be flagged, so items whose non-identity terms cancel within a
 * slice (two torsion-shifted R with odd randomisers: T2 + T2 = O) are not.  flags[i] = 0 clean, 2 bad, 3 malformed (the reference panics on it); *n_bad (optional) = number of
 * non-zero flags.  rand32 as in verify_batch.
 * The slices are defined by n alone, so the flags and *n_bad do not depend on the device count: the host forms of this
 * and of the three localisations below spread a multi-device context's work over up to 8 of its devices (one per 4096
 * signatures), each holding only its own contiguous range of the batch, and return the bytes of a single-device
 * context.  The _dev form (device buffers) needs a single-device context. */
int schnorr_b200_locate_invalid(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                const uint8_t *rand32, uint8_t *flags, uint64_t *n_bad);
int schnorr_b200_locate_invalid_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                    const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                    const uint8_t *rand32, uint8_t *flags);

/* verify_batch (src/batch.rs:31-130) against a registered key set: item i is signature sigs81[i] over message i under
 * key key_idx[i] of ks.  *verdict, lhs97 and rhs97 are, byte for byte, those of verify_batch on the gathered key records
 * pk96[i] = keys[key_idx[i]] (the same group elements, the same affine encodings); an index outside the set makes the
 * batch malformed (verdict 3), as does an item under a key of status 3.  Batch semantics are kept (src/batch.rs:102-106):
 * no subgroup check on the keys, identity keys contribute nothing.
 * The key side of the batch equation is summed per key, sum_i (s_i h_i) P_key(i) = sum_k c_k P_k: one product with the
 * key's table per distinct key instead of one MSM point per signature, so the MSM runs over the n points R_i only.  That
 * reduction of c_k mod q is valid only for keys with [q]P = O: a set that holds a key of status 1 runs every batch on
 * the per-signature points (still the same result) -- register only the keys of status 0 to get the aggregated path.
 * Batches of at most batch_small_max signatures, or with fewer than set_registered_batch_threshold signatures per key
 * of the set, also take the per-signature points.  The host form shards a multi-device context in contiguous slices
 * (one partial per shard from that device's copy of the set, finished on the first device); the _dev form (device
 * buffers, no synchronisation, result216 as in verify_batch_dev) needs a single-device context and a non-NULL msgs. */
int schnorr_b200_verify_batch_registered(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                         const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                         const uint64_t *msg_off, const uint8_t *rand32, int *verdict, uint8_t *lhs97,
                                         uint8_t *rhs97);
int schnorr_b200_verify_batch_registered_dev(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                             const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                             const uint64_t *msg_off, const uint8_t *rand32, uint8_t *result216);
/* locate_invalid (above) against a registered key set: the flags and *n_bad of locate_invalid on the gathered key
 * records; an index outside the set gets flag 3.  Each device gathers the records of its own range from its copy of
 * the set; the flags do not depend on the device count.                          src/batch.rs:102-129 */
int schnorr_b200_locate_invalid_registered(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                           const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                           const uint64_t *msg_off, const uint8_t *rand32, uint8_t *flags,
                                           uint64_t *n_bad);
/* verify_batch (src/batch.rs:31-130) over n 130-byte KeyedSignature wire records (49-byte compressed public key ||
 * 81-byte signature, src/signature.rs:237-271), message i and randomiser i.  *verdict, lhs97 and rhs97 are, byte for
 * byte, those of verify_batch on the FRONT-END records: for a record whose key decodes, its signature bytes and the
 * decoded key; for a record whose key does not decode, the record of an index outside a set (96 bytes of 0xFF,
 * identity flag 0), so the batch is malformed (verdict 3), as unwrapping KeyedSignature::from_bytes panics.  A scalar
 * e >= q is malformed as in verify_batch.  The host form shards a multi-device context in contiguous slices (one
 * partial per shard, finished on the first device); the _dev form (device buffers, no synchronisation, result216 as in
 * verify_batch_dev) needs a single-device context and a non-NULL msgs. */
int schnorr_b200_verify_batch_keyed(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                    const uint64_t *msg_off, const uint8_t *rand32, int *verdict, uint8_t *lhs97,
                                    uint8_t *rhs97);
int schnorr_b200_verify_batch_keyed_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                        const uint64_t *msg_off, const uint8_t *rand32, uint8_t *result216);
/* verify_batch_keyed against a registered key set: the same bytes as verify_batch_keyed on the same records, whatever
 * the set holds (src/signature.rs:237-271, src/batch.rs:31-130).  A record whose key bytes are the encoding of a
 * findable key k (keyset_lookup) takes key k's registered record; every other record (a miss) is decoded as in
 * verify_batch_keyed.  When the rules of verify_batch_registered select the key side summed per key (more than
 * batch_small_max records, no key of status 1 in the set, at least set_registered_batch_threshold records per key),
 * the hits' terms are summed per key and the MSM runs over the n points R_i and the m misses' keys: one path for any
 * mix of hits and misses, since a miss costs one MSM point.  The host form reads m (one synchronisation) and plans the
 * MSM for n + m points; the _dev form does not synchronise and plans for 2n.  Sharding and the _dev form's
 * requirements as in verify_batch_keyed. */
int schnorr_b200_verify_batch_keyed_registered(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                               const uint8_t *keyed130, const uint8_t *msgs, const uint64_t *msg_off,
                                               const uint8_t *rand32, int *verdict, uint8_t *lhs97, uint8_t *rhs97);
int schnorr_b200_verify_batch_keyed_registered_dev(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                   const uint8_t *keyed130, const uint8_t *msgs, const uint64_t *msg_off,
                                                   const uint8_t *rand32, uint8_t *result216);
/* locate_invalid (above) over keyed records, without and with a registered key set: the flags and *n_bad of
 * locate_invalid on the front-end records of verify_batch_keyed; a record whose key does not decode gets flag 3.  Each
 * device builds the records of its own range; the flags do not depend on the device count.
 *                                                    src/signature.rs:237-271, src/batch.rs:31-130 */
int schnorr_b200_locate_invalid_keyed(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                      const uint64_t *msg_off, const uint8_t *rand32, uint8_t *flags, uint64_t *n_bad);
int schnorr_b200_locate_invalid_keyed_registered(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                 const uint8_t *keyed130, const uint8_t *msgs, const uint64_t *msg_off,
                                                 const uint8_t *rand32, uint8_t *flags, uint64_t *n_bad);

/* Batch randomisers from a 32-byte seed: Scalar::random / generate_batch_coefficients (src/batch.rs:56-81, :75-78)
 * computed on the device.  Randomiser i of a seed is
 *     s_i = int_le(SHA-512("schnorr-sig_b200/batch-randomizer/v1" || seed32 || le64(i))) mod q
 * (32 canonical LE bytes): one SHA-512 compression, reduced wide like Scalar::random's 64 random bytes.  The batch
 * equation is sound only while the randomisers are unpredictable to whoever produced the signatures, so the seed must
 * be drawn fresh from a CSPRNG for every batch and kept from the signers until the verdict: a signer who knows the seed
 * in advance can build a batch whose invalid terms cancel.
 *
 * batch_randomizers writes randomisers first_index ... first_index + n - 1 to rand32 (n x 32 B).  EARG for a NULL seed
 * and when the last index, first_index + n - 1, does not fit in a u64.  The host form's bytes do not depend on the
 * device count of the context; the _dev form (seed32 and rand32 on the device, no synchronisation) needs a single-device
 * context.  The randomisers of a failed seeded batch are batch_randomizers(seed32, 0, n); the seeded localisations below
 * generate them on the devices. */
int schnorr_b200_batch_randomizers(schnorr_b200_ctx *ctx, size_t n, const uint8_t *seed32, uint64_t first_index,
                                   uint8_t *rand32);
int schnorr_b200_batch_randomizers_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *seed32, uint64_t first_index,
                                       uint8_t *rand32);
/* Seeded host forms of the four batch verifications (src/batch.rs:31-50 with generate_batch_coefficients, :56-81): the
 * arguments of the parent entry point with a 32-byte seed in place of rand32.  *verdict, lhs97 and rhs97 are, byte for
 * byte, the parent's given rand32 = batch_randomizers(seed32, 0, n).  The randomisers are generated on the device where
 * the batch runs (shard k of a multi-device context generates its own slice), so a call sends 32 bytes of randomness
 * instead of 32 per signature.  Path selection and sharding as in the parent.  EARG for a NULL seed. */
int schnorr_b200_verify_batch_seeded(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                     const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                     const uint8_t *seed32, int *verdict, uint8_t *lhs97, uint8_t *rhs97);
int schnorr_b200_verify_batch_registered_seeded(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                                const uint64_t *msg_off, const uint8_t *seed32, int *verdict,
                                                uint8_t *lhs97, uint8_t *rhs97);
int schnorr_b200_verify_batch_keyed_seeded(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                           const uint64_t *msg_off, const uint8_t *seed32, int *verdict, uint8_t *lhs97,
                                           uint8_t *rhs97);
int schnorr_b200_verify_batch_keyed_registered_seeded(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                      const uint8_t *keyed130, const uint8_t *msgs,
                                                      const uint64_t *msg_off, const uint8_t *seed32, int *verdict,
                                                      uint8_t *lhs97, uint8_t *rhs97);
/* Seeded host forms of the four localisations: the arguments of the parent entry point with a 32-byte seed in place of
 * rand32.  flags and *n_bad are, byte for byte, the parent's given rand32 = batch_randomizers(seed32, 0, n); each device
 * generates the randomisers of its own range, so a call sends 32 bytes of randomness instead of 32 per signature.  EARG
 * for a NULL seed. */
int schnorr_b200_locate_invalid_seeded(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sigs81, const uint8_t *pk96,
                                       const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                                       const uint8_t *seed32, uint8_t *flags, uint64_t *n_bad);
int schnorr_b200_locate_invalid_registered_seeded(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                  const uint8_t *sigs81, const uint32_t *key_idx, const uint8_t *msgs,
                                                  const uint64_t *msg_off, const uint8_t *seed32, uint8_t *flags,
                                                  uint64_t *n_bad);
int schnorr_b200_locate_invalid_keyed_seeded(schnorr_b200_ctx *ctx, size_t n, const uint8_t *keyed130, const uint8_t *msgs,
                                             const uint64_t *msg_off, const uint8_t *seed32, uint8_t *flags,
                                             uint64_t *n_bad);
int schnorr_b200_locate_invalid_keyed_registered_seeded(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, size_t n,
                                                        const uint8_t *keyed130, const uint8_t *msgs,
                                                        const uint64_t *msg_off, const uint8_t *seed32, uint8_t *flags,
                                                        uint64_t *n_bad);

/* MSM points of the last batch verification on this context (all devices of a multi-device context): 2n for
 * verify_batch, n for a registered batch summed per key, 0 for the block-per-signature form of small batches; for
 * keyed records summed per key, n + m (host forms, m misses) or 2n (the _dev form). */
int schnorr_b200_last_batch_points(const schnorr_b200_ctx *ctx, uint64_t *points);
/* Registered batches sum the key side per key when they hold at least `min_signatures_per_key` signatures per key of
 * the set (0: whenever the other rules allow it).  Default 64 (measured crossover, profiles/r4_registered_batch.md). */
int schnorr_b200_set_registered_batch_threshold(schnorr_b200_ctx *ctx, size_t min_signatures_per_key);

/* PublicKey::from(&PrivateKey) = BASEPOINT_TABLE * sk                      src/public.rs:26-32 */
int schnorr_b200_keygen(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sk32, uint8_t *pk96, uint8_t *pk_inf);
int schnorr_b200_keygen_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sk32, uint8_t *pk96, uint8_t *pk_inf);
/* KeyPair::sign(&self, message, rng) with the nonce r supplied by the caller  src/signature.rs:114-129 */
int schnorr_b200_sign_many(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sk32, const uint8_t *pk96,
                           const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                           const uint8_t *nonce32, uint8_t *sigs81);
int schnorr_b200_sign_many_dev(schnorr_b200_ctx *ctx, size_t n, const uint8_t *sk32, const uint8_t *pk96,
                               const uint8_t *pk_inf, const uint8_t *msgs, const uint64_t *msg_off,
                               const uint8_t *nonce32, uint8_t *sigs81);

/* Hierarchical deterministic key derivation (src/derivation.rs), n children per call, one child per thread:
 *   master keys      ExtendedPrivateKey::generate_master_key(seed)                   :66-84
 *                    seeds32: n x 32 B -> xsk64: n x (private key 32 B LE || chain code 32 B)
 *   private children ExtendedPrivateKey::derive_private(i) of ONE parent, hardened (i >= 2^31) or normal by index
 *                                                                                     :90-153
 *   public children  ExtendedPublicKey::derive_normal_public(i) of ONE parent        :249-277
 *                    xpk81 = PublicKey::to_bytes() 49 B || chain code 32 B (= ExtendedPublicKey::to_bytes, :280-286)
 * indices: n little-endian u32 (the reference's `&[u8; 4]`).  ok[i] = 1 where the reference returns Some: non-zero child
 * key / non-identity tweak point, and for public children a non-hardened index.  Records of children whose ok is 0 are
 * what the formulas give and must not be used.  HMAC-SHA512 and the fixed-base multiplication run on the device. */
int schnorr_b200_derive_master_keys(schnorr_b200_ctx *ctx, size_t n, const uint8_t *seeds32, uint8_t *xsk64, uint8_t *ok);
int schnorr_b200_derive_private_children(schnorr_b200_ctx *ctx, size_t n, const uint8_t *parent_xsk64,
                                         const uint32_t *indices, uint8_t *children_xsk64, uint8_t *ok);
int schnorr_b200_derive_public_children(schnorr_b200_ctx *ctx, size_t n, const uint8_t *parent_xpk81,
                                        const uint32_t *indices, uint8_t *children_xpk81, uint8_t *ok);

/* PublicKey::from_bytes / AffinePoint::from_compressed for n 49-byte records  src/public.rs:54-56
 * ok[i] = 1 when the record decodes (CtOption is_some). */
int schnorr_b200_decompress(schnorr_b200_ctx *ctx, size_t n, const uint8_t *in49, uint8_t *pk96, uint8_t *pk_inf,
                            uint8_t *ok);
/* AffinePoint::to_compressed / PublicKey::to_bytes                           src/public.rs:49-51 */
int schnorr_b200_compress(schnorr_b200_ctx *ctx, size_t n, const uint8_t *pk96, const uint8_t *pk_inf,
                          uint8_t *out49);

/* Test hook (no reference counterpart): raw device field operations so that the PTX arithmetic can be
 * checked against the oracle on edge values.  a6, b6: n x 6 canonical limbs (host); out48: n x 48 u64 =
 * fp6_mul(a,b) | fp6_sqr(a) | a+b | a-b | limb-wise a_k*b_k | limb-wise a_k^2 | fp6_inv(a) | limb-wise a_k^(1/7). */
int schnorr_b200_debug_field_ops(schnorr_b200_ctx *ctx, size_t n, const uint64_t *a6, const uint64_t *b6,
                                 uint64_t *out48);

/* Test hook (no reference counterpart): the lazily reduced building blocks of the fast path (csrc/debug_ops.cuh).
 * a6: n x 6 ARBITRARY 64-bit limbs (non-canonical representatives allowed), b6: n x 6 canonical limbs; out48: n x 48
 * u64 = a*rot(a) | a^2-2b | a^2-b-rot(b)*a3 | a*rot(a)-b*a5 | cofactor(b) | norm(b) | b*a0-rot(b)*a1 (nc form) |
 * b*a0-rot(b)*a1, all canonicalised. */
int schnorr_b200_debug_lazy_ops(schnorr_b200_ctx *ctx, size_t n, const uint64_t *a6, const uint64_t *b6,
                                uint64_t *out48);

/* Test hook (no reference counterpart): one operation of the device field core (csrc/fp.cuh) on n items of raw
 * 32-bit words, so that its carry and borrow paths can be driven word by word.  in16, out16: n x 16 u32 (host).
 * Scalar ops: a = in[0:2], b = in[2:4] (little-endian words of a 64-bit value, any value, canonical or not); the
 * reductions take x0..x4 = in[0:5]; FP_MUL_SMALL takes k and FP_SQR_N the count n from in[2]; the raw 64-bit result
 * (not reduced further) goes to out[0:2].  Accumulator ops: the state e0..e4, o1..o3 = in[0:8], a = in[8:10],
 * b = in[10:12], the repeat count of FP_WIDE_MAC_LOOP = in[12]; out[0:8] = the new state, out[8:10] =
 * wide_reduce_nc, out[10:12] = wide_reduce of it.  Unused output words are 0.  A bad op returns SCHNORR_B200_EARG. */
enum {
    SCHNORR_B200_FP_SUB = 0,
    SCHNORR_B200_FP_ADD,
    SCHNORR_B200_FP_NEG,
    SCHNORR_B200_FP_DBL,
    SCHNORR_B200_FP_REDUCE96_NC,
    SCHNORR_B200_FP_REDUCE96,
    SCHNORR_B200_FP_REDUCE160_NC,
    SCHNORR_B200_FP_REDUCE160,
    SCHNORR_B200_FP_CANON_SEL,
    SCHNORR_B200_FP_CANON,
    SCHNORR_B200_FP_MUL_NC,
    SCHNORR_B200_FP_SQR_NC,
    SCHNORR_B200_FP_MUL,
    SCHNORR_B200_FP_SQR,
    SCHNORR_B200_FP_MUL7_NC,
    SCHNORR_B200_FP_MUL_SMALL,
    SCHNORR_B200_FP_SQR_N,
    SCHNORR_B200_FP_INV,
    SCHNORR_B200_FP_WIDE_MAC, /* first accumulator op */
    SCHNORR_B200_FP_WIDE_MAC_SQR,
    SCHNORR_B200_FP_WIDE_ADD64,
    SCHNORR_B200_FP_WIDE_DOUBLE,
    SCHNORR_B200_FP_WIDE_REDUCE,
    SCHNORR_B200_FP_WIDE_MAC_LOOP,
    SCHNORR_B200_FP_OP_COUNT
};
int schnorr_b200_debug_fp_core(schnorr_b200_ctx *ctx, int op, size_t n, const uint32_t *in16, uint32_t *out16);

/* Test hook (no reference counterpart): the point stage of Signature::verify (src/signature.rs:181-205) on a GIVEN
 * challenge, so that exceptional group elements can be placed in chosen stages of one core.  n items of pk96 (affine
 * x || y, not the identity), h32 and e32 (little-endian scalars below q), all n x ... host arrays.  CORE_EXACT runs the
 * complete Jacobian routine (torsion_check_and_mul + fixed_base_accumulate), CORE_FAST the per-thread (X, Y, w) core of
 * k_verify_fast (verify_core_fast), CORE_DIST its six-lane form of k_verify_dist (dverify_core).  result[i] = 0 when
 * [q]P == O, 1 when not, 2 when the core met an exceptional case (never for CORE_EXACT); r97[i] = affine x || y of
 * h*P + e*G and a byte 1 for the identity (meaningful unless result[i] == 2).  A bad core returns SCHNORR_B200_EARG. */
enum { SCHNORR_B200_CORE_EXACT = 0, SCHNORR_B200_CORE_FAST, SCHNORR_B200_CORE_DIST, SCHNORR_B200_CORE_COUNT };
int schnorr_b200_debug_verify_core(schnorr_b200_ctx *ctx, int core, size_t n, const uint8_t *pk96, const uint8_t *h32,
                                   const uint8_t *e32, uint8_t *result, uint8_t *r97);
/* Test hook (no reference counterpart): the point stage of a verification against a registered key on a GIVEN
 * challenge, key key_idx[i] of the set (EARG for an index at or beyond n_keys), h32 / e32 as in debug_verify_core.
 * REG_CORE_THREAD runs the per-thread table core of verify_registered_many's large calls (verify_core_reg),
 * REG_CORE_BLOCK the table tree, + e*G, of its block-per-signature form.  result[i] = 0, or 2 when the core met an
 * exceptional case (the block core only for a collision in its e*G stage, never for e < q); r97 as in
 * debug_verify_core.  Runs on the first device of a multi-device context.  A bad core returns SCHNORR_B200_EARG. */
enum { SCHNORR_B200_REG_CORE_THREAD = 0, SCHNORR_B200_REG_CORE_BLOCK, SCHNORR_B200_REG_CORE_COUNT };
int schnorr_b200_debug_verify_registered_core(schnorr_b200_ctx *ctx, const schnorr_b200_keyset *ks, int core, size_t n,
                                              const uint32_t *key_idx, const uint8_t *h32, const uint8_t *e32,
                                              uint8_t *result, uint8_t *r97);

/* Integer-multiply roofline calibration: runs a register-resident chain of `iters` dependent-free
 * 32x32->64 multiply-adds per thread on a full grid and returns wide multiplies per second. */
int schnorr_b200_imad_peak(schnorr_b200_ctx *ctx, int iters, double *wide_mul_per_s, double *elapsed_ms);

#ifdef __cplusplus
}
#endif
#endif /* SCHNORR_B200_H */
