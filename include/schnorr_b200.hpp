// schnorr_b200.hpp -- header-only C++ host facade over the C ABI (schnorr_b200.h).
//
// The reference is compiled code (Rust); no Rust toolchain exists on this image, so the host side
// above the C ABI is written in C++ and mirrors the reference's public interface for the hot path:
// same names, argument meaning and error behaviour.
//
//   schnorr_sig::Signature::verify(message, pkey)            src/signature.rs:181-205
//   schnorr_sig::PublicKey::verify_signature(sig, message)   src/signature.rs:170-176
//   schnorr_sig::KeyedSignature::verify(message)             src/signature.rs:232-234
//   schnorr_sig::verify_batch(signatures, public_keys, messages, rng)   src/batch.rs:31-50
//   schnorr_sig::SignatureError {InvalidPublicKey, InvalidSignature}     src/error.rs:13-31
//   to_bytes()/from_bytes() of Signature / PublicKey          src/signature.rs:208-227, src/public.rs:49-56
//
// Result<(), SignatureError> is std::optional<SignatureError> (nullopt = Ok).  Inputs on which the
// reference panics (unwrap of a non-canonical encoding, length-mismatch asserts) throw std::logic_error.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <functional>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "schnorr_b200.h"

namespace schnorr_sig {

constexpr size_t SCALAR_LENGTH = 32, BASEFIELD_LENGTH = 48, PUBLIC_KEY_LENGTH = 49, SIGNATURE_LENGTH = 81,
                 KEYED_SIGNATURE_LENGTH = 130;  // src/constants.rs:12-33

enum class SignatureError { InvalidPublicKey = 1, InvalidSignature = 2 };
inline const char* to_string(SignatureError e) {
    return e == SignatureError::InvalidPublicKey ? "The public key is not an element of the prime subgroup."
                                                 : "The signature is invalid or was incorrectly computed.";
}
using Result = std::optional<SignatureError>;  // nullopt == Ok(())

// One engine (CUDA context, tables, scratch) per process and device; not thread-safe per instance.
class Engine {
public:
    explicit Engine(int device = 0) {
        if (schnorr_b200_create(device, &ctx_) != SCHNORR_B200_OK || !ctx_)
            throw std::runtime_error("schnorr_b200_create failed: a CUDA device is required (no CPU fallback)");
    }
    ~Engine() { schnorr_b200_destroy(ctx_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    schnorr_b200_ctx* get() const { return ctx_; }
    static Engine& instance() {
        static Engine e(0);
        return e;
    }
    void check(int rc, const char* what) const {
        if (rc != SCHNORR_B200_OK) throw std::runtime_error(std::string(what) + ": " + schnorr_b200_last_error(ctx_));
    }

private:
    schnorr_b200_ctx* ctx_ = nullptr;
};

inline Result result_from_verdict(int v) {
    switch (v) {
        case 0: return std::nullopt;
        case 1: return SignatureError::InvalidPublicKey;
        case 2: return SignatureError::InvalidSignature;
        default: throw std::logic_error("called `Option::unwrap()` on a `None` value (non-canonical encoding)");
    }
}

struct Signature;
struct KeyedSignature;

// PublicKey(AffinePoint): affine x || y little-endian limbs + identity flag (src/public.rs:24)
struct PublicKey {
    std::array<uint8_t, 96> xy{};
    bool infinity = false;

    std::array<uint8_t, PUBLIC_KEY_LENGTH> to_bytes() const {
        std::array<uint8_t, PUBLIC_KEY_LENGTH> out{};
        uint8_t inf = infinity;
        Engine::instance().check(schnorr_b200_compress(Engine::instance().get(), 1, xy.data(), &inf, out.data()), "compress");
        return out;
    }
    // CtOption<Self>
    static std::optional<PublicKey> from_bytes(const std::array<uint8_t, PUBLIC_KEY_LENGTH>& b) {
        PublicKey k;
        uint8_t inf = 0, ok = 0;
        Engine::instance().check(schnorr_b200_decompress(Engine::instance().get(), 1, b.data(), k.xy.data(), &inf, &ok), "decompress");
        if (!ok) return std::nullopt;
        k.infinity = inf != 0;
        return k;
    }
    Result verify_signature(const Signature& signature, const std::vector<uint8_t>& message) const;
};

// Signature { x: CompressedPoint, e: Scalar } (src/signature.rs:34-40)
struct Signature {
    std::array<uint8_t, 49> x{};
    std::array<uint8_t, 32> e{};

    std::array<uint8_t, SIGNATURE_LENGTH> to_bytes() const {
        std::array<uint8_t, SIGNATURE_LENGTH> out{};
        std::memcpy(out.data(), x.data(), 49);
        std::memcpy(out.data() + 49, e.data(), 32);
        return out;
    }
    static Signature from_raw(const std::array<uint8_t, SIGNATURE_LENGTH>& b) {
        Signature s;
        std::memcpy(s.x.data(), b.data(), 49);
        std::memcpy(s.e.data(), b.data() + 49, 32);
        return s;
    }
    Result verify(const std::vector<uint8_t>& message, const PublicKey& pkey) const {
        auto sig = to_bytes();
        uint64_t off[2] = {0, message.size()};
        uint8_t inf = pkey.infinity, verdict = 255;
        Engine& eng = Engine::instance();
        eng.check(schnorr_b200_verify_many(eng.get(), 1, sig.data(), pkey.xy.data(), &inf,
                                           message.empty() ? nullptr : message.data(), off, &verdict),
                  "verify_many");
        return result_from_verdict(verdict);
    }
};

inline Result PublicKey::verify_signature(const Signature& signature, const std::vector<uint8_t>& message) const {
    return signature.verify(message, *this);
}

// Public keys registered once for many verifications (schnorr_b200_keyset_*): the subgroup check and the per-key
// table are computed at construction; verify_signature(i, ...) gives what Signature::verify gives under keys[i].
class KeySet {
public:
    KeySet(Engine& eng, const std::vector<PublicKey>& keys) : eng_(eng) {
        size_t n = keys.size();
        std::vector<uint8_t> pks(n * 96), inf(n);
        for (size_t i = 0; i < n; i++) {
            std::memcpy(&pks[i * 96], keys[i].xy.data(), 96);
            inf[i] = keys[i].infinity;
        }
        status_.assign(n, 255);
        eng_.check(schnorr_b200_keyset_create(eng_.get(), n, pks.data(), inf.data(), status_.data(), &ks_), "keyset_create");
    }
    explicit KeySet(const std::vector<PublicKey>& keys) : KeySet(Engine::instance(), keys) {}
    ~KeySet() { schnorr_b200_keyset_destroy(ks_); }
    KeySet(const KeySet&) = delete;
    KeySet& operator=(const KeySet&) = delete;
    schnorr_b200_keyset* get() const { return ks_; }
    // per key: 0 = in the prime-order subgroup (identity included), 1 = not, 3 = non-canonical limb
    const std::vector<uint8_t>& status() const { return status_; }
    size_t size() const { return status_.size(); }
    // an index outside the set throws, as indexing past the end of a slice panics.  One signature runs one thread block
    // over the key's table (the latency form, schnorr_b200_set_one_threshold): no doubling chain, no subgroup check
    Result verify_signature(size_t index, const Signature& signature, const std::vector<uint8_t>& message) const {
        auto sig = signature.to_bytes();
        uint64_t off[2] = {0, message.size()};
        uint32_t idx = index < size() ? (uint32_t)index : UINT32_MAX;
        uint8_t verdict = 255;
        eng_.check(schnorr_b200_verify_registered_many(eng_.get(), ks_, 1, sig.data(), &idx,
                                                       message.empty() ? nullptr : message.data(), off, &verdict),
                   "verify_registered_many");
        return result_from_verdict(verdict);
    }
    // index of the key whose encoding is exactly `key49` and which decompresses to its registered record (the smallest
    // such index; schnorr_b200_keyset_lookup), nullopt when there is none
    std::optional<uint32_t> index_of(const std::array<uint8_t, PUBLIC_KEY_LENGTH>& key49) const {
        uint32_t idx = UINT32_MAX;
        eng_.check(schnorr_b200_keyset_lookup(eng_.get(), ks_, 1, key49.data(), &idx), "keyset_lookup");
        if (idx == UINT32_MAX) return std::nullopt;
        return idx;
    }
    std::optional<uint32_t> index_of(const PublicKey& key) const { return index_of(key.to_bytes()); }
    // KeyedSignature::verify(message) (schnorr_b200_verify_keyed_registered_many): the registered path when the key is
    // in the set (one thread block over the key's table, as verify_signature), what KeyedSignature::verify gives
    // otherwise; a key or scalar that does not decode throws
    Result verify_keyed(const std::array<uint8_t, KEYED_SIGNATURE_LENGTH>& keyed, const std::vector<uint8_t>& message) const {
        uint64_t off[2] = {0, message.size()};
        uint8_t verdict = 255;
        eng_.check(schnorr_b200_verify_keyed_registered_many(eng_.get(), ks_, 1, keyed.data(),
                                                             message.empty() ? nullptr : message.data(), off, &verdict),
                   "verify_keyed_registered_many");
        return result_from_verdict(verdict);
    }
    Result verify_keyed(const KeyedSignature& keyed, const std::vector<uint8_t>& message) const;
    // registers `keys` in the next slots (schnorr_b200_keyset_append) -> the index of the first; status() and size()
    // follow
    size_t append(const std::vector<PublicKey>& keys) {
        size_t first = size();
        std::vector<uint8_t> pks, inf, st(keys.size(), 255);
        pack_keys(keys, pks, inf);
        eng_.check(schnorr_b200_keyset_append(eng_.get(), ks_, keys.size(), pks.data(), inf.data(), st.data()), "keyset_append");
        status_.insert(status_.end(), st.begin(), st.end());
        return first;
    }
    // registers keys[j] in slot indices[j] (distinct, inside the set; schnorr_b200_keyset_replace)
    void replace(const std::vector<size_t>& indices, const std::vector<PublicKey>& keys) {
        if (indices.size() != keys.size()) throw std::logic_error("one index per key");
        std::vector<uint32_t> idx = checked_indices(indices);
        std::vector<uint8_t> pks, inf, st(keys.size(), 255);
        pack_keys(keys, pks, inf);
        eng_.check(schnorr_b200_keyset_replace(eng_.get(), ks_, keys.size(), idx.data(), pks.data(), inf.data(), st.data()),
                   "keyset_replace");
        for (size_t j = 0; j < idx.size(); j++) status_[idx[j]] = st[j];
    }
    // removes slots (schnorr_b200_keyset_remove): they keep their index, and using it throws as an index outside the
    // set does (verdict 3); status 3
    void remove(const std::vector<size_t>& indices) {
        std::vector<uint32_t> idx = checked_indices(indices);
        eng_.check(schnorr_b200_keyset_remove(eng_.get(), ks_, idx.size(), idx.data()), "keyset_remove");
        for (uint32_t k : idx) status_[k] = 3;
    }
    // verify_batch(signatures, [keys[i] for i in indices], messages, rng) with the key side summed per key of the set
    // (schnorr_b200_verify_batch_registered); an index outside the set makes the batch malformed, which throws
    Result verify_batch(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                        const std::vector<std::vector<uint8_t>>& messages,
                        const std::function<void(uint8_t*, size_t)>& rng) const;
    // indices of the items whose own term of the batch equation fails (schnorr_b200_locate_invalid_registered); a
    // malformed item or an index outside the set throws
    std::vector<size_t> locate_invalid(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                       const std::vector<std::vector<uint8_t>>& messages,
                                       const std::function<void(uint8_t*, size_t)>& rng) const;
    // verify_batch_keyed (below) with the records whose key is in the set taking its registered record and the key side
    // summed per key (schnorr_b200_verify_batch_keyed_registered): the same result
    Result verify_batch_keyed(const std::vector<KeyedSignature>& keyed, const std::vector<std::vector<uint8_t>>& messages,
                              const std::function<void(uint8_t*, size_t)>& rng) const;
    // locate_invalid_keyed (below) against the set (schnorr_b200_locate_invalid_keyed_registered)
    std::vector<size_t> locate_invalid_keyed(const std::vector<KeyedSignature>& keyed,
                                             const std::vector<std::vector<uint8_t>>& messages,
                                             const std::function<void(uint8_t*, size_t)>& rng) const;
    // the same four with the randomisers generated on the devices from a 32-byte seed (schnorr_b200_batch_randomizers;
    // schnorr_b200_verify_batch_registered_seeded ... schnorr_b200_locate_invalid_keyed_registered_seeded): the seed must
    // be fresh from a CSPRNG for every batch and unknown to the signers until the verdict
    Result verify_batch(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                        const std::vector<std::vector<uint8_t>>& messages, const std::array<uint8_t, 32>& seed) const;
    std::vector<size_t> locate_invalid(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                       const std::vector<std::vector<uint8_t>>& messages,
                                       const std::array<uint8_t, 32>& seed) const;
    Result verify_batch_keyed(const std::vector<KeyedSignature>& keyed, const std::vector<std::vector<uint8_t>>& messages,
                              const std::array<uint8_t, 32>& seed) const;
    std::vector<size_t> locate_invalid_keyed(const std::vector<KeyedSignature>& keyed,
                                             const std::vector<std::vector<uint8_t>>& messages,
                                             const std::array<uint8_t, 32>& seed) const;

private:
    static void pack_keys(const std::vector<PublicKey>& keys, std::vector<uint8_t>& pks, std::vector<uint8_t>& inf) {
        pks.resize(keys.size() * 96);
        inf.resize(keys.size());
        for (size_t i = 0; i < keys.size(); i++) {
            std::memcpy(&pks[i * 96], keys[i].xy.data(), 96);
            inf[i] = keys[i].infinity;
        }
    }
    std::vector<uint32_t> checked_indices(const std::vector<size_t>& indices) const {
        std::vector<uint32_t> idx(indices.size());
        for (size_t j = 0; j < indices.size(); j++) {
            if (indices[j] >= size()) throw std::logic_error("index out of bounds: the key set has fewer slots");
            idx[j] = (uint32_t)indices[j];
        }
        return idx;
    }
    struct BatchInputs {
        std::vector<uint8_t> sigs, rand, blob;
        std::vector<uint32_t> idx;
        std::vector<uint64_t> off;
    };
    BatchInputs batch_inputs(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                             const std::vector<std::vector<uint8_t>>& messages,
                             const std::function<void(uint8_t*, size_t)>& rng) const;
    // batch_inputs without the randomisers
    BatchInputs batch_records(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                              const std::vector<std::vector<uint8_t>>& messages) const;
    Result registered_verdict(const BatchInputs& in, const uint8_t* seed) const;
    std::vector<size_t> registered_located(const BatchInputs& in, const uint8_t* seed) const;
    Engine& eng_;
    schnorr_b200_keyset* ks_ = nullptr;
    std::vector<uint8_t> status_;
};

struct KeyedSignature {
    PublicKey public_key;
    Signature signature;
    Result verify(const std::vector<uint8_t>& message) const { return signature.verify(message, public_key); }
    std::array<uint8_t, KEYED_SIGNATURE_LENGTH> to_bytes() const {
        std::array<uint8_t, KEYED_SIGNATURE_LENGTH> out{};
        auto k = public_key.to_bytes();
        auto s = signature.to_bytes();
        std::memcpy(out.data(), k.data(), PUBLIC_KEY_LENGTH);
        std::memcpy(out.data() + PUBLIC_KEY_LENGTH, s.data(), SIGNATURE_LENGTH);
        return out;
    }
};

inline Result KeySet::verify_keyed(const KeyedSignature& keyed, const std::vector<uint8_t>& message) const {
    return verify_keyed(keyed.to_bytes(), message);
}

// rng(buf, len) fills len random bytes (CryptoRng + RngCore).  One full-width random scalar is drawn
// per signature (src/batch.rs:75-78); 32 bytes with the top two bits cleared are uniform below 2^254 < q.
using Rng = std::function<void(uint8_t*, size_t)>;

// the signature and key records and the messages of a batch
struct BatchArrays {
    std::vector<uint8_t> sigs, pks, inf, blob;
    std::vector<uint64_t> off;
    size_t n() const { return off.size() - 1; }
    const uint8_t* msgs() const { return blob.empty() ? nullptr : blob.data(); }
};
inline BatchArrays batch_arrays(const std::vector<Signature>& signatures, const std::vector<PublicKey>& public_keys,
                                const std::vector<std::vector<uint8_t>>& messages) {
    if (signatures.size() != public_keys.size())
        throw std::logic_error("We should have the same number of signatures than public keys");
    if (messages.size() != public_keys.size())
        throw std::logic_error("We should have the same number of messages than public keys");
    size_t n = signatures.size();
    BatchArrays a;
    a.sigs.resize(n * 81);
    a.pks.resize(n * 96);
    a.inf.resize(n);
    a.off.assign(n + 1, 0);
    for (size_t i = 0; i < n; i++) {
        auto b = signatures[i].to_bytes();
        std::memcpy(&a.sigs[i * 81], b.data(), 81);
        std::memcpy(&a.pks[i * 96], public_keys[i].xy.data(), 96);
        a.inf[i] = public_keys[i].infinity;
        a.blob.insert(a.blob.end(), messages[i].begin(), messages[i].end());
        a.off[i + 1] = a.blob.size();
    }
    return a;
}

inline Result verify_batch(const std::vector<Signature>& signatures, const std::vector<PublicKey>& public_keys,
                           const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) {
    BatchArrays a = batch_arrays(signatures, public_keys, messages);
    size_t n = a.n();
    std::vector<uint8_t> rand(n * 32);
    rng(rand.data(), rand.size());
    for (size_t i = 0; i < n; i++) rand[i * 32 + 31] &= 0x3f;
    int verdict = -1;
    Engine& eng = Engine::instance();
    eng.check(schnorr_b200_verify_batch(eng.get(), n, a.sigs.data(), a.pks.data(), a.inf.data(), a.msgs(), a.off.data(),
                                        rand.data(), &verdict, nullptr, nullptr),
              "verify_batch");
    return result_from_verdict(verdict);
}

// verify_batch with the randomisers generated on the device from a 32-byte seed (schnorr_b200_verify_batch_seeded): the
// seed must be fresh from a CSPRNG for every batch and unknown to the signers until the verdict
inline Result verify_batch(const std::vector<Signature>& signatures, const std::vector<PublicKey>& public_keys,
                           const std::vector<std::vector<uint8_t>>& messages, const std::array<uint8_t, 32>& seed) {
    BatchArrays a = batch_arrays(signatures, public_keys, messages);
    int verdict = -1;
    Engine& eng = Engine::instance();
    eng.check(schnorr_b200_verify_batch_seeded(eng.get(), a.n(), a.sigs.data(), a.pks.data(), a.inf.data(), a.msgs(),
                                               a.off.data(), seed.data(), &verdict, nullptr, nullptr),
              "verify_batch_seeded");
    return result_from_verdict(verdict);
}

// the randomisers 0 ... n - 1 of a seed, as the seeded entry points generate them (schnorr_b200_batch_randomizers)
inline std::vector<uint8_t> batch_randomizers(Engine& eng, size_t n, const std::array<uint8_t, 32>& seed) {
    std::vector<uint8_t> rand(n * 32);
    eng.check(schnorr_b200_batch_randomizers(eng.get(), n, seed.data(), 0, rand.data()), "batch_randomizers");
    return rand;
}

inline KeySet::BatchInputs KeySet::batch_records(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                                 const std::vector<std::vector<uint8_t>>& messages) const {
    if (signatures.size() != indices.size())
        throw std::logic_error("We should have the same number of signatures than public keys");
    if (messages.size() != indices.size())
        throw std::logic_error("We should have the same number of messages than public keys");
    size_t n = signatures.size();
    BatchInputs in;
    in.sigs.resize(n * 81);
    in.idx.resize(n);
    in.off.assign(n + 1, 0);
    for (size_t i = 0; i < n; i++) {
        auto b = signatures[i].to_bytes();
        std::memcpy(&in.sigs[i * 81], b.data(), 81);
        in.idx[i] = indices[i] < size() ? (uint32_t)indices[i] : UINT32_MAX;
        in.blob.insert(in.blob.end(), messages[i].begin(), messages[i].end());
        in.off[i + 1] = in.blob.size();
    }
    return in;
}

inline KeySet::BatchInputs KeySet::batch_inputs(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                                const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) const {
    BatchInputs in = batch_records(indices, signatures, messages);
    size_t n = in.idx.size();
    in.rand.resize(n * 32);
    rng(in.rand.data(), in.rand.size());
    for (size_t i = 0; i < n; i++) in.rand[i * 32 + 31] &= 0x3f;
    return in;
}

// the verdict of a registered batch: randomisers from in.rand, or generated on the device from `seed` when it is not null
inline Result KeySet::registered_verdict(const BatchInputs& in, const uint8_t* seed) const {
    int verdict = -1;
    const uint8_t* msgs = in.blob.empty() ? nullptr : in.blob.data();
    if (seed)
        eng_.check(schnorr_b200_verify_batch_registered_seeded(eng_.get(), ks_, in.idx.size(), in.sigs.data(), in.idx.data(),
                                                               msgs, in.off.data(), seed, &verdict, nullptr, nullptr),
                   "verify_batch_registered_seeded");
    else
        eng_.check(schnorr_b200_verify_batch_registered(eng_.get(), ks_, in.idx.size(), in.sigs.data(), in.idx.data(), msgs,
                                                        in.off.data(), in.rand.data(), &verdict, nullptr, nullptr),
                   "verify_batch_registered");
    return result_from_verdict(verdict);
}

inline Result KeySet::verify_batch(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                   const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) const {
    return registered_verdict(batch_inputs(indices, signatures, messages, rng), nullptr);
}

inline Result KeySet::verify_batch(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                   const std::vector<std::vector<uint8_t>>& messages, const std::array<uint8_t, 32>& seed) const {
    return registered_verdict(batch_records(indices, signatures, messages), seed.data());
}

inline std::vector<size_t> KeySet::locate_invalid(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                                  const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) const {
    return registered_located(batch_inputs(indices, signatures, messages, rng), nullptr);
}

inline std::vector<size_t> KeySet::locate_invalid(const std::vector<size_t>& indices, const std::vector<Signature>& signatures,
                                                  const std::vector<std::vector<uint8_t>>& messages,
                                                  const std::array<uint8_t, 32>& seed) const {
    return registered_located(batch_records(indices, signatures, messages), seed.data());
}

// the culprits of a registered batch: randomisers from in.rand, or generated on the devices from `seed` when it is not null
inline std::vector<size_t> KeySet::registered_located(const BatchInputs& in, const uint8_t* seed) const {
    size_t n = in.idx.size();
    std::vector<uint8_t> flags(n, 0);
    const uint8_t* msgs = in.blob.empty() ? nullptr : in.blob.data();
    if (seed)
        eng_.check(schnorr_b200_locate_invalid_registered_seeded(eng_.get(), ks_, n, in.sigs.data(), in.idx.data(), msgs,
                                                                 in.off.data(), seed, flags.data(), nullptr),
                   "locate_invalid_registered_seeded");
    else
        eng_.check(schnorr_b200_locate_invalid_registered(eng_.get(), ks_, n, in.sigs.data(), in.idx.data(), msgs,
                                                          in.off.data(), in.rand.data(), flags.data(), nullptr),
                   "locate_invalid_registered");
    std::vector<size_t> bad;
    for (size_t i = 0; i < n; i++) {
        if (flags[i] == 3) throw std::logic_error("called `Option::unwrap()` on a `None` value (non-canonical encoding)");
        if (flags[i]) bad.push_back(i);
    }
    return bad;
}

// the 130-byte records, messages and randomisers of a batch over keyed signatures
struct KeyedBatchInputs {
    std::vector<uint8_t> recs, rand, blob;
    std::vector<uint64_t> off;
    size_t n() const { return off.size() - 1; }
};
// keyed_batch_inputs without the randomisers
inline KeyedBatchInputs keyed_batch_records(const std::vector<KeyedSignature>& keyed,
                                            const std::vector<std::vector<uint8_t>>& messages) {
    if (messages.size() != keyed.size()) throw std::logic_error("We should have the same number of messages than signatures");
    size_t n = keyed.size();
    KeyedBatchInputs in;
    in.recs.resize(n * KEYED_SIGNATURE_LENGTH);
    in.off.assign(n + 1, 0);
    for (size_t i = 0; i < n; i++) {
        auto b = keyed[i].to_bytes();
        std::memcpy(&in.recs[i * KEYED_SIGNATURE_LENGTH], b.data(), KEYED_SIGNATURE_LENGTH);
        in.blob.insert(in.blob.end(), messages[i].begin(), messages[i].end());
        in.off[i + 1] = in.blob.size();
    }
    return in;
}
inline KeyedBatchInputs keyed_batch_inputs(const std::vector<KeyedSignature>& keyed,
                                           const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) {
    KeyedBatchInputs in = keyed_batch_records(keyed, messages);
    size_t n = in.n();
    in.rand.resize(n * 32);
    rng(in.rand.data(), in.rand.size());
    for (size_t i = 0; i < n; i++) in.rand[i * 32 + 31] &= 0x3f;
    return in;
}
inline std::vector<size_t> located(const std::vector<uint8_t>& flags) {
    std::vector<size_t> bad;
    for (size_t i = 0; i < flags.size(); i++) {
        if (flags[i] == 3) throw std::logic_error("called `Option::unwrap()` on a `None` value (non-canonical encoding)");
        if (flags[i]) bad.push_back(i);
    }
    return bad;
}

// the verdict of verify_batch_keyed (ks null) or of verify_batch_keyed_registered on prepared records: randomisers from
// in.rand, or generated on the device from `seed` when it is not null
inline Result keyed_verdict(Engine& eng, const schnorr_b200_keyset* ks, const KeyedBatchInputs& in, const uint8_t* seed) {
    int verdict = -1;
    const uint8_t* msgs = in.blob.empty() ? nullptr : in.blob.data();
    if (ks && seed)
        eng.check(schnorr_b200_verify_batch_keyed_registered_seeded(eng.get(), ks, in.n(), in.recs.data(), msgs, in.off.data(),
                                                                    seed, &verdict, nullptr, nullptr),
                  "verify_batch_keyed_registered_seeded");
    else if (ks)
        eng.check(schnorr_b200_verify_batch_keyed_registered(eng.get(), ks, in.n(), in.recs.data(), msgs, in.off.data(),
                                                             in.rand.data(), &verdict, nullptr, nullptr),
                  "verify_batch_keyed_registered");
    else if (seed)
        eng.check(schnorr_b200_verify_batch_keyed_seeded(eng.get(), in.n(), in.recs.data(), msgs, in.off.data(), seed, &verdict,
                                                         nullptr, nullptr),
                  "verify_batch_keyed_seeded");
    else
        eng.check(schnorr_b200_verify_batch_keyed(eng.get(), in.n(), in.recs.data(), msgs, in.off.data(), in.rand.data(),
                                                  &verdict, nullptr, nullptr),
                  "verify_batch_keyed");
    return result_from_verdict(verdict);
}
// the culprits of locate_invalid_keyed (ks null) or of locate_invalid_keyed_registered on prepared records: randomisers
// from in.rand, or generated on the devices from `seed` when it is not null
inline std::vector<size_t> keyed_culprits(Engine& eng, const schnorr_b200_keyset* ks, const KeyedBatchInputs& in,
                                          const uint8_t* seed) {
    std::vector<uint8_t> flags(in.n(), 0);
    const uint8_t* msgs = in.blob.empty() ? nullptr : in.blob.data();
    if (ks && seed)
        eng.check(schnorr_b200_locate_invalid_keyed_registered_seeded(eng.get(), ks, in.n(), in.recs.data(), msgs,
                                                                      in.off.data(), seed, flags.data(), nullptr),
                  "locate_invalid_keyed_registered_seeded");
    else if (ks)
        eng.check(schnorr_b200_locate_invalid_keyed_registered(eng.get(), ks, in.n(), in.recs.data(), msgs, in.off.data(),
                                                               in.rand.data(), flags.data(), nullptr),
                  "locate_invalid_keyed_registered");
    else if (seed)
        eng.check(schnorr_b200_locate_invalid_keyed_seeded(eng.get(), in.n(), in.recs.data(), msgs, in.off.data(), seed,
                                                           flags.data(), nullptr),
                  "locate_invalid_keyed_seeded");
    else
        eng.check(schnorr_b200_locate_invalid_keyed(eng.get(), in.n(), in.recs.data(), msgs, in.off.data(), in.rand.data(),
                                                    flags.data(), nullptr),
                  "locate_invalid_keyed");
    return located(flags);
}

// verify_batch([k.signature ...], [k.public_key ...], messages, rng) over KeyedSignature wire records, the keys decoded on
// the device (schnorr_b200_verify_batch_keyed); a key that does not decode makes the batch malformed, which throws
inline Result verify_batch_keyed(const std::vector<KeyedSignature>& keyed, const std::vector<std::vector<uint8_t>>& messages,
                                 const Rng& rng) {
    return keyed_verdict(Engine::instance(), nullptr, keyed_batch_inputs(keyed, messages, rng), nullptr);
}
// indices of the records whose own term of the batch equation fails (schnorr_b200_locate_invalid_keyed); a record whose
// key or signature does not decode throws
inline std::vector<size_t> locate_invalid_keyed(const std::vector<KeyedSignature>& keyed,
                                                const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) {
    return keyed_culprits(Engine::instance(), nullptr, keyed_batch_inputs(keyed, messages, rng), nullptr);
}
// the same two with the randomisers generated on the devices from a 32-byte seed (schnorr_b200_verify_batch_keyed_seeded,
// schnorr_b200_locate_invalid_keyed_seeded): the seed must be fresh from a CSPRNG for every batch and unknown to the signers until
// the verdict
inline Result verify_batch_keyed(const std::vector<KeyedSignature>& keyed, const std::vector<std::vector<uint8_t>>& messages,
                                 const std::array<uint8_t, 32>& seed) {
    return keyed_verdict(Engine::instance(), nullptr, keyed_batch_records(keyed, messages), seed.data());
}
inline std::vector<size_t> locate_invalid_keyed(const std::vector<KeyedSignature>& keyed,
                                                const std::vector<std::vector<uint8_t>>& messages,
                                                const std::array<uint8_t, 32>& seed) {
    return keyed_culprits(Engine::instance(), nullptr, keyed_batch_records(keyed, messages), seed.data());
}
inline Result KeySet::verify_batch_keyed(const std::vector<KeyedSignature>& keyed,
                                         const std::vector<std::vector<uint8_t>>& messages, const Rng& rng) const {
    return keyed_verdict(eng_, ks_, keyed_batch_inputs(keyed, messages, rng), nullptr);
}
inline std::vector<size_t> KeySet::locate_invalid_keyed(const std::vector<KeyedSignature>& keyed,
                                                        const std::vector<std::vector<uint8_t>>& messages,
                                                        const Rng& rng) const {
    return keyed_culprits(eng_, ks_, keyed_batch_inputs(keyed, messages, rng), nullptr);
}
inline Result KeySet::verify_batch_keyed(const std::vector<KeyedSignature>& keyed,
                                         const std::vector<std::vector<uint8_t>>& messages,
                                         const std::array<uint8_t, 32>& seed) const {
    return keyed_verdict(eng_, ks_, keyed_batch_records(keyed, messages), seed.data());
}
inline std::vector<size_t> KeySet::locate_invalid_keyed(const std::vector<KeyedSignature>& keyed,
                                                        const std::vector<std::vector<uint8_t>>& messages,
                                                        const std::array<uint8_t, 32>& seed) const {
    return keyed_culprits(eng_, ks_, keyed_batch_records(keyed, messages), seed.data());
}

}  // namespace schnorr_sig
