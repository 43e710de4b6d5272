// Hierarchical deterministic key derivation (reference src/derivation.rs:66-277; SURVEY.md §8(f) f4): BIP32-like
// chain codes with HMAC-SHA512 and ONE fixed-base multiplication per public child.  Data-parallel use: many children
// of one parent (wallet scanning, address generation) -- one child per thread.
//
//   ExtendedPrivateKey::generate_master_key   :66-84    I = HMAC("Cheetah - Master extended key seed", seed)
//   derive_hardened_private                    :101-124  I = HMAC(chain, 0^17 || sk || i),        i >= 2^31
//   derive_normal_private                      :130-153  I = HMAC(chain, PublicKey(sk).to_bytes() || i), i < 2^31
//   ExtendedPublicKey::derive_normal_public    :249-277  I = HMAC(chain, pk.to_bytes() || i),  child = I_L G + pk
//   child key = Scalar::from_bytes_non_canonical(I_L) + sk, child chain code = I_R; None when the key is zero / the
//   point I_L G is the identity / the index is of the wrong kind.
//
// SHA-512 / HMAC are plain 64-bit integer code (FIPS 180-4, RFC 2104), compiled for the device and -- for the CPU
// tests only -- for the host.
#pragma once
#include "curve.cuh"

namespace sb {

#if defined(__CUDACC__)
#define SB_SHA_TABLE __device__ static const
#else
#define SB_SHA_TABLE static const
#endif
SB_SHA_TABLE uint64_t SHA512_K[80] = {
    0x428a2f98d728ae22ULL, 0x7137449123ef65cdULL, 0xb5c0fbcfec4d3b2fULL, 0xe9b5dba58189dbbcULL, 0x3956c25bf348b538ULL,
    0x59f111f1b605d019ULL, 0x923f82a4af194f9bULL, 0xab1c5ed5da6d8118ULL, 0xd807aa98a3030242ULL, 0x12835b0145706fbeULL,
    0x243185be4ee4b28cULL, 0x550c7dc3d5ffb4e2ULL, 0x72be5d74f27b896fULL, 0x80deb1fe3b1696b1ULL, 0x9bdc06a725c71235ULL,
    0xc19bf174cf692694ULL, 0xe49b69c19ef14ad2ULL, 0xefbe4786384f25e3ULL, 0x0fc19dc68b8cd5b5ULL, 0x240ca1cc77ac9c65ULL,
    0x2de92c6f592b0275ULL, 0x4a7484aa6ea6e483ULL, 0x5cb0a9dcbd41fbd4ULL, 0x76f988da831153b5ULL, 0x983e5152ee66dfabULL,
    0xa831c66d2db43210ULL, 0xb00327c898fb213fULL, 0xbf597fc7beef0ee4ULL, 0xc6e00bf33da88fc2ULL, 0xd5a79147930aa725ULL,
    0x06ca6351e003826fULL, 0x142929670a0e6e70ULL, 0x27b70a8546d22ffcULL, 0x2e1b21385c26c926ULL, 0x4d2c6dfc5ac42aedULL,
    0x53380d139d95b3dfULL, 0x650a73548baf63deULL, 0x766a0abb3c77b2a8ULL, 0x81c2c92e47edaee6ULL, 0x92722c851482353bULL,
    0xa2bfe8a14cf10364ULL, 0xa81a664bbc423001ULL, 0xc24b8b70d0f89791ULL, 0xc76c51a30654be30ULL, 0xd192e819d6ef5218ULL,
    0xd69906245565a910ULL, 0xf40e35855771202aULL, 0x106aa07032bbd1b8ULL, 0x19a4c116b8d2d0c8ULL, 0x1e376c085141ab53ULL,
    0x2748774cdf8eeb99ULL, 0x34b0bcb5e19b48a8ULL, 0x391c0cb3c5c95a63ULL, 0x4ed8aa4ae3418acbULL, 0x5b9cca4f7763e373ULL,
    0x682e6ff3d6b2b8a3ULL, 0x748f82ee5defb2fcULL, 0x78a5636f43172f60ULL, 0x84c87814a1f0ab72ULL, 0x8cc702081a6439ecULL,
    0x90befffa23631e28ULL, 0xa4506cebde82bde9ULL, 0xbef9a3f7b2c67915ULL, 0xc67178f2e372532bULL, 0xca273eceea26619cULL,
    0xd186b8c721c0c207ULL, 0xeada7dd6cde0eb1eULL, 0xf57d4f7fee6ed178ULL, 0x06f067aa72176fbaULL, 0x0a637dc5a2c898a6ULL,
    0x113f9804bef90daeULL, 0x1b710b35131c471bULL, 0x28db77f523047d84ULL, 0x32caab7b40c72493ULL, 0x3c9ebe0a15c9bebcULL,
    0x431d67c49c100d4cULL, 0x4cc5d4becb3e42b6ULL, 0x597f299cfc657e2aULL, 0x5fcb6fab3ad6faecULL, 0x6c44198c4a475817ULL,
};

struct sha512_state {
    uint64_t h[8];
};
SB_DEV uint64_t sha_rotr(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }
SB_DEV void sha512_init(sha512_state& s) {
    s.h[0] = 0x6a09e667f3bcc908ULL; s.h[1] = 0xbb67ae8584caa73bULL; s.h[2] = 0x3c6ef372fe94f82bULL; s.h[3] = 0xa54ff53a5f1d36f1ULL;
    s.h[4] = 0x510e527fade682d1ULL; s.h[5] = 0x9b05688c2b3e6c1fULL; s.h[6] = 0x1f83d9abfb41bd6bULL; s.h[7] = 0x5be0cd19137e2179ULL;
}
// one 128-byte block (big-endian words)
SB_DEV void sha512_compress(sha512_state& s, const uint8_t* block) {
    uint64_t w[16];
#pragma unroll
    for (int i = 0; i < 16; i++) {
        uint64_t v = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) v = (v << 8) | block[8 * i + k];
        w[i] = v;
    }
    uint64_t a = s.h[0], b = s.h[1], c = s.h[2], d = s.h[3], e = s.h[4], f = s.h[5], g = s.h[6], h = s.h[7];
#pragma unroll 1
    for (int t = 0; t < 80; t++) {
        uint64_t wt;
        if (t < 16) {
            wt = w[t & 15];
        } else {
            uint64_t w15 = w[(t - 15) & 15], w2 = w[(t - 2) & 15];
            uint64_t s0 = sha_rotr(w15, 1) ^ sha_rotr(w15, 8) ^ (w15 >> 7);
            uint64_t s1 = sha_rotr(w2, 19) ^ sha_rotr(w2, 61) ^ (w2 >> 6);
            wt = w[t & 15] + s0 + w[(t - 7) & 15] + s1;
            w[t & 15] = wt;
        }
        uint64_t S1 = sha_rotr(e, 14) ^ sha_rotr(e, 18) ^ sha_rotr(e, 41);
        uint64_t ch = (e & f) ^ (~e & g);
        uint64_t t1 = h + S1 + ch + SHA512_K[t] + wt;
        uint64_t S0 = sha_rotr(a, 28) ^ sha_rotr(a, 34) ^ sha_rotr(a, 39);
        uint64_t mj = (a & b) ^ (a & c) ^ (b & c);
        uint64_t t2 = S0 + mj;
        h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    s.h[0] += a; s.h[1] += b; s.h[2] += c; s.h[3] += d; s.h[4] += e; s.h[5] += f; s.h[6] += g; s.h[7] += h;
}
// SHA-512 of `prefix_blocks` already-compressed 128-byte blocks followed by `len` <= 111 bytes of `data` (one final block)
SB_DEV void sha512_finish_short(sha512_state& s, int prefix_blocks, const uint8_t* data, int len, uint8_t* out64) {
    uint8_t blk[128];
    for (int i = 0; i < 128; i++) blk[i] = i < len ? data[i] : 0;
    blk[len] = 0x80;
    uint64_t bits = ((uint64_t)prefix_blocks * 128 + (uint64_t)len) * 8;
    for (int k = 0; k < 8; k++) blk[127 - k] = (uint8_t)(bits >> (8 * k));
    sha512_compress(s, blk);
    for (int i = 0; i < 8; i++)
        for (int k = 0; k < 8; k++) out64[8 * i + k] = (uint8_t)(s.h[i] >> (56 - 8 * k));
}
// HMAC-SHA512(key, data) for a key of at most 128 bytes and data of at most 111 bytes: 4 compressions
SB_DEV void hmac_sha512_short(const uint8_t* key, int key_len, const uint8_t* data, int data_len, uint8_t* out64) {
    uint8_t pad[128];
    sha512_state inner, outer;
    sha512_init(inner);
    for (int i = 0; i < 128; i++) pad[i] = (uint8_t)((i < key_len ? key[i] : 0) ^ 0x36);
    sha512_compress(inner, pad);
    uint8_t digest[64];
    sha512_finish_short(inner, 1, data, data_len, digest);
    sha512_init(outer);
    for (int i = 0; i < 128; i++) pad[i] = (uint8_t)((i < key_len ? key[i] : 0) ^ 0x5c);
    sha512_compress(outer, pad);
    sha512_finish_short(outer, 1, digest, 64, out64);
}

// ---- batch randomisers (include/schnorr_b200.h, schnorr_b200_batch_randomizers) -------------------------------------
// s_i = int_le(SHA-512(TAG || seed || le64(i))) mod q: one compression of 76 bytes per signature index, reduced wide as
// Scalar::random reduces 64 random bytes
SB_DEV scalar batch_randomizer(const uint8_t* seed32, uint64_t index) {
    const char tag[] = "schnorr-sig_b200/batch-randomizer/v1";
    uint8_t msg[76], d[64];
    for (int i = 0; i < 36; i++) msg[i] = (uint8_t)tag[i];
    for (int i = 0; i < 32; i++) msg[36 + i] = seed32[i];
    for (int b = 0; b < 8; b++) msg[68 + b] = (uint8_t)(index >> (8 * b));
    sha512_state s;
    sha512_init(s);
    sha512_finish_short(s, 0, msg, 76, d);
    return sc_from_u512(sc_load_le(d), sc_load_le(d + 32));
}

// ---- derivation steps (byte layouts: include/schnorr_b200.h) ---------------------------------------------------------
// master: seed32 -> (sk32 || chain32); returns false for a zero key
SB_DEV bool derive_master(const uint8_t* seed32, uint8_t* xsk64) {
    const char label[] = "Cheetah - Master extended key seed";   // src/derivation.rs:67
    uint8_t key[34], I[64];
    for (int i = 0; i < 34; i++) key[i] = (uint8_t)label[i];
    hmac_sha512_short(key, 34, seed32, 32, I);
    scalar k = sc_from_u256(sc_load_le(I));                       // Scalar::from_bytes_non_canonical
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) xsk64[4 * i + b] = (uint8_t)(k.l[i] >> (8 * b));
    for (int i = 0; i < 32; i++) xsk64[32 + i] = I[32 + i];
    return !sc_is_zero(k);
}
// private child of (sk, chain) for index i; parent_pk49 = PublicKey::from(sk).to_bytes() (used by normal children)
SB_DEV bool derive_private_child(const uint8_t* parent_xsk64, const uint8_t* parent_pk49, uint32_t index, uint8_t* child_xsk64) {
    uint8_t data[53], I[64];
    bool hardened = (index >> 31) != 0;
    for (int i = 0; i < 49; i++) data[i] = hardened ? (i < 17 ? 0 : parent_xsk64[i - 17]) : parent_pk49[i];
    for (int b = 0; b < 4; b++) data[49 + b] = (uint8_t)(index >> (8 * b));
    hmac_sha512_short(parent_xsk64 + 32, 32, data, 53, I);
    scalar k = sc_add(sc_from_u256(sc_load_le(I)), sc_from_u256(sc_load_le(parent_xsk64)));
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) child_xsk64[4 * i + b] = (uint8_t)(k.l[i] >> (8 * b));
    for (int i = 0; i < 32; i++) child_xsk64[32 + i] = I[32 + i];
    return !sc_is_zero(k);
}
// public child: I_L (as a scalar) and the child's chain code; the caller adds I_L G to the parent point
SB_DEV scalar derive_public_tweak(const uint8_t* parent_pk49, const uint8_t* chain32, uint32_t index, uint8_t* child_chain32) {
    uint8_t data[53], I[64];
    for (int i = 0; i < 49; i++) data[i] = parent_pk49[i];
    for (int b = 0; b < 4; b++) data[49 + b] = (uint8_t)(index >> (8 * b));
    hmac_sha512_short(chain32, 32, data, 53, I);
    for (int i = 0; i < 32; i++) child_chain32[i] = I[32 + i];
    return sc_from_u256(sc_load_le(I));
}

}  // namespace sb
