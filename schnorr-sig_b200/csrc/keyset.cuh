// Registered key sets (schnorr_b200_keyset_create / schnorr_b200_verify_registered_many): verification of many
// signatures under a small, recurring set of public keys.  Everything in Signature::verify (src/signature.rs:181-205)
// that depends on the key alone is done once per key at registration:
//   - the subgroup check [q]P == O (exact, torsion_check_and_mul) -> a status byte per key;
//   - the doubling chain 2^j P, frozen into a signed-window table of affine multiples of P, the layout of the G table.
// A verification is then the challenge hash plus KT_WINDOWS table additions for h*P and GTAB_WINDOWS for e*G, all in
// the (X, Y, w) coordinates of the fast path (affine.cuh), with the same exceptional-case hand-back to the exact kernel.
// Public keys are public data: the tables are indexed by the challenge digits and are not constant-time (DESIGN.md §7).
// Written once and instantiated by the CUDA kernels (schnorr_b200.cu) and by the host test build (tests/hostsim).
#pragma once
#include <algorithm>
#include <vector>

#include "verify.cuh"

namespace sb {

// Window width of the per-key tables: ktab[key][KT_WINDOWS][KT_ENTRIES], entry d of window i = d * 2^(KT_W i) * P.
// 8 bits: 32 windows x 129 entries x 96 B = 396 KB per key (profiles/r3_registered.md: 7 / 8 / 10 measured).
#ifndef SB_KT_W
#define SB_KT_W 8
#endif
static constexpr int KT_W = SB_KT_W;
static constexpr int KT_WINDOWS = 255 / KT_W + 1;  // challenges are reduced mod q < 2^255
static_assert(KT_WINDOWS * KT_W > 255, "the top window of a challenge must not carry out");
static constexpr int KT_ENTRIES = (1 << (KT_W - 1)) + 1;
static constexpr size_t KT_KEY_U64 = (size_t)KT_WINDOWS * KT_ENTRIES * 12;

// Registration status of a key (schnorr_b200.h)
enum key_status : uint8_t {
    KEY_OK = 0,              // in the prime-order subgroup (the identity included)
    KEY_NOT_TORSION_FREE = 1,
    KEY_MALFORMED = 3,       // a non-canonical limb (ignored for the identity, as k_ingest does)
};
// `d` = storage for the running point of the doubling chain (torsion_check_and_mul)
SB_DEV uint8_t keyset_key_status(const uint64_t* pk12, bool inf, jac_pt* d) {
    if (inf) return KEY_OK;
    fp6 x, y;
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        x.c[k] = pk12[k];
        y.c[k] = pk12[6 + k];
        ok &= x.c[k] < FP_P && y.c[k] < FP_P;
    }
    if (!ok) return KEY_MALFORMED;
    jac_pt r;
    return torsion_check_and_mul(jac_from_affine(x, y, false), sc_zero(), &r, d) ? KEY_OK : KEY_NOT_TORSION_FREE;
}

// ---- signed-window table builder (the G table and the per-key tables) --------------------------------------------
// bases[i] = 2^(w i) P for i < windows: one chain of doublings
SB_DEV void tab_bases(const uint64_t* pt12, int w, int windows, jac_pt* bases) {
    fp6 x, y;
    for (int k = 0; k < 6; k++) {
        x.c[k] = pt12[k];
        y.c[k] = pt12[6 + k];
    }
    jac_pt p = jac_from_affine(x, y, false);
#pragma unroll 1
    for (int i = 0; i < windows; i++) {
        if (i)
#pragma unroll 1
            for (int k = 0; k < w; k++) jac_dbl_mem(&p);
        bases[i] = p;
    }
}
// out12 = affine x || y of d * base (d < 2^w); d = 0 (the identity) is written as zeros and never read
SB_DEV void tab_entry(const jac_pt& base, int w, int d, uint64_t* out12) {
    jac_pt acc = jac_identity();
#pragma unroll 1
    for (int bit = w - 1; bit >= 0; bit--) {
        jac_dbl_mem(&acc);
        if ((d >> bit) & 1) jac_add_mem(&acc, &base, false);
    }
    fp6 x, y;
    bool inf;
    jac_to_affine(acc, x, y, inf);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        out12[k] = x.c[k];
        out12[6 + k] = y.c[k];
    }
}

// ---- verification against a registered key ----------------------------------------------------------------------
// acc += k * P from a signed-window table of affine multiples of P (the layout of gtab, curve.cuh):
//   tab[i][d] = d * 2^(W i) * P,  1 <= d <= 2^(W-1)  (slot 0 unused),  k = sum_i d_i 2^(W i),  |d_i| <= 2^(W-1).
// WINDOWS * W must exceed the bit length of k (no carry out of the top window).  One addition per window, a block
// barrier every fourth (every thread of the block must call this).  `acc_empty` (in / out): acc is the identity.
// `exc` is set when an active addition met x(acc) == x(entry): acc is then not the sum and the caller goes exact.
// verify_core_fast (affine.cuh) keeps its own copy of the G loop: instantiating this helper there changed the SASS of
// k_verify_fast (9704 -> 9688 instructions), the tuned kernel this path must leave as it is.
template <int W, int WINDOWS>
SB_DEV void jf_table_accumulate(jf_pt* acc, bool& acc_empty, bool& exc, const scalar& k, const uint64_t* __restrict__ tab) {
    constexpr int ENTRIES = (1 << (W - 1)) + 1;
    int carry = 0;
    jf_pt T;
    T.w = 1;
#pragma unroll 1
    for (int i = 0; i < WINDOWS; i++) {
        if ((i & 3) == 0) SB_PHASE_SYNC(1);
        int raw = (int)sc_bits(k, W * i, W) + carry;
        bool neg = raw > (1 << (W - 1));
        carry = neg ? 1 : 0;
        int dg = neg ? (1 << W) - raw : raw;
        const uint64_t* ent = tab + ((size_t)i * ENTRIES + (dg ? dg : 1)) * 12;
#if defined(__CUDA_ARCH__)
        const ulonglong2* e2 = reinterpret_cast<const ulonglong2*>(ent);
        ulonglong2 a = e2[0], b = e2[1], c = e2[2], dd = e2[3], ee = e2[4], f = e2[5];
        T.X = fp6{{a.x, a.y, b.x, b.y, c.x, c.y}};
        T.Y = fp6{{dd.x, dd.y, ee.x, ee.y, f.x, f.y}};
#else
        for (int c = 0; c < 6; c++) {
            T.X.c[c] = ent[c];
            T.Y.c[c] = ent[6 + c];
        }
#endif
        exc |= jf_add<true>(acc, &T, jf_add_mode(acc_empty, dg == 0, neg));
        acc_empty = acc_empty && dg == 0;
    }
}

// R = h*P + e*G from the key's table and the G table.  FAST_TORSION_FREE: *R is that point.  FAST_EXCEPTIONAL: an
// addition met x(acc) == x(entry), or the result is the identity -- the exact routine decides.  Every thread of the
// block must call this (block barriers inside the loops).
SB_DEV int verify_core_reg(const scalar& h, const scalar& e, const uint64_t* __restrict__ ktab_key,
                           const uint64_t* __restrict__ gtab, jf_pt* R) {
    R->X = fp6_zero();  // defined contents for the masked additions that read it
    R->Y = fp6_zero();
    R->w = 1;
    bool empty = true;
    bool exc = false;
    jf_table_accumulate<KT_W, KT_WINDOWS>(R, empty, exc, h, ktab_key);
    jf_table_accumulate<GTAB_W, GTAB_WINDOWS>(R, empty, exc, e, gtab);
    return (exc || empty) ? FAST_EXCEPTIONAL : FAST_TORSION_FREE;
}

// Verdict of a signature whose record passed the malformed check and whose key is not the identity, with the
// precedence of verify_points: off-subgroup key, then a non-canonical sig.x, then the comparison x(R) == sig.x
// (src/signature.rs:182-200).  VERDICT_NEEDS_EXACT: finish it with verify_points.
SB_DEV uint8_t reg_verdict(uint8_t status, bool x_ok, int fr, const jf_pt& r, const fp6& sig_x) {
    if (status == KEY_NOT_TORSION_FREE) return VERDICT_INVALID_PUBLIC_KEY;
    if (!x_ok) return VERDICT_MALFORMED;
    if (fr == FAST_EXCEPTIONAL) return VERDICT_NEEDS_EXACT;
    return fp6_eq(r.X, fp6_scale(sig_x, fp_sqr_nc(r.w))) ? VERDICT_OK : VERDICT_INVALID_SIGNATURE;
}

// ---- lookup of compressed keys (KeyedSignature records, src/signature.rs:232-271) --------------------------------
// The encoding of a registered key is compress(pk, inf), the 49 bytes k_compress writes: the x limbs (zeros for the
// identity) and the flag byte.  A key is findable when decompressing its encoding (src/public.rs:54-56) gives back its
// registered record exactly, so a hit can take the registered record in place of the decompressed one.  That one rule
// leaves out non-canonical limbs (they do not decode), points off the curve (y does not round-trip) and an identity
// registered with non-zero coordinates.  The lookup table holds the findable encodings sorted by keyset_cmp, one entry
// per distinct encoding (the smallest index); a query is a binary search: log2(entries) + 1 probes whatever the keys.
static constexpr uint32_t KEYSET_MISS = 0xFFFFFFFFu;
struct keyset_entry {  // 64 bytes: one aligned line pair per probe
    uint64_t x[6];
    uint32_t flag;
    uint32_t index;
    uint64_t pad;
};
static_assert(sizeof(keyset_entry) == 64, "lookup entries are 64 bytes");

// the encoding of (pk12, inf) into x6 / flag; returns whether the key is findable
SB_DEV bool keyset_encode(const uint64_t* pk12, bool inf, uint64_t* x6, uint8_t& flag) {
    fp6 x, y;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        x.c[k] = inf ? 0 : pk12[k];
        y.c[k] = pk12[6 + k];
        x6[k] = x.c[k];
    }
    flag = compress_flags(y, inf);
    fp6 ox, oy;
    bool oinf;
    bool same = decompress_point(x, flag, ox, oy, oinf) && oinf == inf;
#pragma unroll
    for (int k = 0; k < 6; k++) same &= ox.c[k] == pk12[k] && oy.c[k] == pk12[6 + k];
    return same;
}

// order of the lookup table: limbs from the most significant, then the flag byte (< 0: the query sorts first).
// Also compiled for the host, where the table is sorted (keyset_sort_entries).
#if defined(__CUDACC__)
__host__ __device__ __forceinline__
#else
static inline
#endif
int keyset_cmp(const uint64_t* x6, uint32_t flag, const keyset_entry* e) {
#pragma unroll
    for (int k = 5; k >= 0; k--) {
        uint64_t v = e->x[k];
        if (x6[k] != v) return x6[k] < v ? -1 : 1;
    }
    return flag == e->flag ? 0 : (flag < e->flag ? -1 : 1);
}

// index of the registered key whose encoding is exactly (x6, flag), or KEYSET_MISS: a lower-bound search over the
// n_entries entries of `tab`
SB_DEV uint32_t keyset_lookup(const keyset_entry* __restrict__ tab, uint32_t n_entries, const uint64_t* x6, uint32_t flag) {
    uint32_t lo = 0, len = n_entries;
#pragma unroll 1
    while (len > 0) {
        uint32_t half = len >> 1;
        if (keyset_cmp(x6, flag, tab + lo + half) > 0) {
            lo += half + 1;
            len -= half + 1;
        } else {
            len = half;
        }
    }
    return lo < n_entries && keyset_cmp(x6, flag, tab + lo) == 0 ? tab[lo].index : KEYSET_MISS;
}

// Host side of the table build: `entries` holds one entry per findable key (any order); sorts them and keeps the
// smallest index of every encoding.  Returns the number of entries kept at the front.
static inline size_t keyset_sort_entries(keyset_entry* entries, size_t n) {
    std::sort(entries, entries + n, [](const keyset_entry& a, const keyset_entry& b) {
        int c = keyset_cmp(a.x, a.flag, &b);
        return c != 0 ? c < 0 : a.index < b.index;
    });
    size_t m = 0;
    for (size_t i = 0; i < n; i++)
        if (m == 0 || keyset_cmp(entries[i].x, entries[i].flag, &entries[m - 1]) != 0) entries[m++] = entries[i];
    return m;
}

// Host side of an in-place update (schnorr_b200_keyset_append / _replace / _remove).  `all` holds the entry of every
// findable slot, duplicate encodings included, sorted by (encoding, index).  The entries of the slots with
// changed[index] != 0 are deleted, `added` (the new entries of the changed slots that are findable, any order) is
// merged in, and `lut` receives the smallest index of every encoding: what keyset_sort_entries gives from scratch over
// the findable slots, in O(K + m log m) for m added entries instead of a sort of the whole set.
static inline void keyset_update_entries(std::vector<keyset_entry>& all, const uint8_t* changed, size_t n_slots,
                                         std::vector<keyset_entry> added, std::vector<keyset_entry>& lut) {
    auto less = [](const keyset_entry& a, const keyset_entry& b) {
        int c = keyset_cmp(a.x, a.flag, &b);
        return c != 0 ? c < 0 : a.index < b.index;
    };
    size_t m = 0;
    for (size_t i = 0; i < all.size(); i++)
        if (all[i].index >= n_slots || !changed[all[i].index]) all[m++] = all[i];
    all.resize(m);
    std::sort(added.begin(), added.end(), less);
    std::vector<keyset_entry> merged(all.size() + added.size());
    std::merge(all.begin(), all.end(), added.begin(), added.end(), merged.begin(), less);
    all.swap(merged);
    lut.clear();
    for (const keyset_entry& e : all)
        if (lut.empty() || keyset_cmp(e.x, e.flag, &lut.back()) != 0) lut.push_back(e);
}

// ---- batch verification against registered keys (src/batch.rs:84-130) -------------------------------------------
// The key side of the batch equation collapses to one term per distinct key:
//     sum_i t_i (-P_key(i)) = sum_k c_k (-P_k),   t_i = s_i h_i mod q,   c_k = sum_{i: key(i) = k} t_i mod q.
// Reducing the sum mod q is only valid for keys with [q]P_k = O (status KEY_OK): a set that holds a key of status
// KEY_NOT_TORSION_FREE runs its batches on the per-signature points instead (schnorr_b200.h).
//
// c_k from the 64-bit column sums col[j] = sum_i limb_j(t_i) of the eight 32-bit limbs.  Every column is below
// n 2^32 with n < 2^32 items, so the carry chain stays within 64 bits and the value is lo + hi 2^256 with hi < 2^32:
// c = (lo mod q) + hi 2^256 mod q, the second term a Montgomery product of hi with 2^512 mod q.
SB_DEV scalar keyset_sum_reduce(const uint64_t* col) {
    scalar lo, hi = sc_zero(), r2;
    uint64_t carry = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        uint64_t v = col[j] + carry;  // col[j] <= (2^32 - 1)^2 and carry < 2^32: no wrap
        lo.l[j] = (uint32_t)v;
        carry = v >> 32;
    }
    hi.l[0] = (uint32_t)carry;
#pragma unroll
    for (int j = 0; j < 8; j++) r2.l[j] = SB_CONST_R2(j);
    return sc_add(sc_from_u256(lo), sc_montmul(hi, r2));
}

// The addend of window `window` (< KT_WINDOWS) of c (-P) from the key's table: the signed digit recoded as in
// jf_table_accumulate, entry |d| of that window, negated for a positive digit.  The identity (w = 0) for d = 0.
SB_DEV jf_pt keyset_window_term(const scalar& c, int window, const uint64_t* __restrict__ ktab_key) {
    int carry = 0, d = 0;
    bool neg = false;
#pragma unroll 1
    for (int i = 0; i <= window; i++) {
        int raw = (int)sc_bits(c, KT_W * i, KT_W) + carry;
        neg = raw > (1 << (KT_W - 1));
        carry = neg ? 1 : 0;
        d = neg ? (1 << KT_W) - raw : raw;
    }
    jf_pt t;
    t.X = fp6_one();
    t.Y = fp6_one();
    t.w = 0;
    if (d) {
        const uint64_t* ent = ktab_key + ((size_t)window * KT_ENTRIES + d) * 12;
#pragma unroll
        for (int k = 0; k < 6; k++) {
            t.X.c[k] = ent[k];
            t.Y.c[k] = ent[6 + k];
        }
        if (!neg) t.Y = fp6_neg(t.Y);
        t.w = 1;
    }
    return t;
}

}  // namespace sb
