// TEST-ONLY host build of the lookup of compressed keys in registered key sets (schnorr-sig_b200/csrc/keyset.cuh) with
// g++, for tests/test_keyed_registered_hostsim.py.  It extends the registered-key-set host build (registered.cpp,
// included whole) with the exports below; like it, it is not part of the product.
#include "registered.cpp"

// the encoding of a registered key as k_keyset_encode writes it: out49 = x limbs || flag byte; returns findable
API int hs_keyset_encode(const uint8_t* pk96, int inf, uint8_t* out49) {
    uint64_t pt[12], x[6];
    memcpy(pt, pk96, 96);
    uint8_t flag;
    bool findable = keyset_encode(pt, inf != 0, x, flag);
    memcpy(out49, x, 48);
    out49[48] = flag;
    return findable;
}
// the lookup table of n keys as registration builds it (k_keyset_encode, then keyset_sort_entries on the findable
// keys): out = up to n entries of 64 bytes; returns the number of entries
API size_t hs_keyset_table(size_t n, const uint8_t* pk96, const uint8_t* inf, keyset_entry* out) {
    size_t m = 0;
    for (size_t k = 0; k < n; k++) {
        uint64_t pt[12];
        memcpy(pt, pk96 + 96 * k, 96);
        keyset_entry e;
        uint8_t flag;
        if (!keyset_encode(pt, inf[k] != 0, e.x, flag)) continue;
        e.flag = flag;
        e.index = (uint32_t)k;
        e.pad = 0;
        out[m++] = e;
    }
    return keyset_sort_entries(out, m);
}
// keyset_lookup of n 49-byte keys against a table of n_entries entries (hs_keyset_table)
API void hs_keyset_lookup(const keyset_entry* tab, uint32_t n_entries, size_t n, const uint8_t* keys49, uint32_t* out) {
    for (size_t i = 0; i < n; i++) {
        uint64_t x[6];
        memcpy(x, keys49 + 49 * i, 48);
        out[i] = keyset_lookup(tab, n_entries, x, keys49[49 * i + 48]);
    }
}
