// TEST-ONLY host build of the key side of batches against registered key sets (schnorr-sig_b200/csrc/keyset.cuh) with
// g++, for tests/test_registered_batch_hostsim.py.  It extends the registered-key-set host build (registered.cpp,
// included whole) with the exports below; like it, it is not part of the product.
#include "registered.cpp"

// c = (sum of the limb columns col8[0..8) as one integer) mod q, as k_keyset_batch_term reduces the column sums of
// k_keyset_scalar_sum
API void hs_keyset_sum_reduce(const uint64_t* col8, uint8_t* out32) { stsc(out32, keyset_sum_reduce(col8)); }

// c (-P) from the key's table (hs_tab_build at KT_W) as one warp of k_keyset_batch_term forms it: lane i's addend
// (keyset_window_term), then the shuffle tree of exact additions, lane by lane (a lane past the end reads the identity).
// out96 = the affine result; returns 1 for the identity.
API int hs_keyset_key_term(const uint64_t* ktab, const uint8_t* c32, uint8_t* out96) {
    scalar c = ldsc(c32);
    jf_pt lane[32];
    for (int l = 0; l < 32; l++) {
        if (l < KT_WINDOWS) {
            lane[l] = keyset_window_term(c, l, ktab);
        } else {
            lane[l].X = fp6_one();
            lane[l].Y = fp6_one();
            lane[l].w = 0;
        }
    }
    for (int d = 16; d >= 1; d >>= 1) {
        jf_pt next[32];
        for (int l = 0; l < 32; l++) {
            next[l] = lane[l];
            if (l + d < 32) jf_add_exact(&next[l], &lane[l + d]);
        }
        for (int l = 0; l < 32; l++) lane[l] = next[l];
    }
    if (lane[0].w == 0) {
        memset(out96, 0, 96);
        return 1;
    }
    jf_to_affine(lane[0], out96);
    return 0;
}
