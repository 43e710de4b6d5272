// TEST-ONLY host build of the batch randomiser generator (batch_randomizer in schnorr-sig_b200/csrc/derive.cuh, the
// body of k_batch_randomizers) and its wide reduction (sc_from_u512 in scalar.cuh) with g++, for
// tests/test_batch_randomizers_hostsim.py.  It extends the host build of the device headers (hostsim.cpp, included
// whole) with the exports below; like it, it is not part of the product.
#include "hostsim.cpp"

// sc_from_u512 of the 64-byte little-endian integer in512 -> out32 (canonical LE)
API void hs_sc_from_u512(const uint8_t* in512, uint8_t* out32) {
    stsc(out32, sc_from_u512(sc_load_le(in512), sc_load_le(in512 + 32)));
}
// randomisers first ... first + n - 1 of seed32 -> out32 (n x 32 B), as k_batch_randomizers writes them
API void hs_batch_randomizers(size_t n, const uint8_t* seed32, uint64_t first, uint8_t* out32) {
    for (size_t i = 0; i < n; i++) stsc(out32 + 32 * i, batch_randomizer(seed32, first + i));
}
