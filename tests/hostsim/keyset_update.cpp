// TEST-ONLY host build of the lookup-table maintenance of in-place key-set updates (keyset_update_entries in
// schnorr-sig_b200/csrc/keyset.cuh) with g++, for tests/test_keyset_update_hostsim.py.  It extends the host build of
// the device headers (hostsim.cpp, included whole) with the exports below; like it, it is not part of the product.
#include "hostsim.cpp"
#include "../../schnorr-sig_b200/csrc/keyset.cuh"

// keyset_update_entries on a list of n_all sorted entries (all, updated in place: room for n_all + n_added entries;
// *n_all_out = its new length), the changed-slot mask of n_slots bytes and n_added new entries; lut: room for
// n_all + n_added entries.  Returns the number of lookup entries.
API size_t hs_keyset_update_entries(size_t n_all, keyset_entry* all, const uint8_t* changed, size_t n_slots, size_t n_added,
                                    const keyset_entry* added, keyset_entry* lut, size_t* n_all_out) {
    std::vector<keyset_entry> a(all, all + n_all), add(added, added + n_added), l;
    keyset_update_entries(a, changed, n_slots, std::move(add), l);
    std::copy(a.begin(), a.end(), all);
    *n_all_out = a.size();
    std::copy(l.begin(), l.end(), lut);
    return l.size();
}
// keyset_sort_entries: the table registration builds from scratch over n findable entries (any order)
API size_t hs_keyset_sort_entries(size_t n, keyset_entry* entries) { return keyset_sort_entries(entries, n); }
