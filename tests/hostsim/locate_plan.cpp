// TEST-ONLY host build of the localisation tree and its ownership rule (schnorr-sig_b200/csrc/locate_plan.h) with g++,
// for tests/test_locate_plan_hostsim.py.  hs_locate runs locate_bisect the way locate_run (csrc/locate.cuh) schedules
// it over devices, with a model in place of the partial MSMs: item i has an integer term, a range fails iff the sum of
// its terms is not 0, and the per-item check flags an item iff its own term is not 0.  Not part of the product.
#include <cstdint>
#include <vector>

#include "../../schnorr-sig_b200/csrc/locate_plan.h"

#define API extern "C" __attribute__((visibility("default")))

// n items with terms term[0..n) on `count` listed devices (min_per_device: MULTI_MIN_PER_SHARD).  Writes flags[n], the
// owned ranges (owned[2k], owned[2k+1]; *n_owned of them) and one log entry of five words per piece of work:
//   (level, lo, hi, device, kind)   kind 0: a part checked by its owner, 1: the partial of an owned range for the
//                                   whole-batch check over several devices, 2: a leaf range through the item check
// The level of a leaf is the number of checked levels when the item check ran.  Returns 0, -1 when a part or a leaf
// has no owner, -2 when the log is full.
API int hs_locate(size_t n, const int64_t* term, size_t count, size_t min_per_device, uint8_t* flags, uint64_t* owned_out,
                  size_t* n_owned, uint64_t* log, size_t log_cap, size_t* log_len) {
    std::vector<int64_t> pre(n + 1, 0);
    for (size_t i = 0; i < n; i++) pre[i + 1] = pre[i] + term[i];
    auto sum = [&](const locate_range& r) { return pre[r.hi] - pre[r.lo]; };
    std::vector<locate_range> owned = locate_owned(n, locate_devices(count, n, min_per_device));
    *n_owned = owned.size();
    for (size_t k = 0; k < owned.size(); k++) {
        owned_out[2 * k] = owned[k].lo;
        owned_out[2 * k + 1] = owned[k].hi;
    }
    *log_len = 0;
    uint64_t level = 0;
    auto put = [&](const locate_range& r, int dev, int kind) {
        if (*log_len == log_cap) return false;
        uint64_t* e = log + 5 * (*log_len)++;
        e[0] = level;
        e[1] = r.lo;
        e[2] = r.hi;
        e[3] = (uint64_t)(int64_t)dev;
        e[4] = (uint64_t)kind;
        return true;
    };
    for (size_t i = 0; i < n; i++) flags[i] = 0;
    auto check = [&](const std::vector<locate_range>& parts, uint8_t* ok) -> int {
        level++;
        if (locate_owner(owned, parts[0]) < 0) {   // the whole batch over several devices: one partial each
            int64_t s = 0;
            for (size_t k = 0; k < owned.size(); k++) {
                if (!put(owned[k], (int)k, 1)) return -2;
                s += sum(owned[k]);
            }
            ok[0] = s == 0;
            return 0;
        }
        for (size_t j = 0; j < parts.size(); j++) {
            int k = locate_owner(owned, parts[j]);
            if (k < 0) return -1;
            if (!put(parts[j], k, 0)) return -2;
            ok[j] = sum(parts[j]) == 0;
        }
        return 0;
    };
    auto items = [&](const std::vector<locate_range>& leaves) -> int {
        for (const locate_range& r : leaves) {
            int k = locate_owner(owned, r);
            if (k < 0) return -1;
            if (!put(r, k, 2)) return -2;
            for (size_t i = r.lo; i < r.hi; i++) flags[i] = term[i] != 0 ? 2 : 0;
        }
        return 0;
    };
    return locate_bisect(n, check, items);
}
