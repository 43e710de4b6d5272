// The tree of failed-batch localisation and the ownership of its nodes by devices: host code only, no CUDA (the CPU
// suite compiles it, tests/hostsim/locate_plan.cpp).  locate.cuh runs it on one device or over the devices of a
// multi-device context.
//
// The tree is defined by n alone: the whole batch is checked first; a failing range is cut into LOCATE_FANOUT parts of
// ceil(len / LOCATE_FANOUT), each checked by its own partial MSM; ranges of at most LOCATE_LEAF items go to the
// per-item check, and so does every part of a level that has more than LOCATE_MAX_PARTS of them (a batch riddled with
// bad signatures).  Which device checks a part changes no verdict, so the flags do not depend on the device count.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

static constexpr size_t LOCATE_LEAF = 4096;
static constexpr int LOCATE_FANOUT = 8;
static constexpr size_t LOCATE_MAX_PARTS = (size_t)LOCATE_FANOUT * 64;
struct locate_range {
    size_t lo, hi;
};

// The parts of the next level: every suspect range longer than LOCATE_LEAF cut into LOCATE_FANOUT parts (on the first
// level the whole batch is checked as it is, one part); shorter suspects are appended to `leaves`.
static std::vector<locate_range> locate_next_level(const std::vector<locate_range>& suspects, bool first,
                                                   std::vector<locate_range>& leaves) {
    std::vector<locate_range> parts;
    for (const locate_range& r : suspects) {
        size_t len = r.hi - r.lo;
        if (len <= LOCATE_LEAF) {
            leaves.push_back(r);
            continue;
        }
        size_t f = first ? 1 : LOCATE_FANOUT;
        size_t step = (len + f - 1) / f;
        for (size_t lo = r.lo; lo < r.hi; lo += step) parts.push_back({lo, lo + step < r.hi ? lo + step : r.hi});
    }
    return parts;
}

// The bisection of n > 0 items.  check(parts, ok) checks one level and sets ok[k] = 1 for every part whose own batch
// verifies (a non-zero return is an error code); items(leaves) checks what is left item by item.
template <typename Check, typename Items>
static int locate_bisect(size_t n, Check check, Items items) {
    std::vector<locate_range> suspects{{0, n}}, leaves;
    bool first = true;
    while (!suspects.empty()) {
        std::vector<locate_range> parts = locate_next_level(suspects, first, leaves);
        first = false;
        suspects.clear();
        if (parts.size() > LOCATE_MAX_PARTS) {   // the suspects stopped shrinking: finish item by item
            leaves.insert(leaves.end(), parts.begin(), parts.end());
            break;
        }
        if (parts.empty()) break;
        std::vector<uint8_t> ok(parts.size(), 0);
        if (int rc = check(parts, ok.data())) return rc;
        for (size_t k = 0; k < parts.size(); k++)
            if (!ok[k]) suspects.push_back(parts[k]);   // Err or malformed: look inside
    }
    return items(leaves);
}

// Devices that localise n items on a context of `count`: min(count, LOCATE_FANOUT, max(1, n / min_per_device)), and one
// when the whole batch is a leaf.
static size_t locate_devices(size_t count, size_t n, size_t min_per_device) {
    size_t d = n / min_per_device;
    if (d < 1 || n <= LOCATE_LEAF) d = 1;
    if (d > (size_t)LOCATE_FANOUT) d = LOCATE_FANOUT;
    return d < count ? d : count;
}

// The range each of d devices owns: the parts of level 2 (the whole batch cut into LOCATE_FANOUT) in contiguous
// blocks, device j the parts [j P / d, (j + 1) P / d).  A device owns every descendant of its parts, so it checks every
// node of the tree below level 1 that lies in its range, and the first level over several devices is one partial each.
static std::vector<locate_range> locate_owned(size_t n, size_t d) {
    if (d <= 1) return {{0, n}};
    std::vector<locate_range> leaves;
    std::vector<locate_range> l2 = locate_next_level(locate_next_level({{0, n}}, true, leaves), false, leaves);
    size_t p = l2.size();
    if (d > p) d = p;
    std::vector<locate_range> owned;
    for (size_t j = 0; j < d; j++) owned.push_back({l2[j * p / d].lo, l2[(j + 1) * p / d - 1].hi});
    return owned;
}

// The device whose owned range holds r, or -1 when r spans several (the whole batch, on more than one device).
static int locate_owner(const std::vector<locate_range>& owned, const locate_range& r) {
    for (size_t k = 0; k < owned.size(); k++)
        if (owned[k].lo <= r.lo && r.hi <= owned[k].hi) return (int)k;
    return -1;
}
