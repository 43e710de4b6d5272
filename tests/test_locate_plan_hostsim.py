"""CPU model check of the failed-batch localisation tree and its ownership over devices (schnorr-sig_b200/csrc/locate_plan.h,
scheduled as csrc/locate.cuh schedules it), compiled for the host by tests/hostsim/locate_plan.cpp.

Item i carries an integer term; a range fails iff the sum of its terms is not 0, so two items of opposite terms cancel
when they share a range, as two torsion-shifted items do in the batch equation.  For every n and every device count
the flags, the parts of each level and the level at which the cap sends everything to the item check must be those of
one device; every part must be checked exactly once, by a device whose owned range holds it.  The GPU runs of the same
rule are in tests/test_gpu_locate_multi.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(ROOT)
LEAF, FANOUT, MAX_PARTS, MIN_PER_DEVICE = 4096, 8, 8 * 64, 4096
# 2^22: the smallest power of two whose fifth level has more than 8 * 64 parts, where the cap can engage
SIZES = [4096, 4097, 8 * 4096 + 1, 1 << 17, 1 << 20, 1 << 22]
DEVICES = range(1, 10)


@pytest.fixture(scope="module")
def hs():
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_locate_plan.so")
    src = os.path.join(d, "locate_plan.cpp")
    deps = [src, os.path.join(ROOT, "schnorr-sig_b200", "csrc", "locate_plan.h")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", so, src])
    lib = C.CDLL(so)
    lib.hs_locate.restype = C.c_int
    lib.hs_locate.argtypes = [C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p,
                              C.POINTER(C.c_size_t), C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    return lib


def run(hs, term, devices):
    n = len(term)
    term = np.ascontiguousarray(term, dtype=np.int64)
    flags = np.zeros(n, dtype=np.uint8)
    owned = np.zeros(16, dtype=np.uint64)
    n_owned = C.c_size_t(0)
    cap = 1 << 16
    log = np.zeros((cap, 5), dtype=np.uint64)
    log_len = C.c_size_t(0)
    rc = hs.hs_locate(n, term.ctypes.data, devices, MIN_PER_DEVICE, flags.ctypes.data, owned.ctypes.data,
                      C.byref(n_owned), log.ctypes.data, cap, C.byref(log_len))
    assert rc == 0, rc
    owned = [(int(owned[2 * k]), int(owned[2 * k + 1])) for k in range(n_owned.value)]
    log = [tuple(int(v) for v in e[:3]) + (int(np.int64(np.uint64(e[3]))), int(e[4])) for e in log[:log_len.value]]
    return flags, owned, log


def reference_tree(term):
    """The tree written out from its definition: (checked levels, leaves, level of the cap or None)."""
    n = len(term)
    pre = np.concatenate([[0], np.cumsum(np.asarray(term, dtype=np.int64))])
    levels, leaves, capped = [], [], None
    suspects, first = [(0, n)], True
    while suspects:
        parts = []
        for lo, hi in suspects:
            if hi - lo <= LEAF:
                leaves.append((lo, hi))
                continue
            f = 1 if first else FANOUT
            step = -(-(hi - lo) // f)
            parts += [(a, min(a + step, hi)) for a in range(lo, hi, step)]
        first = False
        if len(parts) > MAX_PARTS:
            leaves += parts
            capped = len(levels) + 1
            break
        if not parts:
            break
        levels.append(parts)
        suspects = [(lo, hi) for lo, hi in parts if pre[hi] != pre[lo]]
    return levels, leaves, capped


def workloads(n):
    """Named term vectors of n items: clean, culprits, the cap path and cancelling pairs."""
    rng = np.random.default_rng(n)
    out = {"clean": np.zeros(n, dtype=np.int64)}
    t = np.zeros(n, dtype=np.int64)
    t[n // 3] = 5
    out["one"] = t
    t = np.zeros(n, dtype=np.int64)
    t[rng.choice(n, size=min(16, n), replace=False)] = rng.integers(1, 1000, size=min(16, n))
    out["sixteen"] = t
    t = np.zeros(n, dtype=np.int64)
    t[::40] = 7
    out["one_in_40"] = t
    # a cancelling pair inside one level-2 part (and inside one leaf), next to a real culprit elsewhere
    step = -(-n // FANOUT)
    t = np.zeros(n, dtype=np.int64)
    t[10], t[20] = 3, -3
    t[n - 1] = 1
    out["pair_inside"] = t
    # a cancelling pair across the boundary of the first two level-2 parts (an ownership boundary whenever two or
    # more devices run), next to a real culprit: the two parts fail on their own and both items are flagged
    if n > LEAF:
        t = np.zeros(n, dtype=np.int64)
        t[step - 1], t[step] = 4, -4
        t[n - 1] = 1
        out["pair_across"] = t
        # the same pair with nothing else wrong leaves a batch whose whole check passes: no flag at all
        t = np.zeros(n, dtype=np.int64)
        t[step - 1], t[step] = 4, -4
        t[0], t[n - 1] = 9, -9
        out["pairs_cancel_whole"] = t
    return out


def expected_owned(n, devices):
    d = min(devices, FANOUT, max(1, n // MIN_PER_DEVICE))
    if n <= LEAF:
        d = 1
    if d == 1:
        return [(0, n)]
    step = -(-n // FANOUT)
    l2 = [(a, min(a + step, n)) for a in range(0, n, step)]
    p = len(l2)
    return [(l2[j * p // d][0], l2[(j + 1) * p // d - 1][1]) for j in range(d)]


@pytest.mark.parametrize("n", SIZES)
def test_flags_and_tree_do_not_depend_on_the_device_count(hs, n):
    for name, term in workloads(n).items():
        levels, leaves, capped = reference_tree(term)
        want_flags = np.where(term != 0, 2, 0).astype(np.uint8)
        leaf_mask = np.zeros(n, dtype=bool)
        for lo, hi in leaves:
            leaf_mask[lo:hi] = True
        want_flags[~leaf_mask] = 0
        base = None
        for d in DEVICES:
            flags, owned, log = run(hs, term, d)
            ctx = (name, n, d)
            assert np.array_equal(flags, want_flags), ctx
            assert owned == expected_owned(n, d), ctx
            # every part of every level, exactly once, in tree order; the whole batch over several devices is one
            # partial per owned range
            parts = [e for e in log if e[4] == 0]
            partials = [e for e in log if e[4] == 1]
            if len(owned) > 1 and levels:
                assert [(e[1], e[2]) for e in partials] == owned, ctx
                assert all(e[0] == 1 for e in partials), ctx
                got_levels = [[(0, n)]]
            else:
                assert partials == [], ctx
                got_levels = []
            for e in parts:
                while len(got_levels) < e[0]:
                    got_levels.append([])
                got_levels[e[0] - 1].append((e[1], e[2]))
            assert got_levels == levels, ctx
            # the cap engages at the same level: the item check runs after the same number of levels, on the same ranges
            leaf_log = [e for e in log if e[4] == 2]
            assert sorted((e[1], e[2]) for e in leaf_log) == sorted(leaves), ctx
            assert all(e[0] == len(levels) for e in leaf_log), ctx
            if capped is not None:
                assert capped == len(levels) + 1, ctx
            # each device only touches its owned range
            for e in log:
                lo, hi = owned[e[3]]
                assert lo <= e[1] < e[2] <= hi, (ctx, e)
            # the same work as on one device, once the partials of the whole check stand for the whole batch
            work = [(e[0], e[1], e[2], e[4]) for e in log if e[4] != 1]
            key = (flags.tobytes(), ([(1, 0, n, 0)] if partials else []) + work)
            if base is None:
                base = key
            assert key == base, ctx


def test_workloads_reach_every_path(hs):
    """The cases keep their purpose: 1 in 40 sends every item to the item check (through the cap at 2^22, where the
    fifth level has 4096 parts), the clean batch stops after the whole check, and cancelling pairs inside one part stay
    unflagged."""
    for n in SIZES[1:]:
        w = workloads(n)
        levels, leaves, capped = reference_tree(w["one_in_40"])
        assert sum(hi - lo for lo, hi in leaves) == n, n
        assert (capped is not None) == (n == 1 << 22), n
        levels, leaves, capped = reference_tree(w["clean"])
        assert len(levels) == 1 and leaves == [] and capped is None, n
        flags, _, _ = run(hs, w["pair_inside"], 9)
        assert flags[10] == 0 and flags[20] == 0 and flags[n - 1] == 2, n
        flags, _, _ = run(hs, w["pair_across"], 9)
        step = -(-n // FANOUT)
        assert flags[step - 1] == 2 and flags[step] == 2, n
        flags, _, _ = run(hs, w["pairs_cancel_whole"], 9)
        assert not flags.any(), n
    flags, owned, log = run(hs, workloads(4096)["one"], 9)
    assert owned == [(0, 4096)] and [e[4] for e in log] == [2]


@pytest.mark.parametrize("devices", DEVICES)
def test_ownership_rule(hs, devices):
    """Devices used: min(listed, 8, max(1, n / 4096)); owned ranges are contiguous blocks of whole level-2 parts that
    cover the batch."""
    for n in (4097, 8191, 8192, 3 * 4096 + 5, 8 * 4096 + 1, 1 << 17, (1 << 20) + 3):
        _, owned, _ = run(hs, np.zeros(n, dtype=np.int64), devices)
        assert len(owned) == (1 if n <= LEAF else min(devices, FANOUT, max(1, n // MIN_PER_DEVICE))), (n, devices)
        assert owned[0][0] == 0 and owned[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(owned, owned[1:]))
        step = -(-n // FANOUT)
        assert all(lo % step == 0 for lo, _ in owned)
