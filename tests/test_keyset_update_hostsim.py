"""CPU checks of the lookup-table maintenance of in-place key-set updates (keyset_update_entries in
schnorr-sig_b200/csrc/keyset.cuh, compiled for the host by tests/hostsim/keyset_update.cpp): after every step of random
append / replace / remove sequences, the incrementally maintained table equals the one keyset_sort_entries builds from
scratch over the findable slots -- entries, count and the smallest index of every encoding.  The GPU runs are in
tests/test_gpu_keyset_update.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRY = np.dtype([("x", "<u8", (6,)), ("flag", "<u4"), ("index", "<u4"), ("pad", "<u8")])
assert ENTRY.itemsize == 64


@pytest.fixture(scope="module")
def hostsim():
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_keyset_update.so")
    src = os.path.join(d, "keyset_update.cpp")
    csrc = os.path.join(ROOT, "schnorr-sig_b200", "csrc")
    deps = [src, os.path.join(d, "hostsim.cpp")]
    deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    deps += [os.path.join(ROOT, "include", f) for f in ("cheetah_params.h", "fp_sqrt_tables.h")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", so, src])
    lib = C.CDLL(so)
    lib.hs_keyset_update_entries.restype = C.c_size_t
    lib.hs_keyset_sort_entries.restype = C.c_size_t
    return lib


def p(a):
    return a.ctypes.data_as(C.c_void_p)


class Model:
    """A key set's slots as the lookup sees them: an encoding (x limbs, flag) and whether the slot is findable."""

    def __init__(self, hostsim, rng, pool):
        self.h, self.rng, self.pool = hostsim, rng, pool
        self.enc, self.findable = [], []
        self.all = np.zeros(0, dtype=ENTRY)

    def draw(self):
        r = self.rng.random()
        return int(self.rng.integers(len(self.pool))), bool(r < 0.7)   # 30 %: not findable (status 3, off-curve, ...)

    def entry(self, slot):
        e = np.zeros(1, dtype=ENTRY)
        x, flag = self.pool[self.enc[slot]]
        e["x"][0], e["flag"][0], e["index"][0] = x, flag, slot
        return e

    def update(self, slots):
        """slots: the changed (or appended) slots, whose enc / findable are already set."""
        n_slots = len(self.enc)
        changed = np.zeros(n_slots, dtype=np.uint8)
        changed[slots] = 1
        added = np.concatenate([self.entry(k) for k in slots if self.findable[k]] or [np.zeros(0, dtype=ENTRY)])
        cap = len(self.all) + len(added)
        all_io = np.zeros(max(cap, 1), dtype=ENTRY)
        all_io[:len(self.all)] = self.all
        lut = np.zeros(max(cap, 1), dtype=ENTRY)
        n_all = C.c_size_t(0)
        m = self.h.hs_keyset_update_entries(len(self.all), p(all_io), p(changed), n_slots, len(added), p(added), p(lut),
                                            C.byref(n_all))
        self.all = all_io[:n_all.value].copy()
        return lut[:m]

    def from_scratch(self):
        ents = [self.entry(k) for k in range(len(self.enc)) if self.findable[k]]
        e = np.concatenate(ents) if ents else np.zeros(1, dtype=ENTRY)
        m = self.h.hs_keyset_sort_entries(len(ents), p(e))
        return e[:m]

    def check(self, lut):
        want = self.from_scratch()
        assert lut.tobytes() == want.tobytes()
        first = {}                                    # smallest findable index per encoding
        for k in range(len(self.enc)):
            if self.findable[k]:
                first.setdefault(self.enc[k], k)
        assert len(lut) == len(first)
        assert sorted(int(i) for i in lut["index"]) == sorted(first.values())
        assert len(self.all) == sum(self.findable)    # every findable slot, duplicates included


def encoding_pool(rng, n):
    """n distinct encodings that share limbs in every position, so the order is decided by each limb and the flag."""
    pool = set()
    while len(pool) < n:
        x = tuple(int(v) for v in rng.integers(0, 3, 6, dtype=np.uint64))
        pool.add((x, int(rng.choice([0, 0x40, 0x80]))))
    return sorted(pool)


@pytest.mark.parametrize("seed", range(6))
def test_incremental_table_equals_a_fresh_sort(hostsim, seed):
    rng = np.random.default_rng(1000 + seed)
    steps = 0
    for seq in range(60):
        model = Model(hostsim, rng, encoding_pool(rng, int(rng.choice([1, 3, 8, 40]))))
        n0 = int(rng.choice([1, 7, 30]))
        for _ in range(n0):
            e, f = model.draw()
            model.enc.append(e)
            model.findable.append(f)
        model.check(model.update(list(range(n0))))
        for _ in range(12):
            kind = rng.integers(3)
            n = len(model.enc)
            if kind == 0:                                                   # append 1..5 keys
                m = int(rng.integers(1, 6))
                for _ in range(m):
                    e, f = model.draw()
                    model.enc.append(e)
                    model.findable.append(f)
                slots = list(range(n, n + m))
            elif kind == 1:                                                 # replace distinct slots
                slots = sorted(set(int(k) for k in rng.integers(0, n, int(rng.integers(1, 5)))))
                for k in slots:
                    model.enc[k], model.findable[k] = model.draw()
            else:                                                           # remove: never findable again
                slots = sorted(set(int(k) for k in rng.integers(0, n, int(rng.integers(1, 4)))))
                for k in slots:
                    model.findable[k] = False
            model.check(model.update(slots))
            steps += 1
    assert steps == 60 * 12


def test_replacing_the_lowest_copy_exposes_the_next(hostsim):
    rng = np.random.default_rng(5)
    model = Model(hostsim, rng, encoding_pool(rng, 2))
    model.enc, model.findable = [0, 0, 0, 1], [True, True, True, True]
    lut = model.update([0, 1, 2, 3])
    assert sorted(int(i) for i in lut["index"]) == [0, 3]
    model.enc[0] = 1                                                       # slot 0 now holds the other encoding
    lut = model.update([0])
    model.check(lut)
    assert sorted(int(i) for i in lut["index"]) == [0, 1]
    model.findable[1] = False                                              # removing slot 1 exposes slot 2
    lut = model.update([1])
    model.check(lut)
    assert sorted(int(i) for i in lut["index"]) == [0, 2]
