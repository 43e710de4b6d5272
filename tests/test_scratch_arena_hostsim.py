"""CPU checks of the scratch arena of a single-device context (schnorr-sig_b200/csrc/scratch.cuh), built with g++ against
a stand-in cuda_runtime.h that records every cudaMalloc, cudaFree and cudaStreamSynchronize
(tests/hostsim/scratch_arena.cpp): live regions are 256-byte aligned and never overlap, closing a scope releases
exactly its regions, requests that do not fit take overflow blocks without moving anything, closing the outermost scope
of a call that grew the arena synchronises before it frees and leaves one block of at least the peak on the arena's
device, and repeated calls of one shape make no allocator or synchronisation call at all."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALIGN = 256
EV_MALLOC, EV_FREE, EV_SYNC = 1, 2, 3


@pytest.fixture(scope="module")
def lib():
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_scratch_arena.so")
    src = os.path.join(d, "scratch_arena.cpp")
    deps = [src, os.path.join(d, "stub", "cuda_runtime.h"), os.path.join(ROOT, "schnorr-sig_b200", "csrc", "scratch.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
                               "-I", os.path.join(d, "stub"), "-o", so, src])
    h = C.CDLL(so)
    h.hs_take.argtypes = [C.c_uint64, C.POINTER(C.c_uint64)]
    h.hs_log_size.restype = C.c_uint64
    return h


def padded(n):
    return max(ALIGN, (n + ALIGN - 1) // ALIGN * ALIGN)


class Arena:
    """Drives the arena and checks every region against the blocks the log says are allocated and the live regions."""

    def __init__(self, lib):
        self.h = lib
        self.h.hs_reset()
        self.scopes = []      # regions (address, padded size) taken in each open scope
        self.blocks = {}      # address -> size of every allocated block
        self.seen = 0         # log events already applied

    def log(self):
        n = self.h.hs_log_size()
        a = np.zeros(4 * max(n, 1), dtype=np.uint64)
        self.h.hs_log(a.ctypes.data_as(C.c_void_p))
        return [tuple(int(v) for v in a[4 * i:4 * i + 3]) for i in range(n)]

    def devices(self):
        """the current device of every logged call"""
        n = self.h.hs_log_size()
        a = np.zeros(4 * max(n, 1), dtype=np.uint64)
        self.h.hs_log(a.ctypes.data_as(C.c_void_p))
        return [int(a[4 * i + 3]) for i in range(n)]

    def apply_log(self):
        ev = self.log()
        new = ev[self.seen:]
        self.seen = len(ev)
        for kind, ptr, size in new:
            if kind == EV_MALLOC:
                self.blocks[ptr] = size
            elif kind == EV_FREE:
                assert not self.scopes, "a block freed under an open scope"
                del self.blocks[ptr]
        return new

    def open(self):
        self.h.hs_open()
        self.scopes.append([])
        assert self.apply_log() == []

    def close(self):
        """-> the logged calls: none but for the outermost scope of a call that grew the arena"""
        self.h.hs_close()
        self.scopes.pop()
        new = self.apply_log()
        if new:
            assert not self.scopes
            kinds = [k for k, _, _ in new]
            assert kinds[0] == EV_SYNC and kinds[1:] == [EV_FREE] * (len(kinds) - 2) + [EV_MALLOC] and len(kinds) >= 4
            assert len(self.blocks) == 1
        return new

    def take(self, n):
        out = C.c_uint64(0)
        assert self.h.hs_take(n, C.byref(out)) == 0
        a, size = out.value, padded(n)
        new = self.apply_log()
        assert all(kind == EV_MALLOC for kind, _, _ in new)
        assert a % ALIGN == 0
        assert any(b <= a and a + size <= b + s for b, s in self.blocks.items()), "region outside every block"
        for scope in self.scopes:
            for b, s in scope:
                assert a + size <= b or b + s <= a, "overlapping live regions"
        self.scopes[-1].append((a, size))
        return a

    def live_bytes(self):
        return sum(s for scope in self.scopes for _, s in scope)


def test_regions_are_aligned_and_disjoint_under_random_nesting(lib):
    rng = np.random.default_rng(7)
    ar = Arena(lib)
    peak = 0
    for call in range(300):
        ar.open()
        for _ in range(int(rng.integers(1, 40))):
            op = rng.random()
            if op < 0.55:
                ar.take(int(rng.choice([0, 1, 255, 256, 257, 4000, 1 << 16, int(rng.integers(1, 1 << 20))])))
                peak = max(peak, ar.live_bytes())
            elif op < 0.8 and len(ar.scopes) < 6:
                ar.open()
            elif len(ar.scopes) > 1:
                ar.close()
        while ar.scopes:
            ar.close()
        assert len(ar.blocks) == 1 and list(ar.blocks.values())[0] >= peak   # consolidated at the end of each call
    lib.hs_destroy()
    ar.apply_log()
    assert ar.blocks == {}


def test_closing_a_scope_releases_exactly_its_regions(lib):
    ar = Arena(lib)
    ar.open()
    ar.take(1 << 20)   # one block large enough for what follows
    ar.close()
    n = len(ar.log())
    ar.open()
    a = ar.take(1000)
    ar.open()
    b = ar.take(3000)
    ar.open()
    c = ar.take(100)
    ar.close()
    assert ar.take(100) == c           # the innermost scope's region is free again
    ar.close()
    assert ar.take(3000) == b          # and so are both of the middle scope's, but not the outer one's
    assert b == a + padded(1000)
    ar.close()
    ar.open()
    assert ar.take(1000) == a
    ar.close()
    assert len(ar.log()) == n


def test_overflow_blocks_then_one_consolidated_block(lib):
    ar = Arena(lib)
    sizes = [1000, 5000, 10 ** 6, 300]
    ar.open()
    a = ar.take(sizes[0])
    ar.open()
    b = ar.take(sizes[1])              # does not fit what is left of the first block: an overflow block
    ar.open()
    c = ar.take(sizes[2])
    ar.close()
    d = ar.take(sizes[3])              # c is released: its overflow block is taken again, without a cudaMalloc
    ar.close()
    assert [k for k, _, _ in ar.log()] == [EV_MALLOC] * 3   # nothing freed or moved while scopes were open
    assert len({a, b, c}) == 3 and d == c
    lib.hs_set_device(5)               # the outermost scope closes under another device
    new = ar.close()                   # synchronise, free every block, one block of the peak on the arena's device
    lib.hs_set_device(0)
    assert [k for k, _, _ in new] == [EV_SYNC, EV_FREE, EV_FREE, EV_FREE, EV_MALLOC]
    assert ar.devices()[-5:] == [0] * 5
    peak = sum(padded(s) for s in sizes[:3])
    size = list(ar.blocks.values())[0]
    assert size >= peak and size == peak + peak // 8
    ev = ar.log()
    ar.open()
    ar.take(sizes[0])
    ar.open()
    ar.take(sizes[1])
    ar.open()
    ar.take(sizes[2])                  # the same call again fits the one block
    ar.close()
    ar.close()
    ar.close()
    assert ar.log() == ev


def test_steady_state_makes_no_allocator_or_sync_calls(lib):
    rng = np.random.default_rng(11)
    shape = [(int(rng.integers(0, 3)), int(rng.integers(1, 1 << 18))) for _ in range(25)]   # (scope depth, bytes)

    def call(ar):
        ar.open()
        for depth, n in shape:
            while len(ar.scopes) - 1 < depth:
                ar.open()
            while len(ar.scopes) - 1 > depth:
                ar.close()
            ar.take(n)
        while ar.scopes:
            ar.close()

    ar = Arena(lib)
    call(ar)                           # grows the arena, and consolidates it when it ends
    n = len(ar.log())
    for _ in range(5):
        call(ar)
        assert len(ar.log()) == n
    assert len(ar.blocks) == 1


def test_a_failed_allocation_is_reported_and_the_arena_stays_usable(lib):
    ar = Arena(lib)
    ar.open()
    ar.take(1000)
    lib.hs_fail_next_malloc()
    out = C.c_uint64(0)
    assert lib.hs_take(1 << 20, C.byref(out)) != 0   # reported to the caller
    assert ar.apply_log() == []
    ar.take(1 << 20)                   # the same request succeeds once memory is there, beside the live region
    ar.take(1000)
    lib.hs_fail_next_malloc()          # the consolidating cudaMalloc fails: no call fails, no block is left
    lib.hs_close()
    ar.scopes.pop()
    assert [k for k, _, _ in ar.apply_log()] == [EV_SYNC, EV_FREE, EV_FREE, EV_FREE]
    assert ar.blocks == {}
    ar.open()
    ar.take(1000)                      # the next call allocates what it needs
    assert len(ar.blocks) == 1
    ar.close()
