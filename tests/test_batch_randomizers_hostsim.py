"""CPU checks of the seeded batch randomisers: the wide reduction sc_from_u512 (schnorr-sig_b200/csrc/scalar.cuh) against
Python integers on edge values, and the generator batch_randomizer (csrc/derive.cuh, the body of k_batch_randomizers)
against the hashlib oracle of tests/randomizer_ref.py, both compiled for the host by tests/hostsim/randomizers.cpp.
The GPU runs are in tests/test_gpu_seeded_batch.py."""
import ctypes as C
import hashlib
import os
import random
import subprocess

import numpy as np
import pytest

from pyref import Q
from randomizer_ref import TAG, batch_randomizer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hs():
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_randomizers.so")
    src = os.path.join(d, "randomizers.cpp")
    csrc = os.path.join(ROOT, "schnorr-sig_b200", "csrc")
    deps = [src, os.path.join(d, "hostsim.cpp")]
    deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    deps += [os.path.join(ROOT, "include", f) for f in ("cheetah_params.h", "fp_sqrt_tables.h")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", so, src])
    lib = C.CDLL(so)
    lib.hs_sc_from_u512.argtypes = [C.c_char_p, C.c_char_p]
    lib.hs_batch_randomizers.argtypes = [C.c_size_t, C.c_char_p, C.c_uint64, C.c_char_p]
    return lib


def from_u512(hs, v):
    out = C.create_string_buffer(32)
    hs.hs_sc_from_u512(v.to_bytes(64, "little"), out)
    return int.from_bytes(out.raw, "little")


def edge_values():
    k_big = [2**256 // Q, (2**512 - 1) // Q, (2**511) // Q, 2**255 + 12345, 3**300]
    vals = [0, 1, Q - 1, Q, Q + 1, 2 * Q, 3 * Q - 1, 2**255, 2**256 - 1, 2**256, 2**256 + 1, 2**512 - 1, 2**511]
    for k in k_big:
        vals += [k * Q - 1, k * Q, k * Q + 1]
    # high half at and above q (sc_montmul needs it reduced first), with low halves at their edges
    for hi in (Q - 1, Q, Q + 1, 2 * Q, 2**256 - 1):
        for lo in (0, Q - 1, Q, 2**256 - 1):
            vals.append(hi * 2**256 + lo)
    return [v for v in vals if 0 <= v < 2**512]


def test_sc_from_u512_edges(hs):
    for v in edge_values():
        assert from_u512(hs, v) == v % Q, hex(v)


def test_sc_from_u512_random(hs):
    r = random.Random(20261022)
    for _ in range(3000):
        bits = r.choice((512, 511, 384, 257, 256, 255, 64))
        v = r.getrandbits(bits)
        assert from_u512(hs, v) == v % Q, hex(v)


def test_oracle_is_hashlib_over_the_tagged_input():
    seed = bytes(range(32))
    msg = TAG + seed + (7).to_bytes(8, "little")
    assert len(msg) == 76            # one SHA-512 compression
    want = int.from_bytes(hashlib.sha512(msg).digest(), "little") % Q
    assert batch_randomizer(seed, 7) == want.to_bytes(32, "little")


@pytest.mark.parametrize("first", [0, 1, 12345, 2**32 - 3, 2**63, 2**64 - 64])
def test_generator_matches_the_oracle(hs, first):
    rng = np.random.default_rng(first % 1000003)
    for seed in (bytes(32), b"\xff" * 32, rng.integers(0, 256, 32, dtype=np.uint8).tobytes()):
        n = 64
        out = C.create_string_buffer(32 * n)
        hs.hs_batch_randomizers(n, seed, first, out)
        for k in range(n):
            got = out.raw[32 * k:32 * k + 32]
            assert got == batch_randomizer(seed, first + k), (first, k)
            assert int.from_bytes(got, "little") < Q


def test_generator_depends_on_every_seed_byte_and_the_index(hs):
    seed = bytes(range(100, 132))
    base = batch_randomizer(seed, 5)
    for j in range(32):
        s = bytearray(seed)
        s[j] ^= 1
        out = C.create_string_buffer(32)
        hs.hs_batch_randomizers(1, bytes(s), 5, out)
        assert out.raw != base and out.raw == batch_randomizer(bytes(s), 5)
    assert batch_randomizer(seed, 5) != batch_randomizer(seed, 5 + 2**32)
