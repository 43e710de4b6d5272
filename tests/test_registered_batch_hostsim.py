"""CPU checks of the key side of batches against registered key sets (schnorr-sig_b200/csrc/keyset.cuh compiled for the
host by tests/hostsim/registered_batch.cpp) against the oracle: the reduction of the per-key limb-column sums mod q, the
key term c (-P) a warp of k_keyset_batch_term forms from the key's table, and their composition into the lhs of the
batch equation.  The GPU runs are in tests/test_gpu_registered_batch.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import pyref as o
from util import pt_from96, pt_to96

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hostsim():
    """ctypes handle on the host build of registered.cpp + the registered-batch exports (registered_batch.cpp)."""
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_registered_batch.so")
    src = os.path.join(d, "registered_batch.cpp")
    csrc = os.path.join(ROOT, "schnorr-sig_b200", "csrc")
    deps = [src] + [os.path.join(d, f) for f in ("registered.cpp", "hostsim.cpp")]
    deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    deps += [os.path.join(ROOT, "include", f) for f in ("cheetah_params.h", "fp_sqrt_tables.h")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", so, src])
    return C.CDLL(so)


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def le32(k):
    return np.frombuffer(int(k).to_bytes(32, "little"), dtype=np.uint8).copy()


def columns(values):
    """64-bit column sums of the eight 32-bit limbs, as k_keyset_scalar_sum accumulates them."""
    limbs = np.array([[(v >> (32 * j)) & 0xFFFFFFFF for j in range(8)] for v in values], dtype=np.uint64)
    return limbs.sum(axis=0, dtype=np.uint64)


def reduce(hostsim, col):
    col = np.ascontiguousarray(col, dtype=np.uint64)
    out = np.zeros(32, dtype=np.uint8)
    hostsim.hs_keyset_sum_reduce(p(col), p(out))
    return int.from_bytes(out.tobytes(), "little")


def geometry(hostsim):
    w, win, ent = C.c_int(0), C.c_int(0), C.c_int(0)
    hostsim.hs_kt_geometry(C.byref(w), C.byref(win), C.byref(ent))
    return w.value, win.value, ent.value


def key_table(hostsim, P):
    w, windows, entries = geometry(hostsim)
    out = np.zeros((windows, entries, 12), dtype=np.uint64)
    hostsim.hs_tab_build(p(pt_to96(P)), w, windows, p(out))
    return out


def key_term(hostsim, tab, c):
    out = np.zeros(96, dtype=np.uint8)
    inf = hostsim.hs_keyset_key_term(p(tab), p(le32(c)), p(out))
    return o.INF if inf else pt_from96(out)


def test_sum_reduce_small_sums(hostsim):
    q = o.Q
    rng = np.random.default_rng(61)
    cases = [[q - 1], [q - 1, q - 2], [q - 1, 1], [q - 1, q - 1, 2], [0], [q - 1] * 3]
    cases += [[int.from_bytes(rng.bytes(32), "little") % q for _ in range(k)] for k in (1, 2, 5, 100)]
    for vals in cases:
        assert reduce(hostsim, columns(vals)) == sum(vals) % q, vals


def test_sum_reduce_exact_multiples_of_q(hostsim):
    q = o.Q
    for vals in ([q - 1, 1], [q - 5, 2, 3], [(q - 1) // 2, (q + 1) // 2], [q - 1] * 5 + [5]):
        assert sum(vals) % q == 0
        assert reduce(hostsim, columns(vals)) == 0, vals


def test_sum_reduce_2_20_values_near_q(hostsim):
    q = o.Q
    n = 1 << 20
    d = np.arange(n, dtype=np.uint64) % 7 + 1                  # values q - 1 ... q - 7
    q_limbs = np.array([(q >> (32 * j)) & 0xFFFFFFFF for j in range(8)], dtype=np.uint64)
    # limb 0 of q is far above 7: subtracting d borrows from no other limb
    assert int(q_limbs[0]) > 7
    col = q_limbs * np.uint64(n)
    col[0] -= np.uint64(int(d.sum()))
    total = n * q - int(d.sum())
    assert sum(int(c) << (32 * j) for j, c in enumerate(col)) == total
    assert reduce(hostsim, col) == total % q


def test_sum_reduce_all_ones_columns_at_the_bound(hostsim):
    """2^32 - 1 items whose limbs are all 2^32 - 1 (not reduced values: the largest columns the arithmetic admits)."""
    m = (1 << 32) - 1
    col = np.full(8, m * m, dtype=np.uint64)
    total = sum((m * m) << (32 * j) for j in range(8))
    assert reduce(hostsim, col) == total % o.Q
    col = np.zeros(8, dtype=np.uint64)
    col[7] = m * m                                             # everything in the top column: the largest carry out
    assert reduce(hostsim, col) == ((m * m) << 224) % o.Q


def test_key_term_matches_the_oracle(hostsim):
    w, windows, _ = geometry(hostsim)
    rng = np.random.default_rng(62)
    G = o.generator()
    P = o.pt_mul(G, 0x5eed1234)
    tab = key_table(hostsim, P)
    q = o.Q
    half = 1 << (w - 1)
    cs = [0, 1, 2, half, half + 1, q - 1, q - 2]
    for i in (1, 2, 15, 16, windows - 1):
        b = 1 << (w * i)
        cs += [v % q for v in (b, b - 1, half * b, (half + 1) * b - 1)]
    cs += [sum(half + 1 << (w * i) for i in range(windows - 1)) % q]     # a carry across every boundary
    cs += [int.from_bytes(rng.bytes(32), "little") % q for _ in range(6)]
    for c in cs:
        assert 0 <= c < q
        want = o.pt_mul(P, (q - c) % q)
        assert key_term(hostsim, tab, c) == want, c


def test_batch_lhs_from_key_terms(hostsim):
    """sum s_i R_i (oracle) + sum_k c_k (-P_k) (host build of the key side) == the lhs of the oracle's verify_batch."""
    q = o.Q
    rng = np.random.default_rng(63)
    G = o.generator()
    sks = [int.from_bytes(rng.bytes(32), "little") % q for _ in range(3)]
    keys = [o.pt_mul(G, k) for k in sks]
    idx = [0, 1, 0, 2, 2, 2, 0]
    msgs = [bytes(rng.integers(0, 256, L, dtype=np.uint8)) for L in (8, 0, 7, 14, 8, 3, 21)]
    sigs = [o.sign(sks[k], keys[k], m, int.from_bytes(rng.bytes(32), "little") % q) for k, m in zip(idx, msgs)]
    rand = [int.from_bytes(rng.bytes(32), "little") % q for _ in idx]
    rand[4] = 0                                                      # a zero randomiser contributes nothing
    verdict, lhs, _rhs = o.verify_batch(sigs, [keys[k] for k in idx], msgs, rand)
    assert verdict == o.OK
    acc = o.INF
    t = {k: [] for k in range(len(keys))}
    for (x49, _e), k, m, s in zip(sigs, idx, msgs, rand):
        ok, R = o.decompress(x49)
        assert ok
        acc = o.pt_add(acc, o.pt_mul(R, s))
        h = o.scalar_from_digest(o.hash_message(R[0], keys[k], m))
        t[k].append(h * s % q)
    for k, P in enumerate(keys):
        c = reduce(hostsim, columns(t[k]))
        assert c == sum(t[k]) % q
        acc = o.pt_add(acc, key_term(hostsim, key_table(hostsim, P), c))
    assert acc == lhs
