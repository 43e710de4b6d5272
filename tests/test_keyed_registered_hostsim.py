"""CPU checks of the lookup of compressed keys in registered key sets (schnorr-sig_b200/csrc/keyset.cuh compiled for the
host by tests/hostsim/keyed_registered.cpp): the encoding of a registered key against the oracle's compress, the
findable rule (decompressing the encoding gives back the registered record exactly), and the sorted-table binary
search against a dictionary model.  The GPU runs are in tests/test_gpu_keyed_registered.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cref
import pyref as o
from test_gpu_registered import adversarial_keys
from util import pt_from96, pt_to96, rand_scalars

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MISS = 0xFFFFFFFF


@pytest.fixture(scope="module")
def hostsim():
    """ctypes handle on the host build of registered.cpp + the lookup exports (keyed_registered.cpp)."""
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_keyed_registered.so")
    src = os.path.join(d, "keyed_registered.cpp")
    csrc = os.path.join(ROOT, "schnorr-sig_b200", "csrc")
    deps = [src] + [os.path.join(d, f) for f in ("registered.cpp", "hostsim.cpp")]
    deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    deps += [os.path.join(ROOT, "include", f) for f in ("cheetah_params.h", "fp_sqrt_tables.h")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", so, src])
    lib = C.CDLL(so)
    lib.hs_keyset_table.restype = C.c_size_t
    return lib


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def encode(hostsim, pk96, inf=0):
    out = np.zeros(49, dtype=np.uint8)
    findable = hostsim.hs_keyset_encode(p(np.ascontiguousarray(pk96, dtype=np.uint8)), int(inf), p(out))
    return bytes(out), bool(findable)


def table(hostsim, pk, inf):
    pk, inf = np.ascontiguousarray(pk, dtype=np.uint8), np.ascontiguousarray(inf, dtype=np.uint8)
    out = np.zeros((len(pk), 64), dtype=np.uint8)
    m = hostsim.hs_keyset_table(len(pk), p(pk), p(inf), p(out))
    return out[:m].copy(), m


def lookup(hostsim, tab, m, keys):
    keys = np.ascontiguousarray(np.stack([np.frombuffer(k, dtype=np.uint8) for k in keys]), dtype=np.uint8)
    out = np.zeros(len(keys), dtype=np.uint32)
    hostsim.hs_keyset_lookup(p(tab), C.c_uint32(m), len(keys), p(keys), p(out))
    return [int(v) for v in out]


def honest_keys(seed, n):
    pk, inf = cref.keygen(rand_scalars(np.random.default_rng(seed), n), cref.default_threads())
    return pk, inf


def test_encodings_equal_the_oracle(hostsim):
    pk, inf = honest_keys(1, 64)
    pk = np.concatenate([pk, np.zeros((1, 96), np.uint8)])
    inf = np.concatenate([inf, [1]]).astype(np.uint8)
    for k in range(len(pk)):
        enc, findable = encode(hostsim, pk[k], inf[k])
        assert enc == bytes(cref.compress(pk[k], inf[k])), k
        assert findable, k


def test_findable_rule(hostsim):
    apk, ainf, status = adversarial_keys()
    # status 1 (orders 2, 29, 58, 2q, the cofactor, the KAT point): findable; the identity with zero coordinates:
    # findable; a non-canonical limb (status 3): not; an identity with junk coordinates: not
    want = [True] * 6 + [True, False, False]
    for k in range(len(apk)):
        assert encode(hostsim, apk[k], ainf[k])[1] == want[k], (k, status[k])
    assert status[:6] == [1] * 6 and status[7] == 3
    # the point of order 2 has y = 0: its encoding is still decoded back to it
    assert pt_from96(apk[0])[1] == o.F6_ZERO
    G = o.generator()
    g96 = pt_to96(G)
    off_curve = (G[0], ((G[1][0] + 1) % o.P,) + G[1][1:])
    assert not o.on_curve(off_curve)
    assert not encode(hostsim, pt_to96(off_curve))[1]
    junk_identity = encode(hostsim, g96, 1)                   # the identity flag with the coordinates of G
    assert junk_identity[0] == bytes(48) + b"\x80" and not junk_identity[1]
    for k in (0, 5):                                          # a non-canonical y limb, and x limb 0 + p (same value)
        bad_y = g96.copy()
        bad_y[48 + 8 * k:56 + 8 * k] = 0xFF
        assert not encode(hostsim, bad_y)[1]
    S = small_limb_point()
    assert encode(hostsim, pt_to96(S))[1]
    x_plus_p = pt_to96(S)
    x_plus_p[0:8] = np.frombuffer((S[0][0] + o.P).to_bytes(8, "little"), np.uint8)
    assert not encode(hostsim, x_plus_p)[1]
    assert encode(hostsim, g96)[1] and encode(hostsim, pt_to96(o.pt_neg(G)))[1]


def small_limb_point():
    """a point on the curve whose x limb 0 is below 2^32 - 1, so that limb + p still fits in 64 bits"""
    gx = o.generator()[0]
    for c in range(1, 1000):
        ok, pt = o.decompress(o.f6_to_bytes((c,) + gx[1:]) + b"\x00")
        if ok:
            return pt
    raise AssertionError("no decodable x found")


def model(hostsim, pk, inf):
    """encoding -> smallest findable index, from the encode routine alone"""
    d = {}
    for k in range(len(pk)):
        enc, findable = encode(hostsim, pk[k], inf[k])
        if findable and enc not in d:
            d[enc] = k
    return d


def variants(enc):
    """49-byte strings next to a registered encoding that must be looked up on their own bytes"""
    out = [enc[:48] + bytes([enc[48] ^ 0x40])]
    out += [enc[:48] + bytes([enc[48] | b]) for b in (1, 2, 4, 8, 16, 32)]
    for k in range(6):
        limb = int.from_bytes(enc[8 * k:8 * k + 8], "little")
        if limb + o.P < 2**64:
            out.append(enc[:8 * k] + (limb + o.P).to_bytes(8, "little") + enc[8 * k + 8:])
    return out


@pytest.mark.parametrize("size", [1, 2, 3, 1000])
def test_search_against_a_dictionary(hostsim, size):
    rng = np.random.default_rng(size)
    n_honest = max(1, size * 3 // 5)
    pk, inf = honest_keys(10 + size, n_honest)
    apk, ainf, _ = adversarial_keys()
    extra = [pt_to96(o.pt_neg(pt_from96(pk[0]))), pt_to96(small_limb_point())]   # -P of a key, a small x limb
    pool_pk = np.concatenate([pk, apk, np.stack(extra)])
    pool_inf = np.concatenate([inf, ainf, [0, 0]]).astype(np.uint8)
    if size <= 3:
        sel = rng.choice(len(pool_pk), size, replace=False)
    else:                                                     # every pool key, then duplicates
        sel = np.concatenate([np.arange(len(pool_pk)), rng.integers(0, len(pool_pk), size - len(pool_pk))])
        rng.shuffle(sel)
    spk, sinf = pool_pk[sel], pool_inf[sel]
    want = model(hostsim, spk, sinf)
    tab, m = table(hostsim, spk, sinf)
    assert m == len(want)
    queries = []
    for k in range(len(pool_pk)):
        enc = encode(hostsim, pool_pk[k], pool_inf[k])[0]
        queries += [enc] + variants(enc)
    queries += [bytes(rng.integers(0, 256, 49, dtype=np.uint8)) for _ in range(200)]
    queries += [bytes(49), bytes(48) + b"\x80", bytes(48) + b"\xc0"]
    got = lookup(hostsim, tab, m, queries)
    assert got == [want.get(q, MISS) for q in queries]
    if size == 1000:
        assert len(set(sel.tolist())) == len(pool_pk) and len(want) < size     # duplicates present, found once
        enc = [encode(hostsim, spk[k], sinf[k]) for k in range(size)]
        dup = [k for k in range(size) if enc[k][1] and want[enc[k][0]] != k]
        assert dup                                            # the smallest index wins for a duplicated key
        hits = lookup(hostsim, tab, m, [enc[k][0] for k in dup])
        assert all(h < k for h, k in zip(hits, dup))
