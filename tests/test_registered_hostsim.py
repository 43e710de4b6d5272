"""CPU checks of the registered-key-set path (schnorr-sig_b200/csrc/keyset.cuh compiled for the host by
tests/hostsim/registered.cpp)
against the oracle: the generalised table builder, h*P + e*G from a key table, the full per-signature composition and
the executed-multiply count of cost_model.W_EXECUTED_REG_L8.  The GPU runs are in tests/test_gpu_registered.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cost_model
import cref
import pyref as o
from util import KAT96, make_workload, pt_from96, pt_to96, rand_scalars, int_le

TF, NTF, EXC = 0, 1, 2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hostsim():
    """ctypes handle on the host build of hostsim.cpp + the registered-key-set exports (tests/hostsim/registered.cpp)."""
    d = os.path.join(ROOT, "tests", "hostsim")
    so = os.path.join(d, "libhostsim_registered.so")
    src = os.path.join(d, "registered.cpp")
    csrc = os.path.join(ROOT, "schnorr-sig_b200", "csrc")
    deps = [src, os.path.join(d, "hostsim.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    deps += [os.path.join(ROOT, "include", f) for f in ("cheetah_params.h", "fp_sqrt_tables.h")]
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", so, src])
    lib = C.CDLL(so)
    lib.hs_gtab.restype = C.c_void_p
    return lib


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def le32(k):
    return np.frombuffer(int(k).to_bytes(32, "little"), dtype=np.uint8).copy()


def geometry(hostsim):
    w, win, ent = C.c_int(0), C.c_int(0), C.c_int(0)
    hostsim.hs_kt_geometry(C.byref(w), C.byref(win), C.byref(ent))
    return w.value, win.value, ent.value


def table(hostsim, pt, w, windows):
    out = np.zeros((windows, (1 << (w - 1)) + 1, 12), dtype=np.uint64)
    hostsim.hs_tab_build(p(pt_to96(pt)), w, windows, p(out))
    return out


@pytest.fixture(scope="module")
def kt(hostsim):
    return geometry(hostsim)


def test_geometry(kt):
    w, windows, entries = kt
    assert windows * w > 255 and (windows - 1) * w <= 255 and entries == (1 << (w - 1)) + 1


def test_generalised_builder_gives_the_g_table(hostsim):
    """The builder the G table now comes from reproduces the independently built host G table bit for bit."""
    g = table(hostsim, o.generator(), 13, 20)
    ref = np.ctypeslib.as_array(C.cast(hostsim.hs_gtab(), C.POINTER(C.c_uint64)), shape=(20, 4097, 12))
    assert np.array_equal(g[:, 1:], ref[:, 1:])
    assert not g[:, 0].any()      # slot 0 (the identity) is zeros


def test_key_tables_are_multiples_of_the_key(hostsim, kt):
    w, windows, entries = kt
    rng = np.random.default_rng(51)
    G = o.generator()
    keys = [o.pt_mul(G, int_le(s)) for s in rand_scalars(rng, 3)]
    for P in keys:
        t = table(hostsim, P, w, windows)
        assert not t[:, 0].any()
        for i in sorted({0, 1, windows // 2, windows - 1}):
            B = o.pt_mul(P, 1 << (w * i))
            for d in sorted({1, 2, 3, entries // 2, entries - 2, entries - 1}):
                assert pt_from96(t[i, d].view(np.uint8)) == o.pt_mul(B, d), (i, d)


def test_key_status(hostsim):
    kat = (o.KAT_X, o.KAT_Y)
    n = o.COFACTOR * o.Q
    G = o.generator()
    assert hostsim.hs_keyset_key_status(p(pt_to96(o.pt_mul(G, 99))), 0) == 0
    assert hostsim.hs_keyset_key_status(p(KAT96), 0) == 1
    assert hostsim.hs_keyset_key_status(p(pt_to96(o.pt_mul(kat, n // 2))), 0) == 1
    bad = pt_to96(G).copy()
    bad[8:16] = 0xFF
    assert hostsim.hs_keyset_key_status(p(bad), 0) == 3
    assert hostsim.hs_keyset_key_status(p(bad), 1) == 0          # the identity ignores its coordinates


def test_registered_core_matches_the_oracle(hostsim, kt):
    """h*P + e*G from the key table: exact on random and edge scalars; exceptional cases reported, never wrong."""
    w, windows, _ = kt
    rng = np.random.default_rng(52)
    G = o.generator()
    k = 0x1234567
    P = o.pt_mul(G, k)
    t = table(hostsim, P, w, windows)
    half = 1 << (w - 1)
    carries = sum(half + 1 << (w * i) for i in range(windows - 1)) % o.Q           # a carry across every boundary
    top = (o.Q - 1) >> (w * (windows - 1)) << (w * (windows - 1))                  # a maximal top window
    hs = [0, 1, o.Q - 1, carries, sum((1 << w) - 1 << (w * i) for i in range(windows - 1)), top, top - 1,
          half, half + 1] + [int_le(s) for s in rand_scalars(rng, 6)]
    es = [0, 1, o.Q - 1, 4097] + [int_le(s) for s in rand_scalars(rng, 2)]
    out = np.zeros(96, dtype=np.uint8)
    for h in hs:
        assert h < o.Q
        for e in es:
            fr = hostsim.hs_verify_core_reg(p(t), p(le32(h)), p(le32(e)), p(out))
            want = o.pt_mul2(P, h, G, e)
            if want is o.INF:
                assert fr == EXC
            else:
                assert fr in (TF, EXC)
                if fr == TF:
                    assert pt_from96(out) == want, (h, e)
    # every random pair was decided by the fast path
    for h in hs[-6:]:
        for e in es[-2:]:
            assert hostsim.hs_verify_core_reg(p(t), p(le32(h)), p(le32(e)), p(out)) == TF
    # results the formulas cannot produce are handed back: the identity, h*P + e*G == O ...
    assert hostsim.hs_verify_core_reg(p(t), p(le32(5)), p(le32((-5 * k) % o.Q)), p(out)) == EXC
    assert hostsim.hs_verify_core_reg(p(t), p(le32(0)), p(le32(0)), p(out)) == EXC
    # ... and an accumulation that meets its own addend: h*P = G, then + 1*G (a doubling)
    assert hostsim.hs_verify_core_reg(p(t), p(le32(pow(k, -1, o.Q))), p(le32(1)), p(out)) == EXC


def verify_one_reg(hostsim, kt, sig, pk, inf, msg, tables):
    w, windows, _ = kt
    key = bytes(pk)
    if key not in tables:
        tables[key] = table(hostsim, pt_from96(pk), w, windows) if not inf and \
            hostsim.hs_keyset_key_status(p(pk), 0) == 0 else np.zeros(1, dtype=np.uint64)
    st = hostsim.hs_keyset_key_status(p(pk), int(inf))
    used = C.c_int(0)
    mb = np.frombuffer(msg, dtype=np.uint8).copy() if msg else np.zeros(1, dtype=np.uint8)
    v = hostsim.hs_verify_one_reg(p(sig), p(pk), int(inf), st, p(tables[key]), p(mb), C.c_uint64(len(msg)), C.byref(used))
    return v, used.value


def test_full_path_matches_verify_one(hostsim, kt):
    lens = [8, 0, 7, 80, 160, 3, 8, 8, 14, 8]
    w = make_workload(53, len(lens), lens=lens)
    sigs, pk, inf = w["sigs"].copy(), w["pk"].copy(), w["inf"].copy()
    sigs[1, 49:] = 0                      # e := 0
    pk[2] = KAT96                         # off-subgroup key
    sigs[3, :48] = 0; sigs[3, 48] = 0x80  # x := identity encoding
    sigs[4, 8:16] = 0xFF                  # non-canonical sig.x limb
    n = o.COFACTOR * o.Q
    pk[6] = pt_to96(o.pt_mul((o.KAT_X, o.KAT_Y), n // 2))   # key of order 2
    inf[7] = 1                            # identity key
    pk[8, 16:24] = 0xFF                   # non-canonical key limb
    sigs[9, 49:] = 0xFF                   # e >= q
    sigs[0, 48] ^= 0x40                   # the flag byte is ignored
    want = cref.verify_many(sigs, pk, inf, w["blob"], w["off"])
    assert list(want) == [0, 2, 1, 2, 3, 0, 1, 2, 3, 3]
    tables, used = {}, []
    for i, m in enumerate(w["msgs"]):
        v, u = verify_one_reg(hostsim, kt, sigs[i].copy(), pk[i].copy(), inf[i], m, tables)
        ref = hostsim.hs_verify_one(p(sigs[i].copy()), p(pk[i].copy()), int(inf[i]), p(np.frombuffer(m, dtype=np.uint8).copy()
                                                                                        if m else np.zeros(1, np.uint8)),
                                    C.c_uint64(len(m)))
        assert v == want[i] == ref, i
        used.append(u)
    assert used == [0, 0, 0, 0, 0, 0, 0, 1, 0, 0]       # only the identity key takes the exact routine


def test_executed_multiply_count(hostsim, kt):
    """cost_model.W_EXECUTED_REG_L8: products of one registered verification of an 8-byte message (table prebuilt,
    status known: registration work is not part of a verification)."""
    hostsim.hs_wide_count_reset.restype = C.c_ulonglong
    wl = make_workload(91, 2, lens=[8, 8])
    sig, pk = wl["sigs"][0].copy(), wl["pk"][0].copy()
    w, windows, _ = kt
    t = table(hostsim, pt_from96(pk), w, windows)
    mb = np.frombuffer(wl["msgs"][0], dtype=np.uint8).copy()
    used = C.c_int(0)
    hostsim.hs_gtab()
    hostsim.hs_wide_count_reset()
    v = hostsim.hs_verify_one_reg(p(sig), p(pk), 0, 0, p(t), p(mb), C.c_uint64(8), C.byref(used))
    count = hostsim.hs_wide_count_reset()
    assert v == 0 and used.value == 0
    assert count == cost_model.W_EXECUTED_REG_L8, count
    print({"registered": count, "fast": cost_model.W_EXECUTED_FAST_L8})
