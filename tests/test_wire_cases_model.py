"""The catalogue of adversarial wire encodings (wire_cases.py) on the CPU: every row has the property it is named after
under the big-integer oracle, the C oracle decodes and verifies every row as pyref does (the GPU test compares the
device with the C oracle), and the host build of the device headers decodes every row as pyref does."""
import ctypes as C

import numpy as np
import pytest

import cref
import pyref as o
import wire_cases as W

ROWS = W.points()
IDS = [r[0] for r in ROWS]


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def pt96(pt):
    return bytes(96) if pt is o.INF else o.f6_to_bytes(pt[0]) + o.f6_to_bytes(pt[1])


def limbs(b):
    return tuple(int.from_bytes(b[8 * i:8 * i + 8], "little") for i in range(6))


def test_every_category_is_populated():
    cats = {c for _, _, c in ROWS}
    assert cats == set(W.CATEGORIES)
    assert len(set(IDS)) == len(IDS)
    kinds = [k for k, _ in W.subfield_points()]
    assert kinds.count("fp3") >= 2 and kinds.count("ufp3") >= 2
    assert {c for *_, c in W.records()} == {"honest", "key", "sig", "e"}


@pytest.mark.parametrize("name,b,cat", ROWS, ids=IDS)
def test_named_property_holds(name, b, cat):
    ok, pt = o.decompress(b)
    x, flag = limbs(b), b[48]
    if cat == "honest":
        j = int(name[6])
        _, P = W.honest_keys()[j]
        assert ok and pt == (o.pt_neg(P) if name.endswith("flipped") else P)
        if j == 0:
            assert o.pt_mul(P, o.Q) is o.INF
    elif cat == "identity":
        assert ok == (name == "identity") and pt is o.INF
    elif cat == "reserved":
        assert flag & 0x3F and not ok and o.f6_from_bytes(b[:48]) is not None
    elif cat == "limbs":
        canonical = all(c < o.P for c in x)
        assert canonical == (name.endswith(("_p-1_00", "_p-1_80", "_2^63_00", "_2^63_80")))
        # a canonical x decodes exactly when it is on the curve and the identity flag is clear
        assert ok == (canonical and flag == 0x00 and o.f6_is_square(W.rhs(x)))
        if name.startswith("alias"):                   # the same x written canonically decodes
            k = int(name[-1])
            canon = tuple(c - o.P if i == k else c for i, c in enumerate(x))
            assert all(c < o.P for c in canon) and o.decompress(W.enc(canon, flag))[0]
    elif cat == "offcurve":
        assert all(c < o.P for c in x) and not o.f6_is_square(W.rhs(x)) and not ok and flag in (0x00, 0x40)
    elif cat == "torsion2":
        assert ok and pt == W.t2() and pt[1] == o.F6_ZERO and o.pt_add(pt, pt) is o.INF
        assert o.compress(pt)[48] == 0x00
    elif cat == "subfield":
        assert ok and W.in_fp3(W.rhs(x)) and x[1::2] != (0, 0, 0)
        y = pt[1]
        if "_fp3" in name:
            assert W.in_fp3(y) and y[5] == 0 and y != o.F6_ZERO
        else:
            assert "_ufp3" in name and W.in_u_fp3(y) and y[5] != 0
        assert o.f6_lex_largest(y) == bool(flag & 0x40)
    else:
        raise AssertionError(cat)


def test_c_oracle_decodes_every_row_as_pyref():
    for name, b, _ in ROWS:
        ok, pt = o.decompress(b)
        cok, c96, cinf = cref.decompress(np.frombuffer(b, np.uint8))
        assert cok == ok, name
        if ok:
            assert cinf == (pt is o.INF) and bytes(c96) == pt96(pt), name


def test_host_build_decodes_every_row_as_pyref(hostsim):
    out = np.zeros(96, np.uint8)
    oi = C.c_int(0)
    for name, b, _ in ROWS:
        ok, pt = o.decompress(b)
        rec = np.frombuffer(b, np.uint8).copy()
        assert bool(hostsim.hs_decompress(p(rec), p(out), C.byref(oi))) == ok, name
        if ok:
            assert oi.value == (pt is o.INF) and bytes(out) == pt96(pt), name


def test_records_are_named_for_what_they_hold():
    rows = W.records()
    _, pk, sig = W.honest_record()
    assert rows[0][1] == sig and o.verify(sig[:49], int.from_bytes(sig[49:], "little"), W.MESSAGE, pk) == o.OK
    for name, s, k, inf, cat in rows[1:]:
        changed = [i for i in range(81) if s[i] != sig[i]] if cat != "key" else \
            [48 + i for i in range(96) if k[i] != rows[0][2][i]]
        assert changed, name                            # every row differs from the honest record
        e = int.from_bytes(s[49:], "little")
        if cat == "e":
            assert (e >= o.Q) == (name in ("e_q", "e_q+1", "e_2^256-1", "e_top_gt_q")), name
        elif cat == "sig":
            assert (o.f6_from_bytes(s[:48]) is None) == ("p-1" not in name), name
        else:
            assert (max(limbs(k[:48]) + limbs(k[48:])) >= o.P) == ("p-1" not in name), name


def test_c_oracle_verdicts_on_the_records_equal_pyref():
    """the verdicts the GPU test takes from cref.verify_many, restated by pyref.verify"""
    rows = W.records()
    sigs, pks, inf = W.as_arrays(rows)
    blob = np.frombuffer(W.MESSAGE * len(rows), np.uint8).copy()
    off = np.arange(len(rows) + 1, dtype=np.uint64) * len(W.MESSAGE)
    got = cref.verify_many(sigs, pks, inf, blob, off, cref.default_threads())
    memo = {}
    for i, (name, s, k, pinf, _) in enumerate(rows):
        key = (s, k, pinf)
        if key not in memo:
            pk = o.INF if pinf else (limbs(k[:48]), limbs(k[48:]))
            memo[key] = o.verify(s[:49], int.from_bytes(s[49:], "little"), W.MESSAGE, pk)
        assert got[i] == memo[key], name
