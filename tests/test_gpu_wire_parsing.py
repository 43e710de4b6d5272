"""Point decoding and record parsing at every device entry point, on the adversarial encodings of wire_cases.py.

Each site that decodes or parses caller bytes gets the whole catalogue in one call per form, and is compared with the
oracle byte for byte where there are bytes: k_decompress (decompress, derive_public_children), k_ingest under each
single-verification kernel and the registered path, k_split_keyed / k_keyed_split_lookup / k_keyset_lookup /
k_keyset_encode (keyed records, registered sets), k_batch_small / k_batch_prepare / k_batch_item_check (the R side of
batches) and the key side of keyed batches, where the sign of a decoded key shows in lhs.  test_wire_cases_model.py
checks on the CPU that each row is what it is named after and that cref decodes it as pyref does."""
import numpy as np
import pytest

import cref
import pyref as o
import wire_cases as W
from util import make_workload, pack_msgs, rand_scalars

pytestmark = pytest.mark.gpu

ROWS = W.points()
NAMES = [r[0] for r in ROWS]
ENC = np.stack([np.frombuffer(b, np.uint8) for _, b, _ in ROWS])
MISS = 0xFFFFFFFF


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    return s.default_engine(0)


@pytest.fixture(autouse=True)
def defaults(eng):
    yield
    eng.set_exact_only(False)
    eng.set_one_threshold(512)
    eng.set_dist_threshold(10240)
    eng.set_batch_small_threshold(256)
    eng.set_batch_dist_threshold(2**18)
    eng.set_registered_batch_threshold(64)


def pt96(pt):
    return bytes(96) if pt is o.INF else o.f6_to_bytes(pt[0]) + o.f6_to_bytes(pt[1])


def decoded():
    """pyref.decompress of every row: [(ok, point)]"""
    return [o.decompress(b) for _, b, _ in ROWS]


def front_end_key(ok, pt):
    """the key record a batch sees for a keyed record: the decoded key, or the record of an index outside a set"""
    if not ok:
        return np.full(96, 0xFF, np.uint8), 0
    return np.frombuffer(pt96(pt), np.uint8), int(pt is o.INF)


def same_batch(got, want, what):
    """verdict, and lhs / rhs byte for byte unless the batch is malformed: for verdict 3 the oracle writes zeros and
    the block-per-signature form writes what it summed, and no caller reads those bytes"""
    assert got[0] == want[0], (what, got[0], want[0])
    if want[0] == 3:
        return
    assert bytes(got[1]) == bytes(want[1]), (what, "lhs")
    assert bytes(got[2]) == bytes(want[2]), (what, "rhs")


def test_decompress_and_compress(eng):
    pk, inf, ok = eng.decompress(ENC)
    want = decoded()
    for i, (wok, pt) in enumerate(want):
        assert bool(ok[i]) == wok, NAMES[i]
        if wok:
            assert inf[i] == (pt is o.INF) and bytes(pk[i]) == pt96(pt), NAMES[i]
    dec = np.nonzero(ok)[0]
    comp = eng.compress(pk[dec], inf[dec])
    for j, i in enumerate(dec):
        assert bytes(comp[j]) == bytes(o.compress(want[i][1])), NAMES[i]
        assert (bytes(comp[j]) == ROWS[i][1]) == (NAMES[i] != "t2_40"), NAMES[i]   # canonical except T2 under 0x40
    assert bytes(comp[list(dec).index(NAMES.index("t2_40"))]) == ROWS[NAMES.index("t2_00")][1]


def _record_inputs():
    rows = W.records()
    sigs, pks, inf = W.as_arrays(rows)
    blob, off = pack_msgs([W.MESSAGE] * len(rows))
    return rows, sigs, pks, inf, blob, off


def _force(eng, kernel):
    if kernel == "exact":
        eng.set_exact_only(True)
    elif kernel == "one":
        eng.set_one_threshold(2**62)
    elif kernel == "dist":
        eng.set_one_threshold(0)
        eng.set_dist_threshold(2**62)
    else:
        eng.set_one_threshold(0)
        eng.set_dist_threshold(0)


@pytest.mark.parametrize("kernel", ["one", "dist", "fast", "exact"])
def test_single_verify_on_positional_records(eng, kernel):
    """every key limb, sig.x limb and e edge through k_ingest and one verification kernel"""
    rows, sigs, pks, inf, blob, off = _record_inputs()
    want = cref.verify_many(sigs, pks, inf, blob, off, cref.default_threads())
    assert want[0] == 0 and {0, 2, 3} <= set(int(v) for v in want)
    _force(eng, kernel)
    got = eng.verify_many(sigs, pks, inf, blob, off)
    bad = [(rows[i][0], int(got[i]), int(want[i])) for i in np.nonzero(got != want)[0]]
    assert not bad


def test_registered_verify_on_positional_records(eng):
    """each record's key registered in its own slot: statuses and verdicts of verify_registered_many"""
    rows, sigs, pks, inf, blob, off = _record_inputs()
    ks, status = eng.register_keys(pks, inf)
    for i, (name, _, k, pinf, _) in enumerate(rows):
        if pinf:
            st = 0
        elif max(np.frombuffer(k, np.uint64)) >= o.P:
            st = 3
        else:
            st = 0 if cref.is_torsion_free(np.frombuffer(k, np.uint8)) else 1
        assert status[i] == st, name
    want = cref.verify_many(sigs, pks, inf, blob, off, cref.default_threads())
    got = eng.verify_registered_many(ks, sigs, np.arange(len(rows), dtype=np.uint32), blob, off)
    assert [rows[i][0] for i in np.nonzero(got != want)[0]] == []
    ks.close()


# ---- keyed records and registered sets ---------------------------------------------------------------------------
def _secret(name):
    """secret key of the decoded point of a row, where one is known"""
    if name == "identity":
        return 0
    if name.startswith("honest"):
        sk = W.honest_keys()[int(name[6])][0]
        return (o.Q - sk) if name.endswith("flipped") else sk
    return None


def _keyed_records(pad=0):
    """one keyed record per row (a valid signature under the decoded key where its secret is known, else the honest
    record's signature), then `pad` valid records under honest keys 0 and 1"""
    n = len(ROWS) + pad
    dec = decoded()
    sk = np.zeros((n, 32), np.uint8)
    pk = np.zeros((n, 96), np.uint8)
    inf = np.zeros(n, np.uint8)
    key49 = np.zeros((n, 49), np.uint8)
    signed = np.zeros(n, bool)
    for i in range(n):
        if i < len(ROWS):
            s, (ok, pt), key49[i] = _secret(NAMES[i]), dec[i], ENC[i]
        else:
            s, pt = W.honest_keys()[(i - len(ROWS)) % 2]
            ok = True
            key49[i] = np.frombuffer(o.compress(pt), np.uint8)
        if s is not None and ok:
            sk[i] = np.frombuffer(s.to_bytes(32, "little"), np.uint8)
            pk[i], inf[i] = front_end_key(ok, pt)
            signed[i] = True
    blob, off = pack_msgs([W.MESSAGE] * n)
    nonce = rand_scalars(np.random.default_rng(W.SEED), n)
    sigs = cref.sign_many(sk, pk, inf, blob, off, nonce, cref.default_threads())
    sigs[~signed] = np.frombuffer(W.honest_record()[2], np.uint8)
    return np.ascontiguousarray(np.concatenate([key49, sigs], axis=1)), blob, off, signed


def keyed_oracle(rec, blob, off):
    n = rec.shape[0]
    pk = np.zeros((n, 96), np.uint8)
    inf = np.zeros(n, np.uint8)
    ok = np.zeros(n, bool)
    for i in range(n):
        ok[i], pk[i], inf[i] = cref.decompress(rec[i, :49])
    v = cref.verify_many(np.ascontiguousarray(rec[:, 49:]), pk, inf, blob, off, cref.default_threads())
    v[~ok] = 3
    return v


def registered_set():
    """(pk96, inf): honest keys 0 and 1, an identity registered with non-zero coordinates, an off-curve record with the
    x of honest key 2 and the y of honest key 0, the identity, T2 and the subfield points as they decode under 0x00.
    The two records in the middle are not findable and come before the records their encodings could be confused
    with."""
    hon = [pt for _, pt in W.honest_keys()]
    recs = [(pt96(hon[0]), 0), (pt96(hon[1]), 0), (pt96(hon[0]), 1), (pt96((hon[2][0], hon[0][1])), 0),
            (bytes(96), 1), (pt96(W.t2()), 0)]
    recs += [(pt96(o.decompress(W.enc(x, 0x00))[1]), 0) for _, (x, _) in W.subfield_points()]
    return np.stack([np.frombuffer(r, np.uint8) for r, _ in recs]), np.array([i for _, i in recs], np.uint8)


def findable_model(pk, inf):
    """encoding -> smallest index whose encoding decodes back to the registered record (pyref)"""
    d = {}
    for k in range(len(pk)):
        b = bytes(pk[k])
        pt = o.INF if inf[k] else (tuple(int(v) for v in pk[k, :48].view(np.uint64)),
                                   tuple(int(v) for v in pk[k, 48:].view(np.uint64)))
        e = bytes(o.compress(pt))
        ok, dpt = o.decompress(e)
        if ok and pt96(dpt) == b and (dpt is o.INF) == bool(inf[k]) and e not in d:
            d[e] = k
    return d


def test_keyed_records_and_lookup(eng):
    import torch
    rec, blob, off, signed = _keyed_records(pad=400)
    want = keyed_oracle(rec, blob, off)
    n_rows = len(ROWS)
    assert (want[signed] == 0).all()
    dec = decoded()
    assert all(want[i] == 3 for i in range(n_rows) if not dec[i][0])
    assert np.array_equal(eng.verify_keyed_many(rec, blob, off), want)
    pk, inf = registered_set()
    ks, status = eng.register_keys(pk, inf)
    assert list(status) == [0, 0, 0, 1, 0, 1] + [1] * (len(pk) - 6)
    model = findable_model(pk, inf)
    assert len(model) == len(pk) - 2                         # the two unfindable records
    idx = eng.keyset_lookup(ks, ENC)
    assert [int(v) for v in idx] == [model.get(bytes(e), MISS) for e in ENC]
    for name in NAMES:
        if name == "t2_40" or name.endswith("flipped") or name.startswith("honest2"):
            assert idx[NAMES.index(name)] == MISS, name
    assert idx[NAMES.index("identity")] == 4 and idx[NAMES.index("t2_00")] == 5
    got = eng.verify_keyed_registered_many(ks, rec, blob, off)
    assert [NAMES[i] if i < n_rows else i for i in np.nonzero(got != want)[0]] == []
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(a).to(dev) for a in (rec, blob, off.view(np.int64))]
    out = torch.full((rec.shape[0],), 255, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_keyed_registered_many_dev(ks, rec.shape[0], t[0], t[1], t[2], out)
    eng.synchronize()
    assert np.array_equal(out.cpu().numpy(), want)
    ks.close()


# ---- batches: the R side ------------------------------------------------------------------------------------------
R_FORMS = [("small", 5, 256, 2**18), ("msm", 300, 0, 2**18), ("prepare_hash", 300, 0, 0)]


def _r_batches(n):
    """(honest workload, [sigs with item 2's R replaced by row k])"""
    w = make_workload(W.SEED + n, n)
    out = []
    for _, b, _ in ROWS:
        s = w["sigs"].copy()
        s[2, :49] = np.frombuffer(b, np.uint8)
        out.append(s)
    return w, out


def test_batch_r_side(eng):
    dec = decoded()
    nt = cref.default_threads()
    wants = {}
    for form, n, small, bdist in R_FORMS:
        if n not in wants:
            w, batches = _r_batches(n)
            wants[n] = (w, batches, [cref.verify_batch(s, w["pk"], w["inf"], w["blob"], w["off"], w["rand"], nt)
                                     for s in batches])
        w, batches, want = wants[n]
        eng.set_batch_small_threshold(small)
        eng.set_batch_dist_threshold(bdist)
        for k, s in enumerate(batches):
            assert want[k][0] == (2 if dec[k][0] else 3), NAMES[k]
            got = eng.verify_batch(s, w["pk"], w["inf"], w["blob"], w["off"], w["rand"])
            same_batch(got, want[k], (form, NAMES[k]))


def test_locate_invalid_r_side(eng):
    """every row at its own position of one batch: the flag of each is that of its one-item batch"""
    n = 2 * len(ROWS) + 20
    w = make_workload(W.SEED + 1, n)
    sigs = w["sigs"].copy()
    pos = [2 * k + 1 for k in range(len(ROWS))]
    sigs[pos, :49] = ENC
    flags = eng.locate_invalid(sigs, w["pk"], w["inf"], w["blob"], w["off"], w["rand"])
    assert set(np.nonzero(flags)[0]) <= set(pos)
    for k, i in enumerate(pos):
        blob, off = pack_msgs([w["msgs"][i]])
        one = cref.verify_batch(sigs[i:i + 1], w["pk"][i:i + 1], w["inf"][i:i + 1], blob, off, w["rand"][i:i + 1], 1)[0]
        assert flags[i] == one, NAMES[k]


# ---- batches: the key side of keyed records -----------------------------------------------------------------------
def test_keyed_batch_key_side(eng):
    """row k as the key of item 7 of an honest keyed batch, its signature kept: verify_batch_keyed and
    verify_batch_keyed_registered (summed per key or not) equal cref.verify_batch on the front-end records.  The
    Pippenger form throughout (small threshold 0), so that 64 records can be summed per key."""
    n = 64
    eng.set_batch_small_threshold(0)
    rec, blob, off, _ = _keyed_records(pad=n)
    base = np.ascontiguousarray(rec[len(ROWS):])
    blob, off = pack_msgs([W.MESSAGE] * n)
    rand = rand_scalars(np.random.default_rng(W.SEED + 7), n)
    dec = decoded()
    hon = [pt for _, pt in W.honest_keys()]
    sub_pk = np.stack([np.frombuffer(pt96(hon[0]), np.uint8), np.frombuffer(pt96(hon[1]), np.uint8), np.zeros(96, np.uint8)])
    ks_sub, st = eng.register_keys(sub_pk, np.array([0, 0, 1], np.uint8))
    assert not st.any()
    pk_all, inf_all = registered_set()
    ks_all, _ = eng.register_keys(pk_all, inf_all)
    sigs = np.ascontiguousarray(base[:, 49:])
    fe_pk = np.stack([np.frombuffer(pt96(hon[i % 2]), np.uint8) for i in range(n)])
    fe_inf = np.zeros(n, np.uint8)
    nt = cref.default_threads()
    for k in range(len(ROWS)):
        r = base.copy()
        r[7, :49] = ENC[k]
        pk, inf = fe_pk.copy(), fe_inf.copy()
        pk[7], inf[7] = front_end_key(*dec[k])
        want = cref.verify_batch(sigs, pk, inf, blob, off, rand, nt)
        if NAMES[k] != "honest1":                     # item 7 is signed under honest key 1
            assert want[0] == (2 if dec[k][0] else 3), NAMES[k]
        same_batch(eng.verify_batch_keyed(r, blob, off, rand), want, ("keyed", NAMES[k]))
        for ks, thr in ((ks_sub, 0), (ks_sub, 2**62), (ks_all, 0)):
            eng.set_registered_batch_threshold(thr)
            same_batch(eng.verify_batch_keyed_registered(ks, r, blob, off, rand), want, ("registered", thr, NAMES[k]))
            if ks is ks_sub and thr == 0 and dec[k][0]:
                assert eng.last_batch_points() < 2 * n, NAMES[k]          # the key side was summed per key
    ks_sub.close()
    ks_all.close()


def test_locate_invalid_keyed(eng):
    """every row as the key of its own record of one keyed batch: flags of locate_invalid on the front-end records"""
    n = 2 * len(ROWS) + 20
    rec, blob, off, _ = _keyed_records(pad=n)
    base = np.ascontiguousarray(rec[len(ROWS):])
    blob, off = pack_msgs([W.MESSAGE] * n)
    rand = rand_scalars(np.random.default_rng(W.SEED + 8), n)
    dec = decoded()
    pos = [2 * k + 1 for k in range(len(ROWS))]
    base[pos, :49] = ENC
    hon = [pt for _, pt in W.honest_keys()]
    pk = np.stack([np.frombuffer(pt96(hon[i % 2]), np.uint8) for i in range(n)])
    inf = np.zeros(n, np.uint8)
    for k, i in enumerate(pos):
        pk[i], inf[i] = front_end_key(*dec[k])
    want = eng.locate_invalid(np.ascontiguousarray(base[:, 49:]), pk, inf, blob, off, rand)
    assert all(want[i] == (2 if dec[k][0] else 3) for k, i in enumerate(pos) if not NAMES[k].startswith("honest"))
    assert np.array_equal(eng.locate_invalid_keyed(base, blob, off, rand), want)
    pk_all, inf_all = registered_set()
    ks, _ = eng.register_keys(pk_all, inf_all)
    assert np.array_equal(eng.locate_invalid_keyed_registered(ks, base, blob, off, rand), want)
    ks.close()


# ---- derivation ---------------------------------------------------------------------------------------------------
def test_derive_public_children_of_every_row(eng):
    import schnorr_sig_b200 as s
    chain = bytes(range(32))
    idx = np.array([5, 2**31], np.uint32)
    for (ok, pt), (name, b, _) in zip(decoded(), ROWS):
        if not ok:
            with pytest.raises(s.EngineError, match=r"failed \(-1\): parent extended public key does not decode"):
                eng.derive_public_children(b + chain, idx)
            continue
        kids, kok = eng.derive_public_children(b + chain, idx)
        child, cc, some = o.hd_derive_public(pt, chain, 5)
        assert bool(kok[0]) == some and not kok[1], name
        assert bytes(kids[0]) == bytes(o.compress(child)) + cc, name
