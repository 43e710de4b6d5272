"""Batch randomisers generated on the device from a 32-byte seed (schnorr_b200_batch_randomizers[_dev]) and the seeded
forms of the four batch verifications (schnorr_b200_verify_batch[_registered|_keyed|_keyed_registered]_seeded): the
generator's bytes equal the hashlib oracle of tests/randomizer_ref.py, and every seeded form's verdict, lhs97 and rhs97
equal, byte for byte, its parent's fed with rand32 = batch_randomizers(seed, 0, n)."""
import ctypes as C

import numpy as np
import pytest

import schnorr_sig_b200.synth as synth
from randomizer_ref import batch_randomizers as oracle_randomizers
from test_gpu_keyed_registered import keyed_workload
from test_gpu_registered import keyset_workload

pytestmark = pytest.mark.gpu

EARG = -1


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    e = s.Engine(0)
    yield e
    e.close()


def seed_of(k):
    return np.random.default_rng(1000 + k).integers(0, 256, 32, dtype=np.uint8).tobytes()


def dev_randomizers(eng, n, seed, first):
    import torch
    s = torch.from_numpy(np.frombuffer(seed, dtype=np.uint8).copy()).cuda()
    out = torch.full((max(n, 1), 32), 0xAA, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    eng.batch_randomizers_dev(n, s, first, out)
    eng.synchronize()
    return out[:n].cpu().numpy()


# ---- 1. generator bytes ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 255, 256, 4097, 1 << 16])
def test_generator_equals_the_oracle(eng, n):
    seed = seed_of(n)
    for first in (0, 12345, 2**64 - n):
        want = oracle_randomizers(seed, first, n)
        assert np.array_equal(eng.batch_randomizers(n, seed, first), want), first
        assert np.array_equal(dev_randomizers(eng, n, seed, first), want), first


def test_adjacent_slices_concatenate(eng):
    seed = seed_of(7)
    whole = eng.batch_randomizers(10000, seed, 500)
    for cut in (1, 128, 4097, 9999):
        a = eng.batch_randomizers(cut, seed, 500)
        b = eng.batch_randomizers(10000 - cut, seed, 500 + cut)
        assert np.array_equal(np.concatenate([a, b]), whole)
    assert eng.batch_randomizers(0, seed, 2**64 - 1).shape == (0, 32)


def test_generator_argument_errors(eng):
    L, h = eng._L, eng._h
    seed = np.frombuffer(seed_of(1), dtype=np.uint8).copy()
    out = np.zeros((4, 32), dtype=np.uint8)
    p = lambda a: C.c_void_p(a.ctypes.data)
    assert L.schnorr_b200_batch_randomizers(h, 1, p(seed), 2**64 - 1, p(out)) == 0      # last index 2^64 - 1 fits
    assert L.schnorr_b200_batch_randomizers(h, 2, p(seed), 2**64 - 1, p(out)) == EARG   # 2^64 does not
    assert L.schnorr_b200_batch_randomizers(h, 4, p(seed), 2**64 - 3, p(out)) == EARG
    assert L.schnorr_b200_batch_randomizers(h, 4, None, 0, p(out)) == EARG
    assert L.schnorr_b200_batch_randomizers(h, 4, p(seed), 0, None) == EARG
    assert L.schnorr_b200_batch_randomizers_dev(h, 2, p(seed), 2**64 - 1, p(out)) == EARG
    assert L.schnorr_b200_batch_randomizers_dev(h, 4, None, 0, p(out)) == EARG
    v = C.c_int(-1)
    for name in ("schnorr_b200_verify_batch_seeded", "schnorr_b200_verify_batch_keyed_seeded"):
        fn = getattr(L, name)
        nargs = len(fn.argtypes)
        args = [h, 0] + [None] * (nargs - 2)
        args[nargs - 3] = C.byref(v)
        assert fn(*args) == EARG                                                          # NULL seed, empty batch
    with pytest.raises(ValueError):
        eng.batch_randomizers(1, b"short")
    multi = __import__("schnorr_sig_b200").Engine([0, 0])
    try:
        with pytest.raises(Exception, match="single-device"):
            multi.batch_randomizers_dev(1, seed.ctypes.data, 0, out.ctypes.data)
    finally:
        multi.close()


# ---- 2. seeded forms against the rand32 forms ------------------------------------------------------------------------
SIZES = [200, 4096, 1 << 16]
KINDS = ["valid", "bad", "malformed"]
VERDICT = {"valid": 0, "bad": 2, "malformed": 3}


def plain_workload(eng, n, kind):
    w = synth.signed_workload(eng, 77 + n, n)
    i = n // 3
    if kind == "bad":
        w["sigs"][i, 49:] = 0                        # e := 0
    elif kind == "malformed":
        w["sigs"][i, 49:] = 0xFF                     # e >= q
    return w, i


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", SIZES)
def test_verify_batch_seeded(eng, n, kind):
    w, _ = plain_workload(eng, n, kind)
    seed = seed_of(n)
    args = (w["sigs"], w["pk"], w["inf"], w["blob"], w["off"])
    v, lhs, rhs = eng.verify_batch_seeded(*args, seed)
    wv, wl, wr = eng.verify_batch(*args, eng.batch_randomizers(n, seed))
    assert v == wv == VERDICT[kind]
    if kind != "malformed":
        assert bytes(lhs) == bytes(wl) and bytes(rhs) == bytes(wr)


@pytest.fixture(params=["aggregated", "gathered"])
def reg_mode(eng, request):
    eng.set_registered_batch_threshold(0 if request.param == "aggregated" else 2**62)
    yield request.param
    eng.set_registered_batch_threshold(64)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", SIZES)
def test_verify_batch_registered_seeded(eng, reg_mode, n, kind):
    w = keyset_workload(eng, 91 + n, 16, n, adversarial=False, faults=False)
    i = n // 3
    if kind == "bad":
        w["blob"][int(w["off"][i])] ^= 1
    elif kind == "malformed":
        w["idx"][i] = w["n_keys"] + 5                # an index outside the set
    ks, status = eng.register_keys(w["pk"], w["inf"])
    try:
        seed = seed_of(n + 1)
        args = (ks, w["sigs"], w["idx"], w["blob"], w["off"])
        v, lhs, rhs = eng.verify_batch_registered_seeded(*args, seed)
        points = eng.last_batch_points()
        wv, wl, wr = eng.verify_batch_registered(*args, eng.batch_randomizers(n, seed))
        assert points == eng.last_batch_points()     # the same path
        assert v == wv == VERDICT[kind]
        if kind != "malformed":
            assert bytes(lhs) == bytes(wl) and bytes(rhs) == bytes(wr)
    finally:
        ks.close()


@pytest.mark.parametrize("registered", [False, True])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", SIZES)
def test_verify_batch_keyed_seeded(eng, registered, n, kind):
    w = keyed_workload(eng, 55 + n, n, miss=0.25, n_keys=16)
    i = n // 3
    if kind == "bad":
        w["rec"][i, 49 + 49:] = 0                    # e := 0
    elif kind == "malformed":
        w["rec"][i, :49] = 0xFF                      # an undecodable key
    seed = seed_of(n + 2)
    rand = eng.batch_randomizers(n, seed)
    if registered:
        eng.set_registered_batch_threshold(0)
        ks, _ = eng.register_keys(w["pk"], w["inf"])
        try:
            v, lhs, rhs = eng.verify_batch_keyed_registered_seeded(ks, w["rec"], w["blob"], w["off"], seed)
            wv, wl, wr = eng.verify_batch_keyed_registered(ks, w["rec"], w["blob"], w["off"], rand)
        finally:
            ks.close()
            eng.set_registered_batch_threshold(64)
    else:
        v, lhs, rhs = eng.verify_batch_keyed_seeded(w["rec"], w["blob"], w["off"], seed)
        wv, wl, wr = eng.verify_batch_keyed(w["rec"], w["blob"], w["off"], rand)
    assert v == wv == VERDICT[kind]
    if kind != "malformed":
        assert bytes(lhs) == bytes(wl) and bytes(rhs) == bytes(wr)


def test_dev_generator_feeds_the_dev_batch(eng):
    """batch_randomizers_dev followed by verify_batch_dev: the seeded host form's result"""
    import torch
    n = 4096
    w, _ = plain_workload(eng, n, "bad")
    seed = seed_of(3)
    v, lhs, rhs = eng.verify_batch_seeded(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], seed)
    d = [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).cuda()
         for a in (w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], np.frombuffer(seed, dtype=np.uint8).copy())]
    rand = torch.zeros((n, 32), dtype=torch.uint8, device="cuda")
    res = torch.full((216,), 255, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    eng.batch_randomizers_dev(n, d[5], 0, rand)
    eng.verify_batch_dev(n, d[0], d[1], d[2], d[3], d[4], rand, res)
    eng.synchronize()
    x = res.cpu().numpy()
    assert (int(x[0]), bytes(x[8:105]), bytes(x[112:209])) == (v, bytes(lhs), bytes(rhs)) and v == 2


# ---- 3. multi-device contexts ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
def test_multi_device_equals_single_device(eng, devices):
    import schnorr_sig_b200 as s
    n = 3 * 4096 + 77                                # sharded over every listed device
    seed = seed_of(11)
    w, _ = plain_workload(eng, n, "bad")
    kw = keyed_workload(eng, 12, n, miss=0.25, n_keys=16)
    kw["rec"][7, 49 + 49:] = 0                       # e := 0
    rw = keyset_workload(eng, 13, 16, n, adversarial=False, faults=True)
    multi = s.Engine(devices)
    eng.set_registered_batch_threshold(0)
    multi.set_registered_batch_threshold(0)
    ks1, _ = eng.register_keys(rw["pk"], rw["inf"])
    ksm, _ = multi.register_keys(rw["pk"], rw["inf"])
    kk1, _ = eng.register_keys(kw["pk"], kw["inf"])
    kkm, _ = multi.register_keys(kw["pk"], kw["inf"])
    try:
        assert np.array_equal(multi.batch_randomizers(n, seed, 9), eng.batch_randomizers(n, seed, 9))
        calls = [
            lambda e, ks, kk: e.verify_batch_seeded(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], seed),
            lambda e, ks, kk: e.verify_batch_registered_seeded(ks, rw["sigs"], rw["idx"], rw["blob"], rw["off"], seed),
            lambda e, ks, kk: e.verify_batch_keyed_seeded(kw["rec"], kw["blob"], kw["off"], seed),
            lambda e, ks, kk: e.verify_batch_keyed_registered_seeded(kk, kw["rec"], kw["blob"], kw["off"], seed),
        ]
        for call in calls:
            v1, l1, r1 = call(eng, ks1, kk1)
            vm, lm, rm = call(multi, ksm, kkm)
            assert (v1, bytes(l1), bytes(r1)) == (vm, bytes(lm), bytes(rm))
            assert v1 == 2
    finally:
        for k in (ks1, ksm, kk1, kkm):
            k.close()
        eng.set_registered_batch_threshold(64)
        multi.close()


# ---- 4. localisation with the materialised randomisers ---------------------------------------------------------------
@pytest.mark.parametrize("n", [200, 4096, 1 << 16])
def test_locate_with_the_seeded_randomizers(eng, n):
    seed = seed_of(20 + n)
    w, i = plain_workload(eng, n, "bad")
    args = (w["sigs"], w["pk"], w["inf"], w["blob"], w["off"])
    assert eng.verify_batch_seeded(*args, seed)[0] == 2
    flags = eng.locate_invalid(*args, eng.batch_randomizers(n, seed))
    assert list(np.nonzero(flags)[0]) == [i]
    kw = keyed_workload(eng, 30 + n, n, miss=0.25, n_keys=16)
    kw["rec"][i, 49 + 49:] = 0
    assert eng.verify_batch_keyed_seeded(kw["rec"], kw["blob"], kw["off"], seed)[0] == 2
    flags = eng.locate_invalid_keyed(kw["rec"], kw["blob"], kw["off"], eng.batch_randomizers(n, seed))
    assert list(np.nonzero(flags)[0]) == [i]


# ---- 5. the Python façade ----------------------------------------------------------------------------------------------
def test_python_api_seed():
    import os
    import schnorr_sig_b200 as s
    kp = [s.KeyPair.new() for _ in range(3)]
    idx = [i % 3 for i in range(300)]
    msgs = [b"m%d" % i for i in range(300)]
    sigs = [kp[k].sign(m) for k, m in zip(idx, msgs)]
    keys = [kp[k].public_key for k in idx]
    seed = os.urandom(32)
    assert s.verify_batch(sigs, keys, msgs, seed=seed).is_ok()
    assert s.locate_invalid(sigs, keys, msgs, seed=seed) == []
    bad = list(keys)
    bad[5], bad[6] = bad[6], bad[5]
    assert s.verify_batch(sigs, bad, msgs, seed=seed).is_err()
    assert [i for i, _ in s.locate_invalid(sigs, bad, msgs, seed=seed)] == [5, 6]
    with pytest.raises(ValueError):
        s.verify_batch(sigs, keys, msgs, rng=s.OsRng(), seed=seed)
    with pytest.raises(ValueError):
        s.locate_invalid(sigs, keys, msgs, rng=s.OsRng(), seed=seed)
    with pytest.raises(ValueError):
        s.verify_batch(sigs, keys, msgs, seed=b"\0" * 31)

    keyed = [s.KeyedSignature(k, sg) for k, sg in zip(keys, sigs)]
    assert s.verify_batch_keyed(keyed, msgs, seed=seed).is_ok()
    bad_keyed = [s.KeyedSignature(k, sg) for k, sg in zip(bad, sigs)]
    assert s.verify_batch_keyed(bad_keyed, msgs, seed=seed).is_err()
    assert [i for i, _ in s.locate_invalid_keyed(bad_keyed, msgs, seed=seed)] == [5, 6]
    with pytest.raises(ValueError):
        s.verify_batch_keyed(keyed, msgs, rng=s.OsRng(), seed=seed)

    ks = s.KeySet([k.public_key for k in kp])
    assert ks.verify_batch(idx, sigs, msgs, seed=seed).is_ok()
    bad_idx = list(idx)
    bad_idx[5], bad_idx[6] = bad_idx[6], bad_idx[5]
    assert ks.verify_batch(bad_idx, sigs, msgs, seed=seed).is_err()
    assert [i for i, _ in ks.locate_invalid(bad_idx, sigs, msgs, seed=seed)] == [5, 6]
    assert ks.verify_batch_keyed(keyed, msgs, seed=seed).is_ok()
    assert [i for i, _ in ks.locate_invalid_keyed(bad_keyed, msgs, seed=seed)] == [5, 6]
    with pytest.raises(ValueError):
        ks.verify_batch(idx, sigs, msgs, rng=s.OsRng(), seed=seed)
    with pytest.raises(s.PanicError):
        ks.verify_batch(idx[:-1] + [3], sigs, msgs, seed=seed)
