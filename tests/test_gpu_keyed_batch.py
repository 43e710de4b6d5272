"""Batch verification over KeyedSignature wire records on the GPU (schnorr_b200_verify_batch_keyed*,
schnorr_b200_verify_batch_keyed_registered*, schnorr_b200_locate_invalid_keyed*): verdict, lhs97 and rhs97 equal, byte
for byte, what verify_batch returns on the front-end records -- the decoded key of every record, and for a record whose
key does not decode the record of an index outside a set (96 bytes of 0xFF, identity flag 0) -- and the registered form
equals the form without a set whatever the set holds.  last_batch_points shows which path ran: n + m (m misses) for the
key side summed per key in the host form, 2n for the per-signature points and the _dev form, 0 for a block per
signature."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cref
from test_gpu_keyed_registered import keyed_workload
from test_gpu_registered import adversarial_keys
from util import pack_msgs, rand_scalars

pytestmark = pytest.mark.gpu

EARG = -1
MISS = 0xFFFFFFFF
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    e = s.Engine(0)
    yield e
    e.close()


@pytest.fixture
def aggregate_always(eng):
    eng.set_registered_batch_threshold(0)
    yield
    eng.set_registered_batch_threshold(64)


def front_end(eng, rec):
    """the records verify_batch sees: the decoded keys, 0xFF limbs and identity flag 0 where a key does not decode"""
    pk, inf, ok = eng.decompress(rec[:, :49])
    bad = ok == 0
    pk[bad] = 0xFF
    inf[bad] = 0
    return np.ascontiguousarray(rec[:, 49:]), pk, inf


def want(eng, w, rand):
    sigs, pk, inf = front_end(eng, w["rec"])
    v, lhs, rhs = eng.verify_batch(sigs, pk, inf, w["blob"], w["off"], rand)
    return v, bytes(lhs), bytes(rhs)


def keyed(eng, w, rand, ks=None):
    if ks is None:
        v, lhs, rhs = eng.verify_batch_keyed(w["rec"], w["blob"], w["off"], rand)
    else:
        v, lhs, rhs = eng.verify_batch_keyed_registered(ks, w["rec"], w["blob"], w["off"], rand)
    return v, bytes(lhs), bytes(rhs)


def misses(eng, ks, w):
    return int((eng.keyset_lookup(ks, w["rec"][:, :49]) == MISS).sum())


def to_dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).cuda() for a in arrays]


def dev_result(eng, w, rand, ks=None):
    import torch
    n = len(w["rec"])
    rec, blob, off, r = to_dev(w["rec"], w["blob"], w["off"], rand)
    res = torch.full((216,), 255, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    if ks is None:
        eng.verify_batch_keyed_dev(n, rec, blob, off, r, res)
    else:
        eng.verify_batch_keyed_registered_dev(ks, n, rec, blob, off, r, res)
    eng.synchronize()
    x = res.cpu().numpy()
    return int(x[0]), bytes(x[8:105]), bytes(x[112:209])


UNDECODABLE = ("ones", "flag3f", "limb", "x0")


def damage(eng, w, kind, rng):
    """in place: up to four records get an undecodable key, the identity's encoding, or a scalar e >= q"""
    rec = w["rec"]
    n = len(rec)
    for j, i in enumerate(rng.choice(n, min(n, 4), replace=False)):
        if kind == "undecodable":
            k = UNDECODABLE[j]
            if k == "ones":
                rec[i, :49] = 0xFF
            elif k == "flag3f":
                rec[i, 48] |= 0x3F
            elif k == "limb":
                rec[i, 8:16] = 0xFF           # limb 1 = 2^64 - 1 >= p
            else:
                rec[i, :49] = 0               # x = 0
        elif kind == "identity":
            rec[i, :49] = eng.compress(np.zeros((1, 96), np.uint8), np.ones(1, np.uint8))[0]
        elif kind == "e_ge_q":
            rec[i, 49 + 49:] = 0xFF


# ---- 1. verify_batch_keyed == verify_batch on the front-end records ------------------------------------------------
@pytest.mark.parametrize("kind", ["honest", "undecodable", "identity", "e_ge_q"])
@pytest.mark.parametrize("n", [1, 4, 256, 257, 4096, 1 << 16])
def test_keyed_equals_verify_batch(eng, n, kind):
    w = keyed_workload(eng, 300 + n, n, miss=0.0, n_keys=16)
    rng = np.random.default_rng(n)
    damage(eng, w, kind, rng)
    rand = rand_scalars(rng, n)
    got = keyed(eng, w, rand)
    assert got == want(eng, w, rand)
    assert got[0] == {"honest": 0, "undecodable": 3, "identity": 2, "e_ge_q": 3}[kind]
    assert eng.last_batch_points() == (0 if n <= 256 else 2 * n)


def test_keyed_sample_matches_the_oracle(eng):
    n = 300
    w = keyed_workload(eng, 41, n)            # mixed stream: adversarial, undecodable and faulty records
    rand = rand_scalars(np.random.default_rng(41), n)
    assert keyed(eng, w, rand) == want(eng, w, rand) and want(eng, w, rand)[0] == 3
    sel = np.nonzero(eng.decompress(w["rec"][:, :49])[2] == 1)[0]    # the records whose key decodes
    msgs = [bytes(w["blob"][int(w["off"][i]):int(w["off"][i + 1])]) for i in sel]
    blob, off = pack_msgs(msgs)
    sub = dict(rec=np.ascontiguousarray(w["rec"][sel]), blob=blob, off=off)
    sigs, pk, inf = front_end(eng, sub["rec"])
    cv, cl, cr = cref.verify_batch(sigs, pk, inf, blob, off, rand[sel], cref.default_threads())
    assert keyed(eng, sub, rand[sel]) == (cv, bytes(cl), bytes(cr))


# ---- 2. the registered form == the form without a set ---------------------------------------------------------------
@pytest.mark.parametrize("miss", [0.0, 1 / 1024, 1 / 16, 1 / 2, 1.0])
@pytest.mark.parametrize("n_keys", [1, 7, 64])
@pytest.mark.parametrize("n", [257, 4096, 1 << 16])
def test_registered_equals_keyed(eng, aggregate_always, n, n_keys, miss):
    w = keyed_workload(eng, 500 + n + n_keys, n, miss=miss, n_keys=n_keys)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    rand = rand_scalars(np.random.default_rng(n * n_keys), n)
    base = keyed(eng, w, rand)
    assert base[0] == 0 and base == want(eng, w, rand)
    assert keyed(eng, w, rand, ks) == base
    m = misses(eng, ks, w)
    assert m == int(round(miss * n))
    assert eng.last_batch_points() == n + m


def test_default_threshold_follows_the_existing_rules(eng):
    n = 4096
    for n_keys, points in ((64, lambda m: n + m), (65, lambda m: 2 * n)):   # 4096 / 64 = 64 per key; 4096 / 65 < 64
        w = keyed_workload(eng, 600 + n_keys, n, miss=1 / 16, n_keys=n_keys)
        ks, _ = eng.register_keys(w["pk"], w["inf"])
        rand = rand_scalars(np.random.default_rng(n_keys), n)
        got = keyed(eng, w, rand, ks)
        assert eng.last_batch_points() == points(misses(eng, ks, w))
        assert got == keyed(eng, w, rand)
    w = keyed_workload(eng, 602, 256, miss=0.0, n_keys=1)              # batch_small_max: a block per signature
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(602), 256)
    assert keyed(eng, w, rand, ks) == want(eng, w, rand)
    assert eng.last_batch_points() == 0


# ---- 3. faults, and localisation ----------------------------------------------------------------------------------
FAULTS = ("message", "e0", "R_identity", "flag", "swap_in_set", "swap_outside")


def fault(w, kind, i, other_key49):
    rec, blob, off = w["rec"], w["blob"], w["off"]
    if kind == "message":
        blob[int(off[i])] ^= 1
    elif kind == "e0":
        rec[i, 49 + 49:] = 0
    elif kind == "R_identity":
        rec[i, 49:49 + 48] = 0
        rec[i, 49 + 48] = 0x80
    elif kind == "flag":
        rec[i, 49 + 48] ^= 0x40
    else:
        rec[i, :49] = other_key49


@pytest.mark.parametrize("kind", FAULTS)
def test_faults(eng, aggregate_always, kind):
    """each fault on a hit (and, for the faults of the signature, on a miss too) gives verdict 2 in every form"""
    n, K = 4096, 16
    w = keyed_workload(eng, 700, n, miss=1 / 16, n_keys=K)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(700), n)
    idx = eng.keyset_lookup(ks, w["rec"][:, :49])
    hits, outs = np.nonzero(idx != MISS)[0], np.nonzero(idx == MISS)[0]
    hit, miss = int(hits[10]), int(outs[5])
    if kind == "swap_in_set":
        other = eng.compress(w["pk"], w["inf"])[(idx[hit] + 1) % K]
    else:
        other = w["rec"][int(outs[0]), :49].copy()
    for i in (hit,) if kind.startswith("swap") else (hit, miss):
        fault(w, kind, i, other)
    base = want(eng, w, rand)
    assert base[0] == 2
    assert keyed(eng, w, rand) == base and keyed(eng, w, rand, ks) == base
    assert dev_result(eng, w, rand) == base and dev_result(eng, w, rand, ks) == base
    sigs, pk, inf = front_end(eng, w["rec"])
    flags = eng.locate_invalid(sigs, pk, inf, w["blob"], w["off"], rand)
    assert flags[hit] == 2
    assert np.array_equal(eng.locate_invalid_keyed(w["rec"], w["blob"], w["off"], rand), flags)
    assert np.array_equal(eng.locate_invalid_keyed_registered(ks, w["rec"], w["blob"], w["off"], rand), flags)


def test_locate_flags_undecodable_keys(eng):
    n = 6000
    w = keyed_workload(eng, 42, n, n_keys=64)                # mixed: undecodable keys, adversarial keys and faults
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(42), n)
    sigs, pk, inf = front_end(eng, w["rec"])
    flags = eng.locate_invalid(sigs, pk, inf, w["blob"], w["off"], rand)
    ok = eng.decompress(w["rec"][:, :49])[2]
    assert (flags[ok == 0] == 3).all() and (flags == 2).sum() >= 10
    assert np.array_equal(eng.locate_invalid_keyed(w["rec"], w["blob"], w["off"], rand), flags)
    assert np.array_equal(eng.locate_invalid_keyed_registered(ks, w["rec"], w["blob"], w["off"], rand), flags)
    assert keyed(eng, w, rand) == want(eng, w, rand) == keyed(eng, w, rand, ks)


# ---- 4. sets ----------------------------------------------------------------------------------------------------------
def test_set_edge_cases(eng, aggregate_always):
    n = 4096
    apk, ainf, astatus = adversarial_keys()
    w = keyed_workload(eng, 800, n, miss=1 / 16, n_keys=8)
    rand = rand_scalars(np.random.default_rng(800), n)
    base = keyed(eng, w, rand)
    assert base == want(eng, w, rand)
    # a status-1 key: the per-signature points (2n); a status-3 key; the keys registered twice; the identity key
    for extra in ([0], [7], [6], []):
        pk = np.concatenate([w["pk"], apk[extra], w["pk"][:3]])
        inf = np.concatenate([w["inf"], ainf[extra], w["inf"][:3]])
        ks, status = eng.register_keys(pk, inf)
        assert keyed(eng, w, rand, ks) == base
        m = misses(eng, ks, w)
        assert eng.last_batch_points() == (2 * n if 1 in status else n + m)
        idx = eng.keyset_lookup(ks, w["rec"][:, :49])
        assert (idx[idx != MISS] < 8).all()                          # the smallest index wins over the duplicates
        ks.close()
    # records under the identity key, which is in the set; zero randomisers
    ks, _ = eng.register_keys(np.concatenate([w["pk"], apk[[6]]]), np.concatenate([w["inf"], ainf[[6]]]))
    w2 = dict(w, rec=w["rec"].copy())
    w2["rec"][::97, :49] = eng.compress(apk[[6]], ainf[[6]])[0]
    assert (eng.keyset_lookup(ks, w2["rec"][::97, :49]) == 8).all()
    rand0 = rand.copy()
    rand0[::5] = 0
    for r in (rand, rand0):
        assert keyed(eng, w2, r, ks) == keyed(eng, w2, r) == want(eng, w2, r)
    rand_all0 = np.zeros_like(rand)
    assert keyed(eng, w, rand_all0, ks) == keyed(eng, w, rand_all0) == want(eng, w, rand_all0)


def test_updated_set(eng, aggregate_always):
    n, K = 1 << 14, 32
    w = keyed_workload(eng, 900, n, miss=1 / 16, n_keys=K)
    rand = rand_scalars(np.random.default_rng(900), n)
    base = keyed(eng, w, rand)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    sk = rand_scalars(np.random.default_rng(901), 4)
    fresh, fresh_inf = eng.keygen(sk)
    m0 = misses(eng, ks, w)
    eng.keyset_remove(ks, [3, 4])                       # records under keys 3 and 4 become misses
    assert keyed(eng, w, rand, ks) == base
    m1 = misses(eng, ks, w)
    assert m1 > m0 and eng.last_batch_points() == n + m1
    eng.keyset_replace(ks, [5], fresh[:1], fresh_inf[:1])
    assert keyed(eng, w, rand, ks) == base and misses(eng, ks, w) > m1
    eng.keyset_append(ks, w["pk"][3:5], w["inf"][3:5])  # keys 3 and 4 again, in new slots: hits again
    assert keyed(eng, w, rand, ks) == base
    assert eng.last_batch_points() == n + misses(eng, ks, w)


# ---- 5. MSM geometries ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,T", [(4, 0), (16, 0), (0, 8)])
def test_forced_geometries(eng, aggregate_always, c, T):
    n = 4096
    w = keyed_workload(eng, 1000 + c + T, n, miss=1 / 16, n_keys=16)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(c + T), n)
    base = want(eng, w, rand)
    eng.set_msm_geometry(c, T)
    try:
        assert keyed(eng, w, rand, ks) == base and dev_result(eng, w, rand, ks) == base
        plan = eng.last_batch_plan()
        assert (plan[0] == c or not c) and (plan[3] == T or not T)
    finally:
        eng.set_msm_geometry(0, 0)


# ---- 6. forms ---------------------------------------------------------------------------------------------------------
def test_dev_forms_equal_host_forms(eng, aggregate_always):
    n = 5000
    w = keyed_workload(eng, 1100, n, miss=1 / 16, n_keys=32)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(1100), n)
    host = keyed(eng, w, rand)
    assert dev_result(eng, w, rand) == host and eng.last_batch_points() == 2 * n
    assert keyed(eng, w, rand, ks) == host and eng.last_batch_points() == n + misses(eng, ks, w)
    assert dev_result(eng, w, rand, ks) == host and eng.last_batch_points() == 2 * n
    empty = dict(rec=w["rec"][:0], blob=w["blob"][:0], off=w["off"][:1])
    r0 = rand[:0]
    want0 = want(eng, empty, r0)
    assert keyed(eng, empty, r0) == want0 == keyed(eng, empty, r0, ks) and want0[0] == 0


def test_multi_device_contexts_equal_the_single_device(eng):
    import schnorr_sig_b200 as s
    n = 20000
    w = keyed_workload(eng, 1200, n, miss=1 / 16, n_keys=64)
    w["rec"][77, 49 + 49] ^= 1                          # e changes: the batch fails
    rand = rand_scalars(np.random.default_rng(1200), n)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    one = keyed(eng, w, rand)
    assert one[0] == 2 and keyed(eng, w, rand, ks) == one
    one_flags = eng.locate_invalid_keyed(w["rec"], w["blob"], w["off"], rand)
    for devices in ([0, 0], [0, 0, 0]):
        m = s.Engine(devices)
        ksm, _ = m.register_keys(w["pk"], w["inf"])
        assert keyed(m, w, rand) == one
        assert m.last_batch_points() == 2 * n
        assert keyed(m, w, rand, ksm) == one
        assert m.last_batch_points() == n + misses(eng, ks, w)
        assert np.array_equal(m.locate_invalid_keyed_registered(ksm, w["rec"], w["blob"], w["off"], rand), one_flags)
        with pytest.raises(s.EngineError):                   # device buffers need a single-device context
            m.verify_batch_keyed_dev(1, 1, 1, 1, 1, 1)
        with pytest.raises(s.EngineError):
            m.verify_batch_keyed_registered_dev(ksm, 1, 1, 1, 1, 1, 1)
        ksm.close()
        m.close()


def test_argument_errors(eng):
    import schnorr_sig_b200 as s
    L = s._lib.lib()
    w = keyed_workload(eng, 1300, 8, miss=0.0, n_keys=4)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    other = s.Engine(0)
    ks_other, _ = other.register_keys(w["pk"])
    rand = rand_scalars(np.random.default_rng(1300), 8)
    launches = eng.launch_count
    h = eng._h
    ptr = lambda a: C.c_void_p(a.ctypes.data)       # noqa: E731
    v = C.c_int(77)
    res = np.full(216, 77, np.uint8)
    flags = np.full(8, 77, np.uint8)
    args = [ptr(w["rec"]), ptr(w["blob"]), ptr(w["off"]), ptr(rand)]
    forms = {
        "host": lambda a: L.schnorr_b200_verify_batch_keyed(h, 8, *a, C.byref(v), None, None),
        "dev": lambda a: L.schnorr_b200_verify_batch_keyed_dev(h, 8, *a, ptr(res)),
        "loc": lambda a: L.schnorr_b200_locate_invalid_keyed(h, 8, *a, ptr(flags), None),
    }
    reg = {
        "host": lambda k, a: L.schnorr_b200_verify_batch_keyed_registered(h, k, 8, *a, C.byref(v), None, None),
        "dev": lambda k, a: L.schnorr_b200_verify_batch_keyed_registered_dev(h, k, 8, *a, ptr(res)),
        "loc": lambda k, a: L.schnorr_b200_locate_invalid_keyed_registered(h, k, 8, *a, ptr(flags), None),
    }
    for name in forms:
        assert reg[name](ks_other.handle, args) == EARG
        assert reg[name](None, args) == EARG
        for k in range(4):
            if k == 1 and name != "dev":
                continue                       # a NULL msgs is an error in the host forms only when bytes are due
            bad = list(args)
            bad[k] = None
            assert forms[name](bad) == EARG, (name, k)
            assert reg[name](ks.handle, bad) == EARG, (name, k)
    bad_off = w["off"].copy()
    bad_off[3], bad_off[4] = bad_off[4], bad_off[3]
    bad = args[:2] + [ptr(bad_off)] + args[3:]
    for name in ("host", "loc"):
        assert forms[name](bad) == EARG and reg[name](ks.handle, bad) == EARG
        nomsg = args[:1] + [None] + args[2:]                  # 8 messages of 8 bytes and no blob
        assert forms[name](nomsg) == EARG and reg[name](ks.handle, nomsg) == EARG
    assert L.schnorr_b200_verify_batch_keyed(h, 8, *args, None, None, None) == EARG    # no verdict
    assert eng.launch_count == launches and v.value == 77 and (res == 77).all() and (flags == 77).all()
    with pytest.raises(s.EngineError):
        eng.verify_batch_keyed_registered(ks_other, w["rec"], w["blob"], w["off"], rand)
    ks_other.close()
    other.close()


# ---- 7. the façades -------------------------------------------------------------------------------------------------
def test_python_api():
    import schnorr_sig_b200 as s
    kp = [s.KeyPair.new() for _ in range(3)]
    outsider = s.KeyPair.new()
    ks = s.KeySet([k.public_key for k in kp])
    owners = [kp[i % 3] if i % 10 else outsider for i in range(300)]
    msgs = [b"m%d" % i for i in range(300)]
    keyed_sigs = [k.sign_and_bind_pkey(m) for k, m in zip(owners, msgs)]
    raw = [k.to_bytes() for k in keyed_sigs]
    for recs in (keyed_sigs, raw):
        assert s.verify_batch_keyed(recs, msgs).is_ok() and ks.verify_batch_keyed(recs, msgs).is_ok()
        assert s.locate_invalid_keyed(recs, msgs) == [] and ks.locate_invalid_keyed(recs, msgs) == []
    bad = list(raw)
    bad[5], bad[6] = bad[6], bad[5]
    assert s.verify_batch_keyed(bad, msgs).is_err() and ks.verify_batch_keyed(bad, msgs).is_err()
    assert [i for i, _ in s.locate_invalid_keyed(bad, msgs)] == [5, 6]
    assert [i for i, _ in ks.locate_invalid_keyed(bad, msgs)] == [5, 6]
    undecodable = list(raw)
    undecodable[9] = b"\xff" * 49 + raw[9][49:]
    for fn in (s.verify_batch_keyed, ks.verify_batch_keyed, s.locate_invalid_keyed, ks.locate_invalid_keyed):
        with pytest.raises(s.PanicError):
            fn(undecodable, msgs)
    assert s.verify_batch_keyed([], []).is_ok() and ks.locate_invalid_keyed([], []) == []


CPP = r"""
#include <cstdio>
#include <random>
#include "schnorr_b200.hpp"
using namespace schnorr_sig;
int main() {
    Engine& eng = Engine::instance();
    std::mt19937_64 gen(5);
    Rng rng = [&](uint8_t* p, size_t n) { for (size_t i = 0; i < n; i++) p[i] = (uint8_t)gen(); };
    const size_t K = 3, N = 300;      // key K - 1 is not registered
    std::vector<uint8_t> sk(K * 32), inf(K, 0), pk(K * 96);
    rng(sk.data(), sk.size());
    for (size_t k = 0; k < K; k++) sk[k * 32 + 31] &= 0x3f;
    eng.check(schnorr_b200_keygen(eng.get(), K, sk.data(), pk.data(), inf.data()), "keygen");
    std::vector<PublicKey> keys(K);
    for (size_t k = 0; k < K; k++) std::memcpy(keys[k].xy.data(), &pk[k * 96], 96);
    std::vector<KeyedSignature> recs(N);
    std::vector<std::vector<uint8_t>> msgs(N);
    for (size_t i = 0; i < N; i++) {
        size_t k = i % K;
        msgs[i] = {(uint8_t)i, (uint8_t)(i >> 8), 9};
        uint8_t nonce[32];
        rng(nonce, 32);
        nonce[31] &= 0x3f;
        uint64_t off[2] = {0, msgs[i].size()};
        std::array<uint8_t, 81> raw{};
        eng.check(schnorr_b200_sign_many(eng.get(), 1, &sk[k * 32], &pk[k * 96], &inf[k], msgs[i].data(), off, nonce,
                                         raw.data()), "sign");
        recs[i] = KeyedSignature{keys[k], Signature::from_raw(raw)};
    }
    KeySet ks(std::vector<PublicKey>(keys.begin(), keys.end() - 1));
    bool ok = !verify_batch_keyed(recs, msgs, rng).has_value() && !ks.verify_batch_keyed(recs, msgs, rng).has_value();
    ok &= locate_invalid_keyed(recs, msgs, rng).empty() && ks.locate_invalid_keyed(recs, msgs, rng).empty();
    std::swap(recs[10].public_key, recs[11].public_key);
    Result r = ks.verify_batch_keyed(recs, msgs, rng);
    ok &= r.has_value() && *r == SignatureError::InvalidSignature;
    r = verify_batch_keyed(recs, msgs, rng);
    ok &= r.has_value() && *r == SignatureError::InvalidSignature;
    ok &= ks.locate_invalid_keyed(recs, msgs, rng) == std::vector<size_t>{10, 11};
    ok &= locate_invalid_keyed(recs, msgs, rng) == std::vector<size_t>{10, 11};
    std::printf("%s\n", ok ? "ok" : "FAILED");
    return ok ? 0 : 1;
}
"""


def test_cpp_facade(tmp_path):
    import schnorr_sig_b200 as s
    so = s._lib.library_path()
    s._lib.lib()
    src = tmp_path / "keyed_batch.cpp"
    src.write_text(CPP)
    exe = tmp_path / "keyed_batch"
    cudalib = "/usr/local/cuda/lib64"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                           str(src), "-o", str(exe), "-L" + os.path.dirname(so), "-l:" + os.path.basename(so),
                           "-Wl,-rpath," + os.path.dirname(so), "-L" + cudalib, "-lcudart", "-Wl,-rpath," + cudalib])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr


# ---- 8. full size -----------------------------------------------------------------------------------------------------
def test_full_size(eng):
    """2^20 records under 1024 keys, 1/1024 of them under keys outside the set: equal to verify_batch on the front-end
    records, n + m MSM points."""
    n, K = 1 << 20, 1024
    w = keyed_workload(eng, 1400, n, miss=1 / 1024, n_keys=K)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    rand = rand_scalars(np.random.default_rng(1400), n)
    base = want(eng, w, rand)
    assert base[0] == 0
    assert keyed(eng, w, rand, ks) == base and eng.last_batch_points() == n + misses(eng, ks, w)
    assert keyed(eng, w, rand) == base
    w["rec"][123456, 49 + 60] ^= 1
    base = want(eng, w, rand)
    assert base[0] == 2 and keyed(eng, w, rand, ks) == base
