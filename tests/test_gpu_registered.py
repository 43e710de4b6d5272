"""Registered key sets on the GPU (schnorr_b200_keyset_create / schnorr_b200_verify_registered_many*): the verdict of
every item equals, byte for byte, what verify_many returns for the same signature, message and key, and the oracle's."""
import ctypes as C

import numpy as np
import pytest

import cref
import pyref as o
from util import KAT96, pack_msgs, pt_to96, rand_scalars

pytestmark = pytest.mark.gpu

EARG = -1


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    return s.default_engine(0)


def adversarial_keys():
    """The keys of test_verify_adversarial_public_keys (orders 2, 29, 58, 2q, the cofactor) and the off-subgroup KAT
    point, then the identity, a key with a non-canonical limb, and an identity whose coordinates are not canonical."""
    kat = (o.KAT_X, o.KAT_Y)
    n = o.COFACTOR * o.Q
    pts = [o.pt_mul(kat, n // 2), o.pt_mul(kat, n // 29), o.pt_mul(kat, n // 58),
           o.pt_add(o.generator(), o.pt_mul(kat, n // 2)), o.pt_mul(kat, o.Q)]
    pk = [pt_to96(p) for p in pts] + [KAT96, np.zeros(96, np.uint8), pt_to96(o.generator()).copy(), np.full(96, 0xFF, np.uint8)]
    pk[7][8:16] = 0xFF
    inf = np.array([0] * 6 + [1, 0, 1], dtype=np.uint8)
    return np.stack(pk), inf, [1, 1, 1, 1, 1, 1, 0, 3, 0]


def keyset_workload(eng, seed, n_keys, n, lens=None, adversarial=True, faults=True):
    """n signatures under keys drawn from a set of n_keys honest keys (+ the adversarial keys, mixed into the index
    stream), messages of the given lengths, injected faults; returns the set, the items and the keys per item."""
    rng = np.random.default_rng(seed)
    sk = rand_scalars(rng, n_keys)
    pk, inf = eng.keygen(sk)
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    if lens is None:
        lens = [8] * n
    msgs = [bytes(rng.integers(0, 256, L, dtype=np.uint8)) for L in lens]
    blob, off = pack_msgs(msgs)
    sigs = eng.sign_many(sk[idx], pk[idx], inf[idx], blob, off, rand_scalars(rng, n))
    if adversarial:
        apk, ainf, _ = adversarial_keys()
        pk, inf = np.concatenate([pk, apk]), np.concatenate([inf, ainf])
        for j, i in enumerate(range(3, n, 97)):                      # every 97th item under an adversarial key
            idx[i] = n_keys + j % len(apk)
    if faults:
        for k, i in enumerate(range(50, n, 211)):                    # message flip, e := 0, x := identity, flag byte
            kind = k % 4
            if kind == 0 and lens[i]:
                blob[int(off[i])] ^= 1
            elif kind == 1:
                sigs[i, 49:] = 0
            elif kind == 2:
                sigs[i, :48] = 0
                sigs[i, 48] = 0x80
            else:
                sigs[i, 48] ^= 0x40
    return dict(pk=pk, inf=inf, idx=idx, sigs=sigs, blob=blob, off=off, n_keys=len(pk))


def expected(eng, w, oracle_sample=None):
    """verify_many on the keys of every item (index in range) and the oracle on all items or a sample of them."""
    idx = w["idx"]
    inr = idx < w["n_keys"]
    safe = np.where(inr, idx, 0)
    pk, inf = w["pk"][safe], w["inf"][safe]
    vm = eng.verify_many(w["sigs"], pk, inf, w["blob"], w["off"])
    vm[~inr] = 3
    sel = np.arange(len(idx)) if oracle_sample is None else np.random.default_rng(7).choice(len(idx), oracle_sample, replace=False)
    sel = sel[inr[sel]]
    msgs = [bytes(w["blob"][int(w["off"][i]):int(w["off"][i + 1])]) for i in sel]
    b, of = pack_msgs(msgs)
    ref = cref.verify_many(w["sigs"][sel], pk[sel], inf[sel], b, of, cref.default_threads())
    assert np.array_equal(vm[sel], ref)
    return vm


def test_registration_status(eng):
    rng = np.random.default_rng(1)
    pk, inf = eng.keygen(rand_scalars(rng, 3))
    apk, ainf, want = adversarial_keys()
    ks, status = eng.register_keys(np.concatenate([pk, apk]), np.concatenate([inf, ainf]))
    assert list(status) == [0, 0, 0] + want
    _ks, st2 = eng.register_keys(pk)                       # pk_inf may be omitted
    assert list(st2) == [0, 0, 0]


@pytest.mark.parametrize("n", [1, 127, 129, 1000, 10241, 40000])
def test_verdicts_match_verify_many_and_oracle(eng, n):
    lens = [(0, 7, 14, 8, 3, 21)[i % 6] for i in range(n)]
    w = keyset_workload(eng, 100 + n, 64, n, lens=lens)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    got = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
    want = expected(eng, w, oracle_sample=None if n <= 10241 else 2048)
    assert np.array_equal(got, want)
    if n >= 1000:
        assert {0, 1, 2, 3} <= set(int(v) for v in want)


def test_identity_key_signature(eng):
    rng = np.random.default_rng(3)
    blob, off = pack_msgs([b"identity", b"identity"])
    zeros = np.zeros((2, 96), np.uint8)
    sig = cref.sign_many(np.zeros((2, 32), np.uint8), zeros, np.ones(2, np.uint8), blob, off, rand_scalars(rng, 2))
    sig[1, 60] ^= 1
    pk, inf = eng.keygen(rand_scalars(rng, 1))
    ks, status = eng.register_keys(np.concatenate([pk, zeros[:1]]), np.array([0, 1], np.uint8))
    assert list(status) == [0, 0]
    idx = np.array([1, 1], np.uint32)
    assert list(eng.verify_registered_many(ks, sig, idx, blob, off)) == [0, 2]
    assert list(eng.verify_many(sig, zeros, np.ones(2, np.uint8), blob, off)) == [0, 2]


def test_out_of_range_indices_and_duplicate_keys(eng):
    w = keyset_workload(eng, 4, 5, 300, adversarial=False, faults=False)
    pk = np.concatenate([w["pk"], w["pk"][:2]])              # duplicates are accepted
    ks, status = eng.register_keys(pk)
    assert list(status) == [0] * 7
    idx = w["idx"].copy()
    dup = idx < 2
    idx[dup] += 5                                            # the same keys through their duplicates
    idx[10], idx[11], idx[12] = 7, 2**32 - 1, 1000           # outside the set
    got = eng.verify_registered_many(ks, w["sigs"], idx, w["blob"], w["off"])
    assert list(got[10:13]) == [3, 3, 3]
    mask = np.ones(len(idx), bool)
    mask[10:13] = False
    assert (got[mask] == 0).all() and dup.sum() > 10


def test_exact_count(eng):
    w = keyset_workload(eng, 5, 16, 2000, adversarial=False, faults=True)
    ks, _ = eng.register_keys(w["pk"])
    eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
    assert eng.last_exact_count() == 0
    w = keyset_workload(eng, 6, 16, 2000)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    got = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
    count, ms = eng.last_exact_count(), eng.last_kernel_ms()      # before expected(): verify_many resets both
    assert np.array_equal(got, expected(eng, w))
    # every item under an identity key goes to the exact kernel; off-subgroup keys are decided by their status
    ident = np.isin(w["idx"], np.nonzero(w["inf"])[0]).sum()
    assert ident > 0 and count == ident and ms > 0


def test_dev_form_with_torch_tensors(eng):
    import torch
    w = keyset_workload(eng, 7, 32, 3000)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(w["sigs"]).to(dev), torch.from_numpy(w["idx"].view(np.int32)).to(dev),
         torch.from_numpy(w["blob"]).to(dev), torch.from_numpy(w["off"].view(np.int64)).to(dev)]
    out = torch.full((3000,), 255, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_registered_many_dev(ks, 3000, t[0], t[1], t[2], t[3], out)
    eng.synchronize()
    assert np.array_equal(out.cpu().numpy(), expected(eng, w))


def test_exact_only_gives_the_same_verdicts(eng):
    w = keyset_workload(eng, 8, 64, 5000)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    fast = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
    eng.set_exact_only(True)
    try:
        exact = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        assert eng.last_exact_count() == 0
    finally:
        eng.set_exact_only(False)
    assert np.array_equal(fast, exact) and np.array_equal(fast, expected(eng, w, oracle_sample=512))


def test_multi_device_context_splits_the_call():
    import schnorr_sig_b200 as s
    eng = s.Engine([0, 0])
    n = 20000
    w = keyset_workload(eng, 9, 64, n)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert list(status[64:]) == adversarial_keys()[2]
    before = eng.launch_count
    got = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
    assert eng.launch_count - before == 8                   # gather, ingest, fast, exact on each of the two devices
    assert np.array_equal(got, expected(eng, w, oracle_sample=512))
    before = eng.launch_count
    small = eng.verify_registered_many(ks, w["sigs"][:100], w["idx"][:100], w["blob"][:int(w["off"][100])], w["off"][:101])
    assert eng.launch_count - before == 4 and np.array_equal(small, got[:100])
    with pytest.raises(s.EngineError):                      # device buffers need a single-device context
        eng.verify_registered_many_dev(ks, 1, 1, 1, 1, 1, 1)


def test_argument_errors(eng):
    import schnorr_sig_b200 as s
    L = s._lib.lib()
    w = keyset_workload(eng, 10, 4, 8, adversarial=False, faults=False)
    ks, _ = eng.register_keys(w["pk"])
    other = s.Engine(0)
    ks_other, _ = other.register_keys(w["pk"])
    launches = eng.launch_count
    with pytest.raises(s.EngineError):
        eng.verify_registered_many(ks_other, w["sigs"], w["idx"], w["blob"], w["off"])
    out = np.full(8, 77, np.uint8)
    h = eng._h
    ptr = lambda a: C.c_void_p(a.ctypes.data)       # noqa: E731
    args = [ptr(w["sigs"]), ptr(w["idx"]), ptr(w["blob"]), ptr(w["off"]), ptr(out)]
    for fn in (L.schnorr_b200_verify_registered_many, L.schnorr_b200_verify_registered_many_dev):
        assert fn(h, ks_other.handle, 8, *args) == EARG
        assert fn(h, None, 8, *args) == EARG
        for k in range(5):
            bad = list(args)
            bad[k] = None
            assert fn(h, ks.handle, 8, *bad) == EARG
        assert fn(h, ks.handle, 0, None, None, None, None, None) == 0
        assert fn(h, ks.handle, 0, *args) == 0
    assert eng.launch_count == launches and (out == 77).all()       # nothing was launched, nothing written
    hk = C.c_void_p()
    st = np.zeros(4, np.uint8)
    assert L.schnorr_b200_keyset_create(h, 0, ptr(w["pk"]), None, ptr(st), C.byref(hk)) == EARG and not hk.value
    assert L.schnorr_b200_keyset_create(h, 2**32, ptr(w["pk"]), None, ptr(st), C.byref(hk)) == EARG and not hk.value
    assert L.schnorr_b200_keyset_create(h, 4, None, None, ptr(st), C.byref(hk)) == EARG and not hk.value
    ks_other.close()
    other.close()


def test_python_keyset_api():
    import schnorr_sig_b200 as s
    kp = [s.KeyPair.new() for _ in range(3)]
    keys = [k.public_key for k in kp] + [s.PublicKey(bytes(KAT96))]
    ks = s.KeySet(keys)
    assert list(ks.status) == [0, 0, 0, 1] and len(ks) == 4
    sig = kp[1].sign(b"hello")
    assert ks.verify_signature(1, sig, b"hello").is_ok()
    assert ks.verify_signature(0, sig, b"hello").unwrap_err() == s.SignatureError(s.SignatureError.InvalidSignature)
    assert ks.verify_signature(3, sig, b"hello").unwrap_err() == s.SignatureError(s.SignatureError.InvalidPublicKey)
    for bad in (4, -1, 2**40):
        with pytest.raises(s.PanicError):
            ks.verify_signature(bad, sig, b"hello")


def test_full_size_bench_workload(eng):
    """2^20 signatures under 1024 keys with injected faults: every verdict equals verify_many's, a sample the oracle's."""
    import schnorr_sig_b200 as s
    n, K = 1 << 20, 1024
    w = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED, K)
    rng = np.random.default_rng(11)
    idx = rng.integers(0, K, n).astype(np.uint32)
    blob, off = s.synth.messages(s.synth.DEFAULT_SEED, 99, n, 8)
    nonce = s.synth.scalars(s.synth.DEFAULT_SEED, 98, n)
    sigs = eng.sign_many(w["sk"][idx], w["pk"][idx], w["inf"][idx], blob, off, nonce)
    for i in range(512, n, 1024):                            # one invalid signature per 1024: e +- 1, or a message bit
        if (i >> 10) % 2:
            sigs[i, 49] ^= 1
        else:
            blob[int(off[i])] ^= 1
    item = dict(pk=w["pk"], inf=w["inf"], idx=idx, sigs=sigs, blob=blob, off=off, n_keys=K)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    got = eng.verify_registered_many(ks, sigs, idx, blob, off)
    want = expected(eng, item, oracle_sample=2048)
    assert np.array_equal(got, want)
    assert (want == 2).sum() >= 1000 and (want == 0).sum() >= n - 1100
