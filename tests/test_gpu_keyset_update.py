"""In-place updates of registered key sets on the GPU (schnorr_b200_keyset_append / _replace / _remove): after every
update the set is, byte for byte on every device, what keyset_create builds from the current slot records (a removed
slot's record is 96 bytes of 0xFF with identity flag 0), and every entry point returns what it returns on that fresh
set.  Both registration kernels (one block per key, one thread per key) give the same bytes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cref
import pyref as o
from test_gpu_registered import adversarial_keys, expected
from util import KAT96, pack_msgs, pt_to96, rand_scalars

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG = -1
MISS = 0xFFFFFFFF
SIZE_MAX = 2**64 - 1
REMOVED = np.full(96, 0xFF, np.uint8)
MODES = {"default": 512, "block": SIZE_MAX, "thread": 0}


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    e = s.default_engine(0)
    yield e
    e.set_keyset_block_threshold(512)


def key_pool(eng, seed, n_honest):
    """Honest keys (secret keys known), then the adversarial keys of test_gpu_registered (small order, the off-subgroup
    KAT point, the identity, a non-canonical limb, an identity with junk coordinates) and a point off the curve."""
    rng = np.random.default_rng(seed)
    sk = rand_scalars(rng, n_honest)
    pk, inf = eng.keygen(sk)
    apk, ainf, _ = adversarial_keys()
    off_curve = pt_to96(o.generator()).copy()
    off_curve[48] ^= 1
    pk = np.concatenate([pk, apk, off_curve[None]])
    inf = np.concatenate([inf, ainf, [0]]).astype(np.uint8)
    return sk, pk, inf


def export(eng, ks, device_index=0, tables=True):
    return eng.keyset_debug_export(ks, device_index=device_index, tables=tables)


def assert_same_export(a, b, what=""):
    for k in ("pk96", "inf", "status", "lut"):
        assert np.array_equal(a[k], b[k]), "%s: %s differs" % (what, k)
    if a["tables"] is not None and b["tables"] is not None:
        assert np.array_equal(a["tables"], b["tables"]), "%s: tables differ" % what


def check_model(eng, ks, pk, inf, devices=1, tables=True):
    """The updated set equals a fresh keyset_create over the model records on every device."""
    fresh, st = eng.register_keys(pk, inf)
    for d in range(devices):
        assert_same_export(export(eng, ks, d, tables), export(eng, fresh, d, tables), "device %d" % d)
    assert np.array_equal(export(eng, ks, 0, False)["status"], st)
    fresh.close()
    return st


def random_step(rng, eng, ks, pk, inf, pool_pk, pool_inf):
    """One random append / replace / remove on ks and on the model (pk, inf); returns the new model."""
    n = len(pk)
    kind = int(rng.integers(3))
    if kind == 0:
        m = int(rng.integers(1, 5))
        sel = rng.integers(0, len(pool_pk), m)
        st = eng.keyset_append(ks, pool_pk[sel], pool_inf[sel])
        pk, inf = np.concatenate([pk, pool_pk[sel]]), np.concatenate([inf, pool_inf[sel]])
        assert len(st) == m
    elif kind == 1:
        slots = np.unique(rng.integers(0, n, int(rng.integers(1, 4)))).astype(np.uint32)
        sel = rng.integers(0, len(pool_pk), len(slots))
        eng.keyset_replace(ks, slots, pool_pk[sel], pool_inf[sel])
        pk, inf = pk.copy(), inf.copy()
        pk[slots], inf[slots] = pool_pk[sel], pool_inf[sel]
    else:
        slots = rng.integers(0, n, int(rng.integers(1, 4))).astype(np.uint32)     # repeats allowed
        eng.keyset_remove(ks, slots)
        pk, inf = pk.copy(), inf.copy()
        pk[slots], inf[slots] = REMOVED, 0
    return pk, inf


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("start", [1, 7, 300])
def test_updates_equal_a_fresh_set(eng, start, mode):
    eng.set_keyset_block_threshold(MODES[mode])
    try:
        rng = np.random.default_rng(start * 7 + len(mode))
        _sk, pool_pk, pool_inf = key_pool(eng, start, 6)
        pool_pk = np.concatenate([pool_pk, pool_pk[:2]])                     # duplicate encodings
        pool_inf = np.concatenate([pool_inf, pool_inf[:2]])
        sel = rng.integers(0, len(pool_pk), start)
        pk, inf = pool_pk[sel], pool_inf[sel]
        ks, _ = eng.register_keys(pk, inf)
        steps = 4 if start == 300 else 10
        for _ in range(steps):
            pk, inf = random_step(rng, eng, ks, pk, inf, pool_pk, pool_inf)
            assert ks.n_keys == len(pk)
            check_model(eng, ks, pk, inf)
    finally:
        eng.set_keyset_block_threshold(512)


def test_multi_device_context_updates_every_shard():
    import schnorr_sig_b200 as s
    m = s.Engine([0, 0])
    rng = np.random.default_rng(77)
    _sk, pool_pk, pool_inf = key_pool(m, 77, 6)
    pk, inf = pool_pk[:7].copy(), pool_inf[:7].copy()
    ks, _ = m.register_keys(pk, inf)
    for _ in range(8):
        pk, inf = random_step(rng, m, ks, pk, inf, pool_pk, pool_inf)
        check_model(m, ks, pk, inf, devices=2)


def test_both_registration_kernels_give_the_same_bytes(eng):
    _sk, pk, inf = key_pool(eng, 5, 40)
    want_status = [0] * 40 + adversarial_keys()[2] + [1]
    out = []
    for thr in (SIZE_MAX, 0):
        eng.set_keyset_block_threshold(thr)
        ks, st = eng.register_keys(pk, inf)
        assert list(st) == want_status
        out.append(export(eng, ks))
    eng.set_keyset_block_threshold(512)
    assert_same_export(out[0], out[1], "block against thread kernel")


def signed_items(eng, rng, sk_of_slot, pk, inf, n, n_slots):
    """n items over slots of the model: signed with the slot's secret key where it is known (honest keys), with a
    random key otherwise; a few indices outside the set."""
    idx = rng.integers(0, n_slots, n).astype(np.uint32)
    idx[::97] = n_slots + 3
    msgs = [bytes(rng.integers(0, 256, 8, dtype=np.uint8)) for _ in range(n)]
    blob, off = pack_msgs(msgs)
    sk = rand_scalars(rng, n)
    for i, k in enumerate(idx):
        if k < n_slots and sk_of_slot[k] is not None:
            sk[i] = sk_of_slot[k]
    spk, sinf = eng.keygen(sk)
    sigs = eng.sign_many(sk, spk, sinf, blob, off, rand_scalars(rng, n))
    for i in range(5, n, 101):
        sigs[i, 60] ^= 1
    return dict(idx=idx, sigs=sigs, blob=blob, off=off)


def test_entry_points_match_a_fresh_set(eng):
    import torch
    rng = np.random.default_rng(11)
    sk, pool_pk, pool_inf = key_pool(eng, 11, 96)
    n_h = 96
    pk, inf = pool_pk[:64].copy(), pool_inf[:64].copy()
    sk_of = [sk[k] for k in range(64)]
    ks, _ = eng.register_keys(pk, inf)
    old_pk = pk.copy()
    # replace 8 slots with new honest keys, remove 4, append honest keys, a duplicate and the adversarial keys
    rep = np.arange(0, 64, 8, dtype=np.uint32)
    eng.keyset_replace(ks, rep, pool_pk[64:72], pool_inf[64:72])
    pk[rep], inf[rep] = pool_pk[64:72], pool_inf[64:72]
    for j, k in enumerate(rep):
        sk_of[k] = sk[64 + j]
    rem = np.array([3, 5, 5, 9, 60], dtype=np.uint32)
    eng.keyset_remove(ks, rem)
    pk[rem], inf[rem] = REMOVED, 0
    for k in rem:
        sk_of[k] = None
    app = np.concatenate([np.arange(72, 80), [10], np.arange(n_h, len(pool_pk))])
    eng.keyset_append(ks, pool_pk[app], pool_inf[app])
    pk, inf = np.concatenate([pk, pool_pk[app]]), np.concatenate([inf, pool_inf[app]])
    sk_of += [sk[k] if k < n_h else None for k in app]
    fresh, _ = eng.register_keys(pk, inf)
    n_slots = len(pk)
    w = signed_items(eng, rng, sk_of, pk, inf, 3000, n_slots)
    # independent verification, host and device forms, against the oracle on a sample
    got = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
    assert np.array_equal(got, eng.verify_registered_many(fresh, w["sigs"], w["idx"], w["blob"], w["off"]))
    want = expected(eng, dict(w, pk=pk, inf=inf, n_keys=n_slots), oracle_sample=512)
    assert np.array_equal(got, want)
    assert {0, 1, 2, 3} <= set(int(v) for v in got)
    assert all(got[i] == 3 for i in range(len(got)) if w["idx"][i] < n_slots and w["idx"][i] in rem)
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(w["sigs"]).to(dev), torch.from_numpy(w["idx"].view(np.int32)).to(dev),
         torch.from_numpy(w["blob"]).to(dev), torch.from_numpy(w["off"].view(np.int64)).to(dev)]
    out = torch.full((3000,), 255, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_registered_many_dev(ks, 3000, t[0], t[1], t[2], t[3], out)
    eng.synchronize()
    assert np.array_equal(out.cpu().numpy(), got)
    # lookup: current keys, the keys that were replaced or removed (now misses unless still present)
    keys = eng.compress(np.concatenate([pk, old_pk]), np.concatenate([inf, np.zeros(64, np.uint8)]))
    li = eng.keyset_lookup(ks, keys)
    assert np.array_equal(li, eng.keyset_lookup(fresh, keys))
    assert li[0] == 0 and li[3] == MISS and li[n_slots + 8] == MISS and li[n_slots + 1] == 1   # slot 8 was replaced
    keys_t = torch.from_numpy(keys).to(dev)
    li_t = torch.zeros(len(keys), dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    eng.keyset_lookup_dev(ks, len(keys), keys_t, li_t)
    eng.synchronize()
    assert np.array_equal(li_t.cpu().numpy().view(np.uint32), li)
    # KeyedSignature records, under current keys and under replaced / removed ones
    slot = np.where(w["idx"] < n_slots, w["idx"], 0)
    use_old = (np.arange(3000) % 3 == 0) & (slot < 64)                        # the key the slot held before the updates
    rec_keys = np.where(use_old[:, None], old_pk[np.minimum(slot, 63)], pk[slot])
    rec_inf = np.where(use_old, 0, inf[slot]).astype(np.uint8)
    keyed = np.concatenate([eng.compress(rec_keys, rec_inf), w["sigs"]], axis=1)
    kv = eng.verify_keyed_registered_many(ks, keyed, w["blob"], w["off"])
    assert np.array_equal(kv, eng.verify_keyed_registered_many(fresh, keyed, w["blob"], w["off"]))
    assert np.array_equal(kv, eng.verify_keyed_many(keyed, w["blob"], w["off"]))
    kt = torch.from_numpy(keyed).to(dev)
    torch.cuda.synchronize(dev)
    eng.verify_keyed_registered_many_dev(ks, 3000, kt, t[2], t[3], out)
    eng.synchronize()
    assert np.array_equal(out.cpu().numpy(), kv)
    # batches (verdict, lhs, rhs) and localisation over the honest slots, and with a removed slot
    honest = np.array([k for k in range(n_slots) if sk_of[k] is not None], dtype=np.uint32)
    bw = dict(zip(("blob", "off"), pack_msgs([b"batch%d" % i for i in range(1024)])))
    bidx = honest[rng.integers(0, len(honest), 1024)]
    bsk = np.stack([sk_of[k] for k in bidx])
    spk, sinf = eng.keygen(bsk)
    bsigs = eng.sign_many(bsk, spk, sinf, bw["blob"], bw["off"], rand_scalars(rng, 1024))
    rand = rand_scalars(rng, 1024)
    for idx_case in (bidx, np.where(np.arange(1024) == 7, rem[0], bidx).astype(np.uint32)):
        a = eng.verify_batch_registered(ks, bsigs, idx_case, bw["blob"], bw["off"], rand)
        b = eng.verify_batch_registered(fresh, bsigs, idx_case, bw["blob"], bw["off"], rand)
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
        fa = eng.locate_invalid_registered(ks, bsigs, idx_case, bw["blob"], bw["off"], rand)
        assert np.array_equal(fa, eng.locate_invalid_registered(fresh, bsigs, idx_case, bw["blob"], bw["off"], rand))
    assert a[0] == 3 and fa[7] == 3
    res = torch.zeros(216, dtype=torch.uint8, device=dev)
    bt = [torch.from_numpy(x).to(dev) for x in (bsigs, bidx.view(np.int32), bw["blob"], bw["off"].view(np.int64), rand)]
    torch.cuda.synchronize(dev)
    eng.verify_batch_registered_dev(ks, 1024, *bt, res)
    eng.synchronize()
    b = eng.verify_batch_registered(fresh, bsigs, bidx, bw["blob"], bw["off"], rand)
    r = res.cpu().numpy()
    assert r[0] == b[0] and np.array_equal(r[8:105], b[1]) and np.array_equal(r[112:209], b[2])


def test_aggregation_follows_status_one_keys(eng):
    rng = np.random.default_rng(21)
    sk = rand_scalars(rng, 9)
    pk, inf = eng.keygen(sk)
    ks, _ = eng.register_keys(pk[:8], inf[:8])
    n = 1024
    idx = rng.integers(0, 8, n).astype(np.uint32)
    msgs = [b"agg%d" % i for i in range(n)]
    blob, off = pack_msgs(msgs)
    sigs = eng.sign_many(sk[idx], pk[idx], inf[idx], blob, off, rand_scalars(rng, n))
    rand = rand_scalars(rng, n)

    def batch():
        v = eng.verify_batch_registered(ks, sigs, idx, blob, off, rand)
        return v[0], eng.last_batch_points()

    assert batch() == (0, n)                                   # summed per key
    st = eng.keyset_append(ks, KAT96[None], np.zeros(1, np.uint8))
    assert list(st) == [1]
    assert batch() == (0, 2 * n)                               # a status-1 key: per-signature points
    eng.keyset_replace(ks, [8], pk[8:9], inf[8:9])
    assert batch() == (0, n)                                   # aggregation back on
    eng.keyset_append(ks, KAT96[None], np.zeros(1, np.uint8))
    eng.keyset_remove(ks, [9])
    assert batch() == (0, n)


def test_removed_index_behaves_like_an_index_outside_the_set(eng):
    import schnorr_sig_b200 as s
    kp = [s.KeyPair.new() for _ in range(3)]
    ks = s.KeySet([k.public_key for k in kp])
    msg = b"removed"
    sig = kp[1].sign(msg)
    assert ks.verify_signature(1, sig, msg).is_ok()
    assert ks.index_of(kp[1].public_key) == 1
    ks.remove([1, 1])
    assert list(ks.status) == [0, 3, 0] and len(ks) == 3
    with pytest.raises(s.PanicError):
        ks.verify_signature(1, sig, msg)
    assert ks.index_of(kp[1].public_key) is None
    with pytest.raises(s.PanicError):
        ks.verify_batch([1], [sig], [msg])
    with pytest.raises(s.PanicError):
        ks.locate_invalid([1], [sig], [msg])
    # what the reference gives for the key, once it is back in the slot
    ks.replace([1], [kp[1].public_key])
    assert ks.verify_signature(1, sig, msg).is_ok() and list(ks.status) == [0, 0, 0]
    r = ks.append([kp[2].public_key, kp[0].public_key])
    assert list(r) == [3, 4] and len(ks) == 5 and list(ks.status) == [0] * 5
    assert ks.verify_signature(4, kp[0].sign(msg), msg).is_ok()
    assert ks.index_of(kp[2].public_key) == 2                   # the smallest index of a duplicate
    with pytest.raises(s.PanicError):
        ks.remove([5])


def test_stream_order_and_growth(eng):
    import torch
    rng = np.random.default_rng(31)
    sk = rand_scalars(rng, 210)
    pk, inf = eng.keygen(sk)
    ks, _ = eng.register_keys(pk[:4], inf[:4])
    n = 1 << 15
    idx = np.zeros(n, dtype=np.uint32)
    blob, off = pack_msgs([b"order%d" % i for i in range(n)])
    sigs = eng.sign_many(np.repeat(sk[:1], n, 0), np.repeat(pk[:1], n, 0), np.repeat(inf[:1], n, 0), blob, off,
                         rand_scalars(rng, n))
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(x).to(dev) for x in (sigs, idx.view(np.int32), blob, off.view(np.int64))]
    out = torch.full((n,), 255, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_registered_many_dev(ks, n, t[0], t[1], t[2], t[3], out)     # not synchronised
    eng.keyset_replace(ks, [0], pk[4:5], inf[4:5])                          # the key the call uses
    eng.keyset_append(ks, pk[5:10], inf[5:10])                              # forces a growth
    assert (out.cpu().numpy() == 0).all()                                   # the old key's verdicts
    after = eng.verify_registered_many(ks, sigs[:64], idx[:64], blob[:int(off[64])], off[:65])
    assert (after == 2).all()                                               # the new key's verdicts
    model_pk, model_inf = np.concatenate([pk[4:5], pk[1:4], pk[5:10]]), np.concatenate([inf[4:5], inf[1:4], inf[5:10]])
    for k in range(10, 210):                                                # single-key appends across several growths
        eng.keyset_append(ks, pk[k:k + 1], inf[k:k + 1])
    model_pk, model_inf = np.concatenate([model_pk, pk[10:210]]), np.concatenate([model_inf, inf[10:210]])
    check_model(eng, ks, model_pk, model_inf)


def test_argument_errors_leave_the_set_unchanged(eng):
    import schnorr_sig_b200 as s
    L = eng._L
    rng = np.random.default_rng(41)
    pk, inf = eng.keygen(rand_scalars(rng, 6))
    ks, _ = eng.register_keys(pk[:4], inf[:4])
    before = export(eng, ks)
    other = s.Engine(0)
    h = ks.handle
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    idx_ok = np.array([1], np.uint32)
    cases = [
        L.schnorr_b200_keyset_append(other._h, h, 1, p(pk), None, None),              # a set of another context
        L.schnorr_b200_keyset_replace(other._h, h, 1, p(idx_ok), p(pk), None, None),
        L.schnorr_b200_keyset_remove(other._h, h, 1, p(idx_ok)),
        L.schnorr_b200_keyset_append(eng._h, h, 1, None, None, None),                  # NULL buffers with n > 0
        L.schnorr_b200_keyset_replace(eng._h, h, 1, None, p(pk), None, None),
        L.schnorr_b200_keyset_replace(eng._h, h, 1, p(idx_ok), None, None, None),
        L.schnorr_b200_keyset_remove(eng._h, h, 1, None),
        L.schnorr_b200_keyset_replace(eng._h, h, 1, p(np.array([4], np.uint32)), p(pk), None, None),   # index >= n_keys
        L.schnorr_b200_keyset_remove(eng._h, h, 2, p(np.array([0, 4], np.uint32))),
        L.schnorr_b200_keyset_replace(eng._h, h, 2, p(np.array([2, 2], np.uint32)), p(pk), None, None),  # duplicates
        L.schnorr_b200_keyset_append(eng._h, h, 2**32 - 4, p(pk), None, None),        # 2^32 slots
        L.schnorr_b200_keyset_debug_export(eng._h, h, 1, 0, 1, None, None, None, None, None, None),
        L.schnorr_b200_keyset_debug_export(eng._h, h, 0, 3, 2, None, None, None, None, None, None),
    ]
    assert cases == [EARG] * len(cases)
    assert_same_export(export(eng, ks), before, "after the errors")
    assert ks.n_keys == 4
    for fn, args in ((L.schnorr_b200_keyset_append, (None, None, None)), (L.schnorr_b200_keyset_remove, (None,)),
                     (L.schnorr_b200_keyset_replace, (None, None, None, None))):
        assert fn(eng._h, h, 0, *args) == 0                                            # n == 0: a no-op
    assert_same_export(export(eng, ks), before, "after the no-ops")
    with pytest.raises(ValueError):
        eng.keyset_replace(ks, [0, 1], pk[:1])


def test_full_size_updated_set(eng):
    """16 384 keys, 1024 slots replaced and 1024 removed, 2^20 signatures: the verdicts of the fresh model set."""
    import schnorr_sig_b200 as s
    K, n = 16384, 1 << 20
    rng = np.random.default_rng(51)
    sk = rand_scalars(rng, K + 1024)
    pk, inf = eng.keygen(sk)
    ks, _ = eng.register_keys(pk[:K], inf[:K])
    slots = rng.permutation(K)
    rep, rem = slots[:1024].astype(np.uint32), slots[1024:2048].astype(np.uint32)
    eng.keyset_replace(ks, rep, pk[K:], inf[K:])
    eng.keyset_remove(ks, rem)
    mpk, minf, msk = pk[:K].copy(), inf[:K].copy(), sk[:K].copy()
    mpk[rep], minf[rep], msk[rep] = pk[K:], inf[K:], sk[K:]
    mpk[rem] = REMOVED
    idx = rng.integers(0, K, n).astype(np.uint32)
    blob, off = pack_msgs([b"%08d" % i for i in range(n)])
    spk = mpk.copy()
    spk[rem] = pk[rem]                                  # signed under the key the slot held (verdict 3 either way)
    sigs = eng.sign_many(msk[idx], spk[idx], minf[idx], blob, off, rand_scalars(rng, n))
    got = eng.verify_registered_many(ks, sigs, idx, blob, off)
    fresh, _ = eng.register_keys(mpk, minf)
    want = eng.verify_registered_many(fresh, sigs, idx, blob, off)
    assert np.array_equal(got, want)
    assert ((want == 3) == np.isin(idx, rem)).all() and (want[~np.isin(idx, rem)] == 0).all()
    sel = rng.choice(n, 256, replace=False)
    msgs = [bytes(blob[int(off[i]):int(off[i + 1])]) for i in sel]
    b, of = pack_msgs(msgs)
    assert np.array_equal(got[sel], cref.verify_many(sigs[sel], mpk[idx[sel]], minf[idx[sel]], b, of, cref.default_threads()))


CPP = r"""
#include <cstdio>
#include <random>
#include "schnorr_b200.hpp"
using namespace schnorr_sig;
int main() {
    Engine& eng = Engine::instance();
    std::mt19937_64 gen(5);
    const size_t K = 4;
    std::vector<uint8_t> sk(K * 32), inf(K, 0), pk(K * 96);
    for (auto& b : sk) b = (uint8_t)gen();
    for (size_t k = 0; k < K; k++) sk[k * 32 + 31] &= 0x3f;
    eng.check(schnorr_b200_keygen(eng.get(), K, sk.data(), pk.data(), inf.data()), "keygen");
    std::vector<PublicKey> keys(K);
    for (size_t k = 0; k < K; k++) std::memcpy(keys[k].xy.data(), &pk[k * 96], 96);
    std::vector<uint8_t> msg = {1, 2, 3};
    auto sign = [&](size_t k) {
        uint8_t nonce[32];
        for (auto& b : nonce) b = (uint8_t)gen();
        nonce[31] &= 0x3f;
        uint64_t off[2] = {0, msg.size()};
        std::array<uint8_t, 81> raw{};
        eng.check(schnorr_b200_sign_many(eng.get(), 1, &sk[k * 32], &pk[k * 96], &inf[k], msg.data(), off, nonce, raw.data()), "sign");
        return Signature::from_raw(raw);
    };
    KeySet ks(std::vector<PublicKey>{keys[0], keys[1]});
    bool ok = ks.size() == 2;
    ok &= ks.append({keys[2], keys[3]}) == 2 && ks.size() == 4 && ks.status() == std::vector<uint8_t>(4, 0);
    ok &= !ks.verify_signature(3, sign(3), msg).has_value();
    ks.replace({0}, {keys[3]});
    ok &= !ks.verify_signature(0, sign(3), msg).has_value();
    Result r = ks.verify_signature(0, sign(0), msg);
    ok &= r.has_value() && *r == SignatureError::InvalidSignature;
    ok &= ks.index_of(keys[3]) == std::optional<uint32_t>(0);
    ks.remove({1});
    ok &= ks.status()[1] == 3 && ks.size() == 4 && !ks.index_of(keys[1]).has_value();
    bool threw = false;
    try { ks.verify_signature(1, sign(1), msg); } catch (const std::logic_error&) { threw = true; }
    ok &= threw;
    threw = false;
    try { ks.replace({4}, {keys[0]}); } catch (const std::logic_error&) { threw = true; }
    ok &= threw;
    std::printf("%s\n", ok ? "ok" : "FAILED");
    return ok ? 0 : 1;
}
"""


def test_cpp_facade(tmp_path):
    import schnorr_sig_b200 as s
    so = s._lib.library_path()
    s._lib.lib()
    src = tmp_path / "keyset_update.cpp"
    src.write_text(CPP)
    exe = tmp_path / "keyset_update"
    cudalib = "/usr/local/cuda/lib64"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                           str(src), "-o", str(exe), "-L" + os.path.dirname(so), "-l:" + os.path.basename(so),
                           "-Wl,-rpath," + os.path.dirname(so), "-L" + cudalib, "-lcudart", "-Wl,-rpath," + cudalib])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr
