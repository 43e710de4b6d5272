"""Batch verification against registered key sets on the GPU (schnorr_b200_verify_batch_registered*,
schnorr_b200_locate_invalid_registered): verdict, lhs97 and rhs97 equal, byte for byte, what verify_batch returns on the
gathered key records, and last_batch_points shows which path ran (n: key side summed per key, 2n: per-signature points,
0: block per signature)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cref
from test_gpu_registered import adversarial_keys, keyset_workload
from util import pack_msgs, rand_scalars

pytestmark = pytest.mark.gpu

EARG = -1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    e = s.Engine(0)
    yield e
    e.close()


def gathered(w, idx=None):
    """The key record of every item; an index outside the set gets all-ones limbs (what k_keyset_gather writes)."""
    idx = w["idx"] if idx is None else idx
    inr = idx < w["n_keys"]
    safe = np.where(inr, idx, 0)
    pk = np.where(inr[:, None], w["pk"][safe], 0xFF).astype(np.uint8)
    inf = np.where(inr, w["inf"][safe], 0).astype(np.uint8)
    return pk, inf


def check(eng, ks, w, rand, points, idx=None):
    """registered batch == verify_batch on the gathered records; the registered call used `points` MSM points"""
    idx = w["idx"] if idx is None else idx
    v, lhs, rhs = eng.verify_batch_registered(ks, w["sigs"], idx, w["blob"], w["off"], rand)
    got_points = eng.last_batch_points()
    pk, inf = gathered(w, idx)
    wv, wl, wr = eng.verify_batch(w["sigs"], pk, inf, w["blob"], w["off"], rand)
    assert (v, bytes(lhs), bytes(rhs)) == (wv, bytes(wl), bytes(wr))
    assert got_points == points
    return v


@pytest.fixture
def aggregate_always(eng):
    eng.set_registered_batch_threshold(0)
    yield
    eng.set_registered_batch_threshold(64)


@pytest.mark.parametrize("n_keys", [1, 7, 64])
@pytest.mark.parametrize("n", [257, 4096, 1 << 16])
def test_honest_batches(eng, aggregate_always, n_keys, n):
    w = keyset_workload(eng, 1000 + n + n_keys, n_keys, n, adversarial=False, faults=False)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    rand = rand_scalars(np.random.default_rng(n + n_keys), n)
    assert check(eng, ks, w, rand, n) == 0


def test_faults_and_oracle(eng, aggregate_always):
    n = 4096
    w = keyset_workload(eng, 21, 16, n, adversarial=False, faults=True)   # message flip, e := 0, R := O, flag byte
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(21), n)
    assert check(eng, ks, w, rand, n) == 2
    # each fault kind on its own, and a sample of ~300 items against the oracle
    for k, i in enumerate(range(50, 50 + 4 * 211, 211)):
        sel = np.r_[np.arange(300, 600), i]
        msgs = [bytes(w["blob"][int(w["off"][j]):int(w["off"][j + 1])]) for j in sel]
        blob, off = pack_msgs(msgs)
        sub = dict(w, sigs=w["sigs"][sel], idx=w["idx"][sel], blob=blob, off=off)
        r = rand[sel]
        assert check(eng, ks, sub, r, len(sel)) == 2, k
        pk, inf = gathered(sub)
        want = cref.verify_batch(sub["sigs"], pk, inf, blob, off, r, cref.default_threads())
        got = eng.verify_batch_registered(ks, sub["sigs"], sub["idx"], blob, off, r)
        assert (got[0], bytes(got[1]), bytes(got[2])) == (want[0], bytes(want[1]), bytes(want[2]))


def test_identity_and_duplicate_keys_and_zero_randomisers(eng, aggregate_always):
    rng = np.random.default_rng(22)
    n = 3000
    sk = rand_scalars(rng, 5)
    sk[4] = 0                                                   # key 4: the identity
    pk, inf = eng.keygen(sk)
    assert inf[4] == 1
    keys_pk, keys_inf = np.concatenate([pk, pk[:2]]), np.concatenate([inf, inf[:2]])   # keys 5, 6 duplicate 0, 1
    idx = rng.integers(0, 7, n).astype(np.uint32)
    blob, off = pack_msgs([bytes(rng.integers(0, 256, 8, dtype=np.uint8)) for _ in range(n)])
    src = np.where(idx >= 5, idx - 5, idx)
    sigs = eng.sign_many(sk[src], pk[src], inf[src], blob, off, rand_scalars(rng, n))
    w = dict(pk=keys_pk, inf=keys_inf, idx=idx, sigs=sigs, blob=blob, off=off, n_keys=7)
    ks, status = eng.register_keys(keys_pk, keys_inf)
    assert not status.any() and (idx == 4).sum() > 100 and (idx >= 5).sum() > 100
    rand = rand_scalars(rng, n)
    rand[::7] = 0
    assert check(eng, ks, w, rand, n) == 0


@pytest.mark.parametrize("geometry", [(4, 0), (16, 0), (0, 8)])
def test_one_key_forced_geometries(eng, geometry):
    w = keyset_workload(eng, 23, 1, 4096, adversarial=False, faults=False)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(23), 4096)
    eng.set_msm_geometry(*geometry)
    try:
        assert check(eng, ks, w, rand, 4096) == 0
    finally:
        eng.set_msm_geometry(0, 0)


def test_off_subgroup_key_in_the_set_takes_the_gathered_path(eng):
    n = 4096
    w = keyset_workload(eng, 24, 16, n, adversarial=True, faults=False)   # the set holds keys of status 1
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert (status == 1).any()
    rand = rand_scalars(np.random.default_rng(24), n)
    check(eng, ks, w, rand, 2 * n)
    honest = w["idx"] < 16                                        # the same set, only honest keys used: still gathered
    sub = dict(w, sigs=w["sigs"][honest], idx=w["idx"][honest])
    msgs = [bytes(w["blob"][int(w["off"][j]):int(w["off"][j + 1])]) for j in np.nonzero(honest)[0]]
    sub["blob"], sub["off"] = pack_msgs(msgs)
    assert check(eng, ks, sub, rand[honest], 2 * int(honest.sum())) == 0


def test_malformed_key_and_out_of_range_index(eng):
    n = 2048
    w = keyset_workload(eng, 25, 8, n, adversarial=False, faults=False)
    apk, ainf, astat = adversarial_keys()
    bad = [k for k, s in enumerate(astat) if s == 3][0]
    pk, inf = np.concatenate([w["pk"], apk[bad:bad + 1]]), np.concatenate([w["inf"], ainf[bad:bad + 1]])
    ks, status = eng.register_keys(pk, inf)
    assert list(status) == [0] * 8 + [3]
    w = dict(w, pk=pk, inf=inf, n_keys=9)
    rand = rand_scalars(np.random.default_rng(25), n)
    assert check(eng, ks, w, rand, n) == 0                       # the status-3 key is in the set, unused
    idx = w["idx"].copy()
    idx[100] = 8                                                 # an item under the status-3 key
    assert check(eng, ks, w, rand, n, idx) == 3
    idx = w["idx"].copy()
    idx[101] = 2**32 - 1                                         # outside the set, among valid items
    assert check(eng, ks, w, rand, n, idx) == 3
    assert check(eng, ks, w, rand, n) == 0                       # the accumulator of the next batch is intact


def test_sizes_around_the_selections(eng):
    rng = np.random.default_rng(26)
    small = 256                                                 # the default batch_small_max
    w = keyset_workload(eng, 26, 4, 600, adversarial=False, faults=False)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(rng, 600)

    def head(m):
        msgs = [bytes(w["blob"][int(w["off"][j]):int(w["off"][j + 1])]) for j in range(m)]
        blob, off = pack_msgs(msgs)
        return dict(w, sigs=w["sigs"][:m], idx=w["idx"][:m], blob=blob, off=off)

    assert check(eng, ks, head(small), rand[:small], 0) == 0                         # block per signature
    assert check(eng, ks, head(small + 1), rand[:small + 1], small + 1) == 0        # 257 >= 64 per key
    w64 = keyset_workload(eng, 27, 64, 4096, adversarial=False, faults=False)
    ks64, _ = eng.register_keys(w64["pk"], w64["inf"])
    r64 = rand_scalars(rng, 4096)
    below = dict(w64, sigs=w64["sigs"][:4095], idx=w64["idx"][:4095], off=w64["off"][:4096])
    assert check(eng, ks64, below, r64[:4095], 2 * 4095) == 0                        # fewer than 64 per key
    assert check(eng, ks64, w64, r64, 4096) == 0
    eng.set_registered_batch_threshold(0)
    try:                                                                              # as many keys as signatures
        wn = keyset_workload(eng, 28, 1000, 1000, adversarial=False, faults=False)
        ksn, _ = eng.register_keys(wn["pk"], wn["inf"])
        assert check(eng, ksn, wn, rand_scalars(rng, 1000), 1000) == 0
    finally:
        eng.set_registered_batch_threshold(64)


def test_empty_batch(eng):
    w = keyset_workload(eng, 29, 4, 8, adversarial=False, faults=False)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    e = dict(w, sigs=w["sigs"][:0], idx=w["idx"][:0], off=w["off"][:1])
    check(eng, ks, e, rand_scalars(np.random.default_rng(29), 0), 0)


def test_multi_device_contexts_equal_the_single_device(eng):
    import schnorr_sig_b200 as s
    n = 20000
    w = keyset_workload(eng, 30, 64, n, adversarial=False, faults=True)
    rand = rand_scalars(np.random.default_rng(30), n)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    one = eng.verify_batch_registered(ks, w["sigs"], w["idx"], w["blob"], w["off"], rand)
    assert eng.last_batch_points() == n and one[0] == 2
    for devices in ([0, 0], [0, 0, 0]):
        m = s.Engine(devices)
        ksm, _ = m.register_keys(w["pk"], w["inf"])
        got = m.verify_batch_registered(ksm, w["sigs"], w["idx"], w["blob"], w["off"], rand)
        assert (got[0], bytes(got[1]), bytes(got[2])) == (one[0], bytes(one[1]), bytes(one[2]))
        assert m.last_batch_points() == n
        with pytest.raises(s.EngineError):                   # device buffers need a single-device context
            m.verify_batch_registered_dev(ksm, 1, 1, 1, 1, 1, 1, 1)
        ksm.close()
        m.close()


def test_dev_form_equals_the_host_form(eng):
    import torch
    n = 5000
    w = keyset_workload(eng, 31, 32, n, adversarial=False, faults=True)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(31), n)
    host = eng.verify_batch_registered(ks, w["sigs"], w["idx"], w["blob"], w["off"], rand)
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(w["sigs"]).to(dev), torch.from_numpy(w["idx"].view(np.int32)).to(dev),
         torch.from_numpy(w["blob"]).to(dev), torch.from_numpy(w["off"].view(np.int64)).to(dev),
         torch.from_numpy(rand).to(dev)]
    res = torch.full((216,), 255, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_batch_registered_dev(ks, n, t[0], t[1], t[2], t[3], t[4], res)
    eng.synchronize()
    r = res.cpu().numpy()
    assert eng.last_batch_points() == n
    assert (int(r[0]), bytes(r[8:105]), bytes(r[112:209])) == (host[0], bytes(host[1]), bytes(host[2]))


def test_argument_errors(eng):
    import schnorr_sig_b200 as s
    L = s._lib.lib()
    w = keyset_workload(eng, 32, 4, 8, adversarial=False, faults=False)
    ks, _ = eng.register_keys(w["pk"])
    other = s.Engine(0)
    ks_other, _ = other.register_keys(w["pk"])
    rand = rand_scalars(np.random.default_rng(32), 8)
    launches = eng.launch_count
    h = eng._h
    ptr = lambda a: C.c_void_p(a.ctypes.data)       # noqa: E731
    v = C.c_int(77)
    res = np.full(216, 77, np.uint8)
    flags = np.full(8, 77, np.uint8)
    args = [ptr(w["sigs"]), ptr(w["idx"]), ptr(w["blob"]), ptr(w["off"]), ptr(rand)]
    host = lambda ks_, a: L.schnorr_b200_verify_batch_registered(h, ks_, 8, *a, C.byref(v), None, None)   # noqa: E731
    dev = lambda ks_, a: L.schnorr_b200_verify_batch_registered_dev(h, ks_, 8, *a, ptr(res))               # noqa: E731
    loc = lambda ks_, a: L.schnorr_b200_locate_invalid_registered(h, ks_, 8, *a, ptr(flags), None)          # noqa: E731
    for fn in (host, dev, loc):
        assert fn(ks_other.handle, args) == EARG
        assert fn(None, args) == EARG
        for k in range(5):
            bad = list(args)
            bad[k] = None
            assert fn(ks.handle, bad) == EARG, k
    bad_off = w["off"].copy()
    bad_off[3], bad_off[4] = bad_off[4], bad_off[3]
    assert bad_off[3] > bad_off[4]
    for fn in (host, loc):
        assert fn(ks.handle, args[:3] + [ptr(bad_off)] + args[4:]) == EARG
    assert L.schnorr_b200_verify_batch_registered(h, ks.handle, 8, *args, None, None, None) == EARG   # no verdict
    assert eng.launch_count == launches and v.value == 77 and (res == 77).all() and (flags == 77).all()
    with pytest.raises(s.EngineError):
        eng.verify_batch_registered(ks_other, w["sigs"], w["idx"], w["blob"], w["off"], rand)
    ks_other.close()
    other.close()


def test_locate_invalid_registered(eng):
    n = 6000
    w = keyset_workload(eng, 33, 16, n, adversarial=False, faults=True)     # includes flipped y-sign flags
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    rand = rand_scalars(np.random.default_rng(33), n)
    got = eng.locate_invalid_registered(ks, w["sigs"], w["idx"], w["blob"], w["off"], rand)
    pk, inf = gathered(w)
    want = eng.locate_invalid(w["sigs"], pk, inf, w["blob"], w["off"], rand)
    assert np.array_equal(got, want) and (got == 2).sum() >= 20
    assert got[50 + 3 * 211] == 2                                   # the flipped flag (Signature::verify accepts it)
    idx = w["idx"].copy()
    idx[7] = 2**32 - 1
    got = eng.locate_invalid_registered(ks, w["sigs"], idx, w["blob"], w["off"], rand)
    assert got[7] == 3 and np.array_equal(np.delete(got, 7), np.delete(want, 7))
    flags = np.zeros(n, np.uint8)
    nb = C.c_uint64(0)
    L = eng._L
    ptr = lambda a: C.c_void_p(a.ctypes.data)       # noqa: E731
    assert L.schnorr_b200_locate_invalid_registered(eng._h, ks.handle, n, ptr(w["sigs"]), ptr(idx), ptr(w["blob"]),
                                                    ptr(w["off"]), ptr(rand), ptr(flags), C.byref(nb)) == 0
    assert nb.value == np.count_nonzero(flags) == np.count_nonzero(want != 0) + 1


def test_python_keyset_batch_api():
    import schnorr_sig_b200 as s
    kp = [s.KeyPair.new() for _ in range(3)]
    ks = s.KeySet([k.public_key for k in kp])
    idx = [i % 3 for i in range(300)]
    msgs = [b"m%d" % i for i in range(300)]
    sigs = [kp[k].sign(m) for k, m in zip(idx, msgs)]
    assert ks.verify_batch(idx, sigs, msgs).is_ok() and ks.locate_invalid(idx, sigs, msgs) == []
    bad = list(idx)
    bad[5], bad[6] = bad[6], bad[5]
    assert ks.verify_batch(bad, sigs, msgs).is_err()
    assert [i for i, _ in ks.locate_invalid(bad, sigs, msgs)] == [5, 6]
    for out in (3, -1, 2**40):
        with pytest.raises(s.PanicError):
            ks.verify_batch(idx[:-1] + [out], sigs, msgs)
        with pytest.raises(s.PanicError):
            ks.locate_invalid(idx[:-1] + [out], sigs, msgs)


CPP = r"""
#include <cstdio>
#include <random>
#include "schnorr_b200.hpp"
using namespace schnorr_sig;
int main() {
    Engine& eng = Engine::instance();
    std::mt19937_64 gen(3);
    Rng rng = [&](uint8_t* p, size_t n) { for (size_t i = 0; i < n; i++) p[i] = (uint8_t)gen(); };
    const size_t K = 2, N = 300;
    std::vector<uint8_t> sk(K * 32), inf(K, 0);
    rng(sk.data(), sk.size());
    for (size_t k = 0; k < K; k++) sk[k * 32 + 31] &= 0x3f;
    std::vector<PublicKey> keys(K);
    std::vector<uint8_t> pk(K * 96);
    eng.check(schnorr_b200_keygen(eng.get(), K, sk.data(), pk.data(), inf.data()), "keygen");
    for (size_t k = 0; k < K; k++) std::memcpy(keys[k].xy.data(), &pk[k * 96], 96);
    std::vector<size_t> idx(N);
    std::vector<Signature> sigs(N);
    std::vector<std::vector<uint8_t>> msgs(N);
    for (size_t i = 0; i < N; i++) {
        idx[i] = i % K;
        msgs[i] = {(uint8_t)i, (uint8_t)(i >> 8), 7};
        uint8_t nonce[32];
        rng(nonce, 32);
        nonce[31] &= 0x3f;
        uint64_t off[2] = {0, msgs[i].size()};
        std::array<uint8_t, 81> raw{};
        eng.check(schnorr_b200_sign_many(eng.get(), 1, &sk[idx[i] * 32], &pk[idx[i] * 96], &inf[idx[i]], msgs[i].data(), off,
                                         nonce, raw.data()), "sign");
        sigs[i] = Signature::from_raw(raw);
    }
    KeySet ks(keys);
    bool ok = !ks.verify_batch(idx, sigs, msgs, rng).has_value() && ks.locate_invalid(idx, sigs, msgs, rng).empty();
    std::swap(idx[10], idx[11]);
    Result r = ks.verify_batch(idx, sigs, msgs, rng);
    ok &= r.has_value() && *r == SignatureError::InvalidSignature;
    ok &= ks.locate_invalid(idx, sigs, msgs, rng) == std::vector<size_t>{10, 11};
    idx[0] = K;
    bool threw = false;
    try { ks.verify_batch(idx, sigs, msgs, rng); } catch (const std::logic_error&) { threw = true; }
    ok &= threw;
    std::printf("%s\n", ok ? "ok" : "FAILED");
    return ok ? 0 : 1;
}
"""


def test_cpp_facade(tmp_path):
    import schnorr_sig_b200 as s
    so = s._lib.library_path()
    s._lib.lib()
    src = tmp_path / "keyset_batch.cpp"
    src.write_text(CPP)
    exe = tmp_path / "keyset_batch"
    cudalib = "/usr/local/cuda/lib64"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                           str(src), "-o", str(exe), "-L" + os.path.dirname(so), "-l:" + os.path.basename(so),
                           "-Wl,-rpath," + os.path.dirname(so), "-L" + cudalib, "-lcudart", "-Wl,-rpath," + cudalib])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr


def test_full_size(eng):
    """2^20 signatures under 64 keys with one invalid signature per 1024: equal to verify_batch, n MSM points."""
    import schnorr_sig_b200 as s
    n, K = 1 << 20, 64
    w = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED, K)
    rng = np.random.default_rng(12)
    idx = rng.integers(0, K, n).astype(np.uint32)
    blob, off = s.synth.messages(s.synth.DEFAULT_SEED, 99, n, 8)
    sigs = eng.sign_many(w["sk"][idx], w["pk"][idx], w["inf"][idx], blob, off, s.synth.scalars(s.synth.DEFAULT_SEED, 98, n))
    item = dict(pk=w["pk"], inf=w["inf"], idx=idx, sigs=sigs, blob=blob, off=off, n_keys=K)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    rand = s.synth.scalars(s.synth.DEFAULT_SEED, 97, n)
    assert check(eng, ks, item, rand, n) == 0
    sigs[12345, 49] ^= 1
    assert check(eng, ks, item, rand, n) == 2
