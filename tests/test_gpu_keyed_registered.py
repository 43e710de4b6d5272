"""KeyedSignature wire records against registered key sets on the GPU (schnorr_b200_verify_keyed_registered_many*,
schnorr_b200_keyset_lookup*): every verdict equals, byte for byte, what verify_keyed_many returns for the same record,
and the oracle's (decompress + verify_many); lookups equal a dictionary of the set's findable encodings."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cref
from test_gpu_registered import adversarial_keys
from util import pack_msgs, rand_scalars

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG = -1
MISS = 0xFFFFFFFF
HOST_MAX_MISS = 0.4       # KEYED_REG_MAX_MISS_FRACTION: host calls above this miss fraction run verify_many


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    return s.default_engine(0)


def keyed_workload(eng, seed, n, miss=None, n_keys=64, lens=None):
    """n keyed records under a set of n_keys honest keys.  miss=None: a mixed stream -- keys outside the set, the
    adversarial keys of test_gpu_registered (status 1 and 3, the identity, an identity with junk coordinates), keys
    registered twice, undecodable keys and the four fault kinds of keyset_workload.  miss=f: honest records, exactly
    round(f n) of them under keys outside the set.  Returns the records, messages and the set (pk, inf)."""
    rng = np.random.default_rng(seed)
    sk = rand_scalars(rng, n_keys + 16)                     # the last 16 keys are not registered
    pk, inf = eng.keygen(sk)
    owner = rng.integers(0, n_keys, n)
    if miss is None:
        owner[rng.random(n) < 0.05] = n_keys + rng.integers(0, 16)
    else:
        owner[rng.choice(n, int(round(miss * n)), replace=False)] = n_keys + rng.integers(0, 16, int(round(miss * n)))
    lens = lens or [8] * n
    msgs = [bytes(rng.integers(0, 256, L, dtype=np.uint8)) for L in lens]
    blob, off = pack_msgs(msgs)
    sigs = eng.sign_many(sk[owner], pk[owner], inf[owner], blob, off, rand_scalars(rng, n))
    key49 = eng.compress(pk[owner], inf[owner])
    set_pk, set_inf = pk[:n_keys], inf[:n_keys]
    if miss is None:
        apk, ainf, _ = adversarial_keys()
        set_pk = np.concatenate([set_pk, apk, set_pk[:2]])           # the first two keys registered twice
        set_inf = np.concatenate([set_inf, ainf, set_inf[:2]])
        akey = eng.compress(apk, ainf)
        for j, i in enumerate(range(3, n, 97)):
            key49[i] = akey[j % len(apk)]
        for j, i in enumerate(range(5, n, 101)):                     # undecodable: flag bits, random bytes
            if j % 2:
                key49[i, 48] |= 1 << (j % 6)
            else:
                key49[i] = rng.integers(0, 256, 49, dtype=np.uint8)
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
    rec = np.ascontiguousarray(np.concatenate([key49, sigs], axis=1))
    return dict(rec=rec, blob=blob, off=off, pk=set_pk, inf=set_inf.astype(np.uint8))


def oracle(rec, blob, off, sel):
    """KeyedSignature::from_bytes + verify on the C oracle for the records `sel`"""
    pk = np.zeros((len(sel), 96), np.uint8)
    inf = np.zeros(len(sel), np.uint8)
    ok = np.zeros(len(sel), bool)
    for j, i in enumerate(sel):
        ok[j], pk[j], inf[j] = cref.decompress(rec[i, :49])
    msgs = [bytes(blob[int(off[i]):int(off[i + 1])]) for i in sel]
    b, of = pack_msgs(msgs)
    v = cref.verify_many(rec[sel, 49:], pk, inf, b, of, cref.default_threads())
    v[~ok] = 3
    return v


def expected(eng, w, oracle_sample=None):
    want = eng.verify_keyed_many(w["rec"], w["blob"], w["off"])
    n = len(want)
    sel = np.arange(n) if oracle_sample is None or n <= oracle_sample else \
        np.random.default_rng(7).choice(n, oracle_sample, replace=False)
    assert np.array_equal(want[sel], oracle(w["rec"], w["blob"], w["off"], sel))
    return want


def findable_model(eng, pk, inf):
    """encoding -> smallest index of a key whose encoding decompresses back to its registered record"""
    enc = eng.compress(pk, inf)
    dpk, dinf, ok = eng.decompress(enc)
    d = {}
    for k in range(len(pk)):
        if ok[k] and np.array_equal(dpk[k], pk[k]) and dinf[k] == inf[k] and bytes(enc[k]) not in d:
            d[bytes(enc[k])] = k
    return d


@pytest.mark.parametrize("n", [1, 384, 385, 1000, 10241, 40000])
def test_verdicts_match_verify_keyed_many_and_oracle(eng, n):
    lens = [(0, 7, 14, 8, 3, 21)[i % 6] for i in range(n)]
    w = keyed_workload(eng, 200 + n, n, lens=lens)
    ks, status = eng.register_keys(w["pk"], w["inf"])
    got = eng.verify_keyed_registered_many(ks, w["rec"], w["blob"], w["off"])
    want = expected(eng, w, oracle_sample=2048)
    assert np.array_equal(got, want)
    if n >= 1000:
        assert {0, 1, 2, 3} <= set(int(v) for v in want)
        assert 1 in status and 3 in status


@pytest.mark.parametrize("miss", [0, 1 / 1024, 1 / 2, 1])
def test_miss_fractions(eng, miss):
    import torch
    n = 20000
    w = keyed_workload(eng, 300, n, miss=miss)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    want = expected(eng, w, oracle_sample=512)
    n_miss = int(round(miss * n))
    got = eng.verify_keyed_registered_many(ks, w["rec"], w["blob"], w["off"])
    host_exact = eng.last_exact_count()
    assert np.array_equal(got, want)
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(a).to(dev) for a in (w["rec"], w["blob"], w["off"].view(np.int64))]
    out = torch.full((n,), 255, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_keyed_registered_many_dev(ks, n, t[0], t[1], t[2], out)
    eng.synchronize()
    dev_exact = eng.last_exact_count()
    assert np.array_equal(out.cpu().numpy(), want)
    assert dev_exact >= n_miss                                # the _dev form hands every miss to the exact kernel
    if n_miss <= HOST_MAX_MISS * n:
        assert host_exact == dev_exact
    else:                                                     # the host form ran verify_many on the decoded records
        assert host_exact < n_miss
    if miss == 0:
        idx = eng.keyset_lookup(ks, w["rec"][:, :49])
        assert (idx != MISS).all()
        sigs = np.ascontiguousarray(w["rec"][:, 49:])
        assert np.array_equal(eng.verify_registered_many(ks, sigs, idx, w["blob"], w["off"]), want)
        assert eng.last_exact_count() == host_exact


def test_exact_only_gives_the_same_verdicts(eng):
    w = keyed_workload(eng, 400, 5000)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    fast = eng.verify_keyed_registered_many(ks, w["rec"], w["blob"], w["off"])
    eng.set_exact_only(True)
    try:
        exact = eng.verify_keyed_registered_many(ks, w["rec"], w["blob"], w["off"])
        assert eng.last_exact_count() == 0
    finally:
        eng.set_exact_only(False)
    assert np.array_equal(fast, exact) and np.array_equal(fast, expected(eng, w, oracle_sample=512))


def test_dev_forms_equal_the_host_forms(eng):
    import torch
    n = 3000
    w = keyed_workload(eng, 500, n)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    dev = torch.device("cuda", 0)
    t_rec = torch.from_numpy(w["rec"]).to(dev)
    t_blob, t_off = torch.from_numpy(w["blob"]).to(dev), torch.from_numpy(w["off"].view(np.int64)).to(dev)
    t_key = torch.from_numpy(np.ascontiguousarray(w["rec"][:, :49])).to(dev)
    out = torch.full((n,), 255, dtype=torch.uint8, device=dev)
    idx = torch.full((n,), 7, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    eng.verify_keyed_registered_many_dev(ks, n, t_rec, t_blob, t_off, out)
    eng.keyset_lookup_dev(ks, n, t_key, idx)
    eng.synchronize()
    assert np.array_equal(out.cpu().numpy(), eng.verify_keyed_registered_many(ks, w["rec"], w["blob"], w["off"]))
    assert np.array_equal(idx.cpu().numpy().view(np.uint32), eng.keyset_lookup(ks, w["rec"][:, :49]))
    assert np.array_equal(out.cpu().numpy(), expected(eng, w, oracle_sample=512))


def test_multi_device_context_equals_one_device(eng):
    import schnorr_sig_b200 as s
    multi = s.Engine([0, 0])
    n = 20000
    w = keyed_workload(eng, 600, n)
    ks1, st1 = eng.register_keys(w["pk"], w["inf"])
    ks2, st2 = multi.register_keys(w["pk"], w["inf"])
    assert np.array_equal(st1, st2)
    one = eng.verify_keyed_registered_many(ks1, w["rec"], w["blob"], w["off"])
    two = multi.verify_keyed_registered_many(ks2, w["rec"], w["blob"], w["off"])
    assert np.array_equal(one, two) and np.array_equal(one, expected(eng, w, oracle_sample=512))
    assert np.array_equal(eng.keyset_lookup(ks1, w["rec"][:, :49]), multi.keyset_lookup(ks2, w["rec"][:, :49]))
    with pytest.raises(s.EngineError):                      # device buffers need a single-device context
        multi.verify_keyed_registered_many_dev(ks2, 1, 1, 1, 1, 1)
    with pytest.raises(s.EngineError):
        multi.keyset_lookup_dev(ks2, 1, 1, 1)
    ks2.close()
    multi.close()


def test_argument_errors(eng):
    import schnorr_sig_b200 as s
    L = s._lib.lib()
    w = keyed_workload(eng, 700, 8, n_keys=4)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    other = s.Engine(0)
    ks_other, _ = other.register_keys(w["pk"], w["inf"])
    launches = eng.launch_count
    with pytest.raises(s.EngineError):
        eng.verify_keyed_registered_many(ks_other, w["rec"], w["blob"], w["off"])
    with pytest.raises(s.EngineError):
        eng.keyset_lookup(ks_other, w["rec"][:, :49])
    out = np.full(8, 77, np.uint8)
    idx = np.full(8, 77, np.uint32)
    keys = np.ascontiguousarray(w["rec"][:, :49])
    h = eng._h
    ptr = lambda a: C.c_void_p(a.ctypes.data)       # noqa: E731
    args = [ptr(w["rec"]), ptr(w["blob"]), ptr(w["off"]), ptr(out)]
    for fn in (L.schnorr_b200_verify_keyed_registered_many, L.schnorr_b200_verify_keyed_registered_many_dev):
        assert fn(h, ks_other.handle, 8, *args) == EARG
        assert fn(h, None, 8, *args) == EARG
        for k in range(4):
            bad = list(args)
            bad[k] = None
            assert fn(h, ks.handle, 8, *bad) == EARG
        assert fn(h, ks.handle, 0, None, None, None, None) == 0
        assert fn(h, ks.handle, 0, *args) == 0
    for fn in (L.schnorr_b200_keyset_lookup, L.schnorr_b200_keyset_lookup_dev):
        assert fn(h, ks_other.handle, 8, ptr(keys), ptr(idx)) == EARG
        assert fn(h, None, 8, ptr(keys), ptr(idx)) == EARG
        assert fn(h, ks.handle, 8, None, ptr(idx)) == EARG
        assert fn(h, ks.handle, 8, ptr(keys), None) == EARG
        assert fn(h, ks.handle, 0, None, None) == 0
    assert eng.launch_count == launches and (out == 77).all() and (idx == 77).all()   # nothing launched or written
    ks_other.close()
    other.close()


def test_lookup_against_a_dictionary_and_batches(eng):
    rng = np.random.default_rng(800)
    w = keyed_workload(eng, 800, 4000)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    want = findable_model(eng, w["pk"], w["inf"])
    enc = eng.compress(w["pk"], w["inf"])
    queries = [bytes(k) for k in w["rec"][:, :49]] + [bytes(e) for e in enc]
    for e in enc[:40]:
        e = bytes(e)
        queries += [e[:48] + bytes([e[48] ^ 0x40]), e[:48] + bytes([e[48] | 0x20]), e[:48] + bytes([e[48] | 0x01])]
    queries += [bytes(rng.integers(0, 256, 49, dtype=np.uint8)) for _ in range(500)]
    q = np.stack([np.frombuffer(x, np.uint8) for x in queries])
    got = eng.keyset_lookup(ks, q)
    assert [int(v) for v in got] == [want.get(x, MISS) for x in queries]
    assert len(want) < len(w["pk"]) and (got != MISS).sum() > 3000
    # indices from the lookup feed the registered batch: equal to verify_batch on the decompressed keys
    n = 4000
    idx = got[:n]
    hit = np.nonzero(idx != MISS)[0]
    sigs = np.ascontiguousarray(w["rec"][hit, 49:])
    msgs = [bytes(w["blob"][int(w["off"][i]):int(w["off"][i + 1])]) for i in hit]
    blob, off = pack_msgs(msgs)
    rand = rand_scalars(rng, len(hit))
    dpk, dinf, ok = eng.decompress(np.ascontiguousarray(w["rec"][hit, :49]))
    assert ok.all()
    for sub in (slice(0, 300), slice(0, len(hit))):
        m = len(range(len(hit))[sub])
        o_off = off[:m + 1]
        a = eng.verify_batch_registered(ks, sigs[sub], idx[hit][sub], blob[:int(o_off[-1])], o_off, rand[sub])
        b = eng.verify_batch(sigs[sub], dpk[sub], dinf[sub], blob[:int(o_off[-1])], o_off, rand[sub])
        assert a[0] == b[0] and bytes(a[1]) == bytes(b[1]) and bytes(a[2]) == bytes(b[2])


def test_python_keyset_api():
    import schnorr_sig_b200 as s
    kp = [s.KeyPair.new() for _ in range(3)]
    other = s.KeyPair.new()
    ks = s.KeySet([kp[0].public_key, kp[1].public_key, kp[1].public_key, kp[2].public_key])
    assert ks.index_of(kp[1].public_key) == 1 and ks.index_of(kp[2].public_key.to_bytes()) == 3
    assert ks.index_of(other.public_key) is None
    assert ks.index_of(bytes(48) + b"\x01") is None
    keyed = kp[2].sign_and_bind_pkey(b"hello")
    assert ks.verify_keyed(keyed, b"hello").is_ok()
    assert ks.verify_keyed(keyed.to_bytes(), b"hello!").unwrap_err() == s.SignatureError(s.SignatureError.InvalidSignature)
    outside = other.sign_and_bind_pkey(b"hello")
    assert ks.verify_keyed(outside, b"hello").is_ok()
    bad = bytearray(keyed.to_bytes())
    bad[48] |= 1                                              # the key does not decode: KeyedSignature::from_bytes fails
    with pytest.raises(s.PanicError):
        ks.verify_keyed(bytes(bad), b"hello")


CPP = r"""
#include <cstdio>
#include <random>
#include "schnorr_b200.hpp"
using namespace schnorr_sig;
int main() {
    Engine& eng = Engine::instance();
    std::mt19937_64 gen(5);
    const size_t K = 3;
    std::vector<uint8_t> sk(K * 32), pk(K * 96), inf(K, 0);
    for (auto& b : sk) b = (uint8_t)gen();
    for (size_t k = 0; k < K; k++) sk[k * 32 + 31] &= 0x3f;
    eng.check(schnorr_b200_keygen(eng.get(), K, sk.data(), pk.data(), inf.data()), "keygen");
    std::vector<PublicKey> keys(K);
    for (size_t k = 0; k < K; k++) std::memcpy(keys[k].xy.data(), &pk[k * 96], 96);
    KeySet ks(std::vector<PublicKey>{keys[0], keys[1]});
    bool ok = ks.index_of(keys[1]) == std::optional<uint32_t>(1) && !ks.index_of(keys[2]).has_value();
    std::vector<uint8_t> msg = {1, 2, 3};
    for (size_t k = 0; k < K; k++) {
        uint8_t nonce[32];
        for (auto& b : nonce) b = (uint8_t)gen();
        nonce[31] &= 0x3f;
        uint64_t off[2] = {0, msg.size()};
        std::array<uint8_t, 81> raw{};
        eng.check(schnorr_b200_sign_many(eng.get(), 1, &sk[k * 32], &pk[k * 96], &inf[k], msg.data(), off, nonce, raw.data()),
                  "sign");
        KeyedSignature ksig{keys[k], Signature::from_raw(raw)};
        ok &= !ks.verify_keyed(ksig, msg).has_value();
        std::vector<uint8_t> other = {1, 2, 4};
        Result r = ks.verify_keyed(ksig.to_bytes(), other);
        ok &= r.has_value() && *r == SignatureError::InvalidSignature;
    }
    std::printf("%s\n", ok ? "ok" : "FAILED");
    return ok ? 0 : 1;
}
"""


def test_cpp_facade(tmp_path):
    import schnorr_sig_b200 as s
    so = s._lib.library_path()
    s._lib.lib()
    src = tmp_path / "keyset_keyed.cpp"
    src.write_text(CPP)
    exe = tmp_path / "keyset_keyed"
    cudalib = "/usr/local/cuda/lib64"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include",
                           str(src), "-o", str(exe), "-L" + os.path.dirname(so), "-l:" + os.path.basename(so),
                           "-Wl,-rpath," + os.path.dirname(so), "-L" + cudalib, "-lcudart", "-Wl,-rpath," + cudalib])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr


def test_full_size(eng):
    """2^20 records under 1024 keys, one invalid signature per 1024: every verdict equals verify_keyed_many's, a sample
    the oracle's."""
    import schnorr_sig_b200 as s
    n, K = 1 << 20, 1024
    w = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED, K)
    idx = np.random.default_rng(13).integers(0, K, n).astype(np.uint32)
    blob, off = s.synth.messages(s.synth.DEFAULT_SEED, 99, n, 8)
    sigs = eng.sign_many(w["sk"][idx], w["pk"][idx], w["inf"][idx], blob, off, s.synth.scalars(s.synth.DEFAULT_SEED, 98, n))
    for i in range(512, n, 1024):
        sigs[i, 49] ^= 1
    rec = np.ascontiguousarray(np.concatenate([eng.compress(w["pk"], w["inf"])[idx], sigs], axis=1))
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    got = eng.verify_keyed_registered_many(ks, rec, blob, off)
    want = expected(eng, dict(rec=rec, blob=blob, off=off), oracle_sample=2048)
    assert np.array_equal(got, want)
    assert (want == 2).sum() == n // 1024 and (want == 0).sum() == n - n // 1024
