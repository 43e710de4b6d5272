"""Registered calls of a few signatures on one thread block per signature (k_verify_reg_one, one_reg.cuh): verdicts equal,
byte for byte, verify_many's on the gathered key records and the oracle's, whichever of the two registered kernels
set_one_threshold selects; the block kernel hands to the exact kernel only what k_verify_one hands back; its point
stage on planned challenges (the debug hook) is h*P + e*G."""
import numpy as np
import pytest

import cref
import registered_one_model as RM
import verify_exceptional_model as M
from test_gpu_registered import expected, keyset_workload
from test_gpu_verify_exceptional import embedded
from util import pack_msgs, rand_scalars

pytestmark = pytest.mark.gpu

Q = M.Q


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    return s.default_engine(0)


@pytest.fixture(autouse=True)
def defaults(eng):
    yield
    eng.set_exact_only(False)
    eng.set_dist_threshold(10240)
    eng.set_one_threshold(512)


def lens_for(n):
    lens = [(0, 7, 14, 8, 3, 21)[i % 6] for i in range(n)]
    lens[n // 2] = 10240                     # one 10 KB message
    return lens


def workload(eng, n, seed):
    w = keyset_workload(eng, seed, 16, n, lens=lens_for(n))
    if n >= 2:
        w["idx"][n - 1] = w["n_keys"] + 3    # an index outside the set
    return w


def identity_items(w):
    idx = w["idx"]
    inr = idx < w["n_keys"]
    return int(np.sum(w["inf"][np.where(inr, idx, 0)][inr] != 0))


@pytest.mark.parametrize("n", [1, 2, 31, 32, 127, 128, 129, 512])
def test_small_calls_match_verify_many_and_oracle(eng, n):
    w = workload(eng, n, 300 + n)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    try:
        got = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        assert np.array_equal(got, expected(eng, w))
        assert eng.last_exact_count() == identity_items(w)
        assert eng.last_kernel_ms() > 0
    finally:
        ks.close()


@pytest.mark.parametrize("n", [1000, 5000])
def test_block_and_thread_kernels_agree(eng, n):
    w = workload(eng, n, 500 + n)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    try:
        eng.set_one_threshold(0)
        thread = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        eng.set_one_threshold(2**62)
        block = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        assert eng.last_exact_count() == identity_items(w)
        assert np.array_equal(thread, block)
        assert np.array_equal(block, expected(eng, w, oracle_sample=512))
    finally:
        ks.close()


@pytest.mark.parametrize("where", ["alone", "embedded"])
def test_exceptional_signatures_on_the_block_kernel(eng, where):
    """Planned collisions, R = O and small-order keys (status 1) with the block kernel forced: oracle verdicts, and no
    item handed back (no identity key among them)."""
    if where == "alone":
        items = M.sig_cases()
        arrays = M.case_arrays(items)
    else:
        arrays, items = embedded()
    sigs, pk, inf, blob, off = arrays
    want = cref.verify_many(*arrays, cref.default_threads())
    keys, idx = np.unique(pk, axis=0, return_inverse=True)
    ks, _ = eng.register_keys(keys, np.zeros(len(keys), dtype=np.uint8))
    try:
        eng.set_one_threshold(2**62)
        got = eng.verify_registered_many(ks, sigs, idx.astype(np.uint32).reshape(-1), blob, off)
        bad = np.nonzero(got != want)[0]
        assert not len(bad), [(items[i].name, got[i], want[i]) for i in bad[:8]]
        assert eng.last_exact_count() == 0
        keyed = np.ascontiguousarray(np.concatenate([np.stack([cref.compress(p) for p in pk]), sigs], axis=1))
        got = eng.verify_keyed_registered_many(ks, keyed, blob, off)
        assert np.array_equal(got, want)
        assert eng.last_exact_count() == 0
    finally:
        ks.close()


def hook_cases():
    """(name, h, e) on a key a*G: edge challenges, planned digits, e*G = +-h*P, and the challenge whose two halves are
    the same multiple of the key (a doubling at the last level of the tree)."""
    rng = np.random.default_rng(21)
    a = int.from_bytes(rng.bytes(32), "little") % Q

    def r():
        return int.from_bytes(rng.bytes(32), "little") % Q

    h_zero_windows = RM.from_digits([0] * 8 + [5] + [0] * 15 + [-3] + [0] * 6 + [1])
    h_128 = RM.from_digits([128, -127, 128, 0] * 7 + [128, 0, -127, 1])
    h_same, _, _ = RM.plan_same_halves()
    cases = [("h0", 0, r()), ("h0_e0", 0, 0), ("e0", r(), 0), ("zero_windows", h_zero_windows, r()),
             ("digits_128_carry", h_128, r()), ("same_halves", h_same, r()), ("same_halves_e0", h_same, 0),
             ("q-1", Q - 1, r())]
    for name, h in (("random", r()), ("zero_windows", h_zero_windows), ("same_halves", h_same)):
        cases.append(("eG=hP_" + name, h, h * a % Q))
        cases.append(("eG=-hP_" + name, h, -h * a % Q))
    for name, h, _ in cases:
        assert 0 <= h < Q, name
        assert RM.from_digits(RM.recode(h)) == h
    return a, cases


@pytest.mark.parametrize("core", ["thread", "block"])
def test_hook_planned_challenges(eng, core):
    a, cases = hook_cases()
    base = M.base_of(1)
    pk = base.point(a)[0]
    # the key at index 1 of a set of three, so that the index reaches the table
    other = base.point(12345)[0]
    ks, status = eng.register_keys(np.stack([other, pk, other]))
    try:
        assert list(status) == [0, 0, 0]
        h = np.stack([M._le32(hh) for _, hh, _ in cases])
        e = np.stack([M._le32(ee) for _, _, ee in cases])
        res, r97 = eng.debug_verify_registered_core(ks, core, np.ones(len(cases), np.uint32), h, e)
        for i, (name, hh, ee) in enumerate(cases):
            want = M.reg_core(a, hh, ee, base)[0] if core == "thread" else M.TF
            assert res[i] == want, (name, res[i], want)
            if want != M.EXC:
                pt, inf = M.oracle_r(base, a, hh, ee)
                assert r97[i, 96] == inf, name
                if not inf:
                    assert bytes(r97[i, :96]) == bytes(pt), name
    finally:
        ks.close()


def test_hook_rejects_bad_arguments(eng):
    import schnorr_sig_b200 as s
    ks, _ = eng.register_keys(M.base_of(1).point(7)[0][None])
    z = np.zeros((1, 32), dtype=np.uint8)
    try:
        with pytest.raises(s.EngineError):
            eng.debug_verify_registered_core(ks, 2, np.zeros(1, np.uint32), z, z)
        with pytest.raises(s.EngineError):
            eng.debug_verify_registered_core(ks, "block", np.ones(1, np.uint32), z, z)
    finally:
        ks.close()


def honest(eng, n, seed, n_keys=8):
    rng = np.random.default_rng(seed)
    sk = rand_scalars(rng, n_keys)
    pk, inf = eng.keygen(sk)
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    blob, off = pack_msgs([rng.bytes(int(L)) for L in rng.integers(0, 40, n)])
    sigs = eng.sign_many(sk[idx], pk[idx], inf[idx], blob, off, rand_scalars(rng, n))
    rec = np.ascontiguousarray(np.concatenate([eng.compress(pk[idx], inf[idx]), sigs], axis=1))
    return dict(pk=pk, inf=inf, idx=idx, sigs=sigs, blob=blob, off=off, rec=rec, rng=rng)


@pytest.mark.parametrize("kind", ["all_found", "one_miss", "undecodable"])
def test_keyed_host_form(eng, kind):
    n = 64
    w = honest(eng, n, 41)
    rec = w["rec"].copy()
    if kind == "one_miss":
        pk2, inf2 = eng.keygen(rand_scalars(w["rng"], 1))
        rec[5, :49] = eng.compress(pk2, inf2)[0]            # a valid key outside the set
    elif kind == "undecodable":
        rec[9, :48] = 0xFF                                   # non-canonical limbs: the key does not decode
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    try:
        want = eng.verify_keyed_many(rec, w["blob"], w["off"])
        got = eng.verify_keyed_registered_many(ks, rec, w["blob"], w["off"])
        assert np.array_equal(got, want)
        if kind == "all_found":
            assert (want == 0).all()
        elif kind == "one_miss":
            assert want[5] == 2 and (np.delete(want, 5) == 0).all()
        else:
            assert want[9] == 3 and (np.delete(want, 9) == 0).all()
        if kind != "undecodable":                            # (an undecodable key is verified as the identity, then masked)
            assert eng.last_exact_count() == 0
    finally:
        ks.close()


def test_dev_forms(eng):
    import torch
    n = 96
    w = honest(eng, n, 43)
    w["sigs"][3, 49:] = 0                                   # e := 0: an invalid signature
    w["rec"][3, 49:] = w["sigs"][3]
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    try:
        host = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        keyed_host = eng.verify_keyed_registered_many(ks, w["rec"], w["blob"], w["off"])
        assert np.array_equal(host, keyed_host) and host[3] == 2 and (np.delete(host, 3) == 0).all()
        dev = torch.device("cuda", 0)
        t_sig, t_idx = torch.from_numpy(w["sigs"]).to(dev), torch.from_numpy(w["idx"].view(np.int32)).to(dev)
        t_rec = torch.from_numpy(w["rec"]).to(dev)
        t_blob, t_off = torch.from_numpy(w["blob"]).to(dev), torch.from_numpy(w["off"].view(np.int64)).to(dev)
        out1 = torch.full((n,), 255, dtype=torch.uint8, device=dev)
        out2 = torch.full((n,), 255, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        eng.verify_registered_many_dev(ks, n, t_sig, t_idx, t_blob, t_off, out1)
        eng.verify_keyed_registered_many_dev(ks, n, t_rec, t_blob, t_off, out2)
        eng.synchronize()
        assert np.array_equal(out1.cpu().numpy(), host)
        assert np.array_equal(out2.cpu().numpy(), keyed_host)
    finally:
        ks.close()


def test_exact_only(eng):
    n = 600
    w = workload(eng, n, 77)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    try:
        want = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        assert np.array_equal(want, expected(eng, w, oracle_sample=256))
        eng.set_exact_only(True)
        assert np.array_equal(eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"]), want)
    finally:
        ks.close()


def test_multi_device_slices_pick_their_own_kernel(eng):
    """One GPU listed twice: calls below 2 x 4096 items stay on the first device, so 8192 items make two 4096-item
    slices; with one_max = 4096 each slice takes the block kernel although the whole call is larger."""
    import schnorr_sig_b200 as s
    n = 8192
    w = workload(eng, n, 79)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    try:
        want = eng.verify_registered_many(ks, w["sigs"], w["idx"], w["blob"], w["off"])
        assert np.array_equal(want, expected(eng, w, oracle_sample=256))
    finally:
        ks.close()
    h = honest(eng, n, 81)
    keyed_want = eng.verify_keyed_many(h["rec"], h["blob"], h["off"])
    multi = s.Engine([0, 0])
    try:
        multi.set_one_threshold(4096)
        ks2, _ = multi.register_keys(w["pk"], w["inf"])
        try:
            got = multi.verify_registered_many(ks2, w["sigs"], w["idx"], w["blob"], w["off"])
            assert np.array_equal(got, want)
            assert multi.last_exact_count() == identity_items(w)
            assert multi.last_kernel_ms() > 0
        finally:
            ks2.close()
        ks2, _ = multi.register_keys(h["pk"], h["inf"])
        try:
            got = multi.verify_keyed_registered_many(ks2, h["rec"], h["blob"], h["off"])
            assert np.array_equal(got, keyed_want)
            assert multi.last_exact_count() == 0
        finally:
            ks2.close()
    finally:
        multi.close()
