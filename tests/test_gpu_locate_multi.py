"""Failed-batch localisation over the devices of a multi-device context, and the seeded localisations.

The tree of the bisection is defined by n alone (schnorr-sig_b200/csrc/locate_plan.h, model-checked on the CPU by
tests/test_locate_plan_hostsim.py): the flags and n_bad of every host form on a context of 2, 3, 8 or 9 devices must be
those of a single-device context, byte for byte.  On a box with fewer GPUs the device list wraps around (independent
contexts on the same GPU), which runs the same sharded code.  The seeded forms must equal their parents fed with
rand32 = batch_randomizers(seed, 0, n), on one device and on three."""
import ctypes as C

import numpy as np
import pytest

import test_batch_exceptional_model as M
from test_gpu_keyed_registered import keyed_workload
from test_gpu_registered import keyset_workload
from util import KAT96, make_workload, pack_msgs

pytestmark = pytest.mark.gpu

DEVICES = [2, 3, 8, 9]
EARG = -1


def _device_list(want):
    import torch
    c = torch.cuda.device_count()
    return [k % c for k in range(want)]


@pytest.fixture(scope="module")
def engines():
    import schnorr_sig_b200 as s
    one = s.Engine(0)
    multi = {d: s.Engine(_device_list(d)) for d in DEVICES}
    yield one, multi
    for e in multi.values():
        e.close()
    one.close()


def seed_of(k):
    return np.random.default_rng(7000 + k).integers(0, 256, 32, dtype=np.uint8).tobytes()


def locate(e, w, sigs=None, pk=None):
    """schnorr_b200_locate_invalid -> (flags, n_bad)"""
    sigs = np.ascontiguousarray(w["sigs"] if sigs is None else sigs)
    pk = np.ascontiguousarray(w["pk"] if pk is None else pk)
    n = sigs.shape[0]
    flags = np.zeros(n, dtype=np.uint8)
    nb = C.c_uint64(12345)
    p = lambda a: C.c_void_p(a.ctypes.data)    # noqa: E731
    rc = e._L.schnorr_b200_locate_invalid(e._h, n, p(sigs), p(pk), p(w["inf"]), p(w["blob"]), p(w["off"]), p(w["rand"]),
                                          p(flags), C.byref(nb))
    assert rc == 0, rc
    return flags, int(nb.value)


def same_everywhere(engines, call):
    """call(engine) on the single-device context and on every multi-device one: equal results; returns it."""
    one, multi = engines
    want = call(one)
    for d, e in multi.items():
        got = call(e)
        if isinstance(want, tuple):
            assert all(np.array_equal(a, b) for a, b in zip(got, want)), d
        else:
            assert np.array_equal(got, want), d
    return want


def splice(w, placed):
    """w with rows replaced: placed = {position: (source workload, source row)}; messages repacked."""
    out = {k: w[k].copy() for k in ("sigs", "pk", "inf", "rand")}
    msgs = [bytes(w["blob"][int(w["off"][i]):int(w["off"][i + 1])]) for i in range(len(w["sigs"]))]
    for pos, (src, j) in placed.items():
        for k in ("sigs", "pk", "inf", "rand"):
            out[k][pos] = src[k][j]
        msgs[pos] = bytes(src["blob"][int(src["off"][j]):int(src["off"][j + 1])])
    out["blob"], out["off"] = pack_msgs(msgs)
    return out


# ---- 1. the culprit kinds of test_gpu_locate.py ------------------------------------------------------------------------
def test_every_kind_of_culprit(engines):
    n = 40000
    w = make_workload(37, n, msg_len=8)
    sigs, pk = w["sigs"].copy(), w["pk"].copy()
    culprits = {}
    rng = np.random.default_rng(5)
    for k, i in enumerate(sorted(int(v) for v in rng.choice(n - 1, 60, replace=False))):
        kind = k % 5
        if kind == 0:
            sigs[i, 49 + 3] ^= 0x10                  # e changed
        elif kind == 1:
            sigs[i, 48] ^= 0x40                      # y-sign flag flipped
        elif kind == 2:
            pk[i] = KAT96                            # off-subgroup key
        elif kind == 3:
            pk[i] = w["pk"][(i + 1) % n]             # another signer's key
        else:
            sigs[i, 48] = 0x07                       # reserved flag bits: malformed
        culprits[i] = 3 if kind == 4 else 2
    flags, nb = same_everywhere(engines, lambda e: locate(e, w, sigs, pk))
    assert {int(i): int(flags[i]) for i in np.nonzero(flags)[0]} == culprits and nb == len(culprits)


@pytest.mark.parametrize("where", ["first", "last", "clean"])
def test_one_culprit_in_the_first_and_last_level2_part(engines, where):
    import schnorr_sig_b200 as s
    n = 1 << 17
    w = s.synth.signed_workload(engines[0], 0x10CA7E, n, msg_len=8)
    sigs = w["sigs"].copy()
    want = {"first": [3], "last": [n - 2], "clean": []}[where]
    for i in want:
        sigs[i, 49] ^= 1
    flags, nb = same_everywhere(engines, lambda e: locate(e, w, sigs))
    assert list(np.nonzero(flags)[0]) == want and nb == len(want)


def test_one_in_40_takes_the_per_item_path(engines):
    import schnorr_sig_b200 as s
    n = 1 << 15
    w = s.synth.signed_workload(engines[0], 0x10CA7E + 15, n, msg_len=8)
    sigs = w["sigs"].copy()
    want = list(range(7, n, 40))
    sigs[want, 49] ^= 1
    flags, nb = same_everywhere(engines, lambda e: locate(e, w, sigs))
    assert list(np.nonzero(flags)[0]) == want and nb == len(want)


# ---- 2. torsion-shifted culprits and cancelling pairs ------------------------------------------------------------------
@pytest.fixture(scope="module")
def torsion():
    """Two independent torsion-culprit cases (one TORSION_ODD item each) and the two-torsion case."""
    a, ka, _, _ = M.case_torsion_culprits(400, 40, 400)
    b, kb, _, _ = M.case_torsion_culprits(400, 40, 401)
    return a, ka, b, kb, M.case_two_torsion()


def test_torsion_culprits_inside_one_part_and_across_the_boundaries(engines, torsion):
    import schnorr_sig_b200 as s
    a, ka, b, kb, two = torsion
    n = 1 << 15
    step = n // 8                                # level-2 parts; 2 and 8 devices own blocks of them
    fill = s.synth.signed_workload(engines[0], 0x70551, n, msg_len=8)
    odd_a, odd_b = int(np.nonzero(ka == M.TORSION_ODD)[0][0]), int(np.nonzero(kb == M.TORSION_ODD)[0][0])
    wrong_e = [int(i) for i in np.nonzero(ka == M.WRONG_E)[0]]
    quiet = [int(i) for i in np.nonzero(np.isin(ka, [M.TORSION_EVEN, M.ZERO_RAND]))[0]]
    cases = {
        # T2 + T2 = O inside one part, beside a wrong e in another: the pair is never flagged
        "pair_inside": ({100: (a, odd_a), 300: (b, odd_b), n - 5: (a, wrong_e[0])}, [n - 5]),
        # the same pair across the level-2 boundary in the middle (an ownership boundary on 2 and 8 devices)
        "pair_across": ({4 * step - 1: (a, odd_a), 4 * step: (b, odd_b), 17: (a, wrong_e[0])}, [17, 4 * step - 1, 4 * step]),
        # items whose own term is O (even randomiser on a torsion shift, randomiser 0) on every boundary
        "quiet": ({k * step + d: (a, quiet[(2 * k + d + 1) % len(quiet)]) for k in range(1, 8) for d in (-1, 0)}
                  | {5 * step + 9: (a, wrong_e[1])}, [5 * step + 9]),
        # the pair with nothing else wrong: the whole batch passes
        "pair_only": ({step - 1: (a, odd_a), step: (b, odd_b)}, []),
        # the two-torsion items across the boundary in the middle and at the ends
        "two_torsion": ({4 * step - 3 + j: (two, j) for j in range(6)} | {0: (a, odd_a), n - 1: (a, wrong_e[2])}, None),
    }
    for name, (placed, want) in cases.items():
        w = splice(fill, placed)
        flags, nb = same_everywhere(engines, lambda e: locate(e, w))
        if want is not None:
            assert list(np.nonzero(flags)[0]) == sorted(want) and (flags[want] == 2).all(), name
        assert nb == int(np.count_nonzero(flags)), name


# ---- 3. the other three forms ------------------------------------------------------------------------------------------
def test_registered_with_a_removed_index_and_a_status_1_key(engines):
    one, multi = engines
    n = 1 << 15
    w = keyset_workload(one, 91, 64, n)
    rand = np.random.default_rng(93).integers(0, 256, (n, 32), dtype=np.uint8)
    rand[:, 31] &= 0x0F
    w["idx"][1234] = 7

    def call(e):
        ks, status = e.register_keys(w["pk"], w["inf"])
        try:
            assert (status[64:70] == 1).all()
            e.keyset_remove(ks, [7])                                     # item 1234 and every other user of key 7
            return e.locate_invalid_registered(ks, w["sigs"], w["idx"], w["blob"], w["off"], rand)
        finally:
            ks.close()
    flags = same_everywhere(engines, call)
    assert flags[1234] == 3 and (flags[w["idx"] == 7] == 3).all()
    assert np.count_nonzero(flags == 2) > 0


@pytest.mark.parametrize("registered", [False, True])
def test_keyed_with_undecodable_keys_hits_and_misses(engines, registered):
    one, _ = engines
    n = 1 << 15
    w = keyed_workload(one, 95, n, n_keys=64)
    rand = np.random.default_rng(96).integers(0, 256, (n, 32), dtype=np.uint8)
    rand[:, 31] &= 0x0F

    def call(e):
        if not registered:
            return e.locate_invalid_keyed(w["rec"], w["blob"], w["off"], rand)
        ks, _ = e.register_keys(w["pk"], w["inf"])
        try:
            return e.locate_invalid_keyed_registered(ks, w["rec"], w["blob"], w["off"], rand)
        finally:
            ks.close()
    flags = same_everywhere(engines, call)
    assert (flags[106::202] == 3).all()                              # keys with reserved flag bits set
    assert np.count_nonzero(flags == 2) > 0


# ---- 4. seeded localisation ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [5000, 1 << 15])
def test_seeded_forms_equal_their_parents(engines, n):
    import schnorr_sig_b200 as s
    one, multi = engines
    seed = seed_of(n)
    rand = one.batch_randomizers(n, seed)
    w = s.synth.signed_workload(one, 0x5EED + n, n, msg_len=8)
    w["sigs"][[11, n // 2, n - 1], 49] ^= 1
    kw = keyed_workload(one, 97, n, n_keys=64)
    rw = keyset_workload(one, 98, 64, n)
    for e in (one, multi[3]):
        want = e.locate_invalid(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], rand)
        assert list(np.nonzero(want)[0]) == [11, n // 2, n - 1]
        assert np.array_equal(e.locate_invalid_seeded(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], seed), want)
        want = e.locate_invalid_keyed(kw["rec"], kw["blob"], kw["off"], rand)
        assert want.any()
        assert np.array_equal(e.locate_invalid_keyed_seeded(kw["rec"], kw["blob"], kw["off"], seed), want)
        ks, _ = e.register_keys(kw["pk"], kw["inf"])
        try:
            want = e.locate_invalid_keyed_registered(ks, kw["rec"], kw["blob"], kw["off"], rand)
            got = e.locate_invalid_keyed_registered_seeded(ks, kw["rec"], kw["blob"], kw["off"], seed)
            assert np.array_equal(got, want)
        finally:
            ks.close()
        ks, _ = e.register_keys(rw["pk"], rw["inf"])
        try:
            want = e.locate_invalid_registered(ks, rw["sigs"], rw["idx"], rw["blob"], rw["off"], rand)
            assert want.any()
            got = e.locate_invalid_registered_seeded(ks, rw["sigs"], rw["idx"], rw["blob"], rw["off"], seed)
            assert np.array_equal(got, want)
        finally:
            ks.close()


def test_seeded_argument_errors(engines):
    one, multi = engines
    nb = C.c_uint64(99)
    for e in (one, multi[3]):
        L, h = e._L, e._h
        for name in ("schnorr_b200_locate_invalid_seeded", "schnorr_b200_locate_invalid_registered_seeded",
                     "schnorr_b200_locate_invalid_keyed_seeded", "schnorr_b200_locate_invalid_keyed_registered_seeded"):
            fn = getattr(L, name)
            nargs = len(fn.argtypes)
            reg = "registered" in name
            ks = None
            if reg:
                ks, _ = e.register_keys(make_workload(3, 2)["pk"])
            try:
                args = [h, 0] + [None] * (nargs - 2)
                if reg:
                    args = [h, ks.handle, 0] + [None] * (nargs - 3)
                args[nargs - 1] = C.byref(nb)
                seed_pos = nargs - 3
                assert fn(*args) == EARG, name                           # NULL seed, empty batch
                seed = np.frombuffer(seed_of(1), dtype=np.uint8).copy()
                args[seed_pos] = C.c_void_p(seed.ctypes.data)
                nb.value = 99
                assert fn(*args) == 0 and nb.value == 0, name            # n = 0: OK, no culprits
            finally:
                if ks is not None:
                    ks.close()


def test_python_seed_localisations_equal_the_rand32_path():
    import os
    import schnorr_sig_b200 as s
    from schnorr_sig_b200 import api
    kp = [s.KeyPair.new() for _ in range(3)]
    n = 9000
    idx = [i % 3 for i in range(n)]
    msgs = [b"m%d" % i for i in range(n)]
    sigs = [kp[k].sign(m) for k, m in zip(idx, msgs)]
    keys = [kp[k].public_key for k in idx]
    bad = list(keys)
    bad[5], bad[6] = bad[6], bad[5]
    bad[8500], bad[8501] = bad[8501], bad[8500]
    seed = os.urandom(32)
    eng = s.default_engine(0)
    rand = eng.batch_randomizers(n, seed)
    arrays = api._batch_arrays(sigs, bad, msgs)
    want = [int(i) for i in np.nonzero(eng.locate_invalid(*arrays, rand))[0]]
    assert want == [5, 6, 8500, 8501]
    assert [i for i, _ in s.locate_invalid(sigs, bad, msgs, seed=seed)] == want
    keyed = [s.KeyedSignature(k, sg) for k, sg in zip(bad, sigs)]
    assert [i for i, _ in s.locate_invalid_keyed(keyed, msgs, seed=seed)] == want
    ks = s.KeySet([k.public_key for k in kp])
    bad_idx = list(idx)
    bad_idx[5], bad_idx[6] = bad_idx[6], bad_idx[5]
    bad_idx[8500], bad_idx[8501] = bad_idx[8501], bad_idx[8500]
    assert [i for i, _ in ks.locate_invalid(bad_idx, sigs, msgs, seed=seed)] == want
    assert [i for i, _ in ks.locate_invalid_keyed(keyed, msgs, seed=seed)] == want
