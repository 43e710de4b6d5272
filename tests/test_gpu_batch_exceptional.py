"""Batch verification on exceptional group elements, on the device, against the oracle.

The inputs come from test_batch_exceptional_model.py: every point a multiple of one base point, so that cancelling,
doubling and small-order values land in chosen stages of the pipeline (buckets, segments, window sums, the fold, Horner,
the block-per-signature form, the registered key side, partials).  Each case asserts (verdict, lhs97, rhs97) byte-equal
to cref.verify_batch, and that the device ran the plan (last_batch_plan, last_batch_points) in which the model placed
its events; test_batch_exceptional_model.py checks, without a GPU, that those events happen under that plan.
"""
import numpy as np
import pytest

import cref
import test_batch_exceptional_model as M

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    return s.default_engine(0)


@pytest.fixture(autouse=True)
def defaults(eng):
    yield
    eng.set_msm_geometry(0, 0)
    eng.set_batch_small_threshold(256)
    eng.set_batch_dist_threshold(2**18)
    eng.set_registered_batch_threshold(64)


# (name, batch_small_threshold): the default, Pippenger forced, one block per signature forced
FORMS = [("default", 256), ("msm", 0), ("small", 2**62)]


def _same(got, want):
    assert got[0] == want[0], (got[0], want[0])
    assert (got[1] == want[1]).all(), "lhs differs from the oracle"
    assert (got[2] == want[2]).all(), "rhs differs from the oracle"


def run(eng, w, small_max=256, c=0, T=0, dist=True, want=None):
    """verify_batch on the device in the form `small_max` selects; checks the oracle and the plan of the model."""
    eng.set_batch_small_threshold(small_max)
    eng.set_batch_dist_threshold(2**18 if dist else 0)
    eng.set_msm_geometry(c, T)
    got = eng.verify_batch(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], w["rand"])
    want = M.oracle(w) if want is None else want
    _same(got, want)
    form = "small" if w["n"] <= small_max else "msm"
    _, _, plan, npts = M.model_run(w, form, c, T)
    assert eng.last_batch_plan() == plan
    assert eng.last_batch_points() == npts
    return got


def run_forms(eng, w, c=0, T=0):
    want = M.oracle(w)
    for _, small_max in FORMS:
        if small_max and small_max >= 2**62 and w["n"] > 2048:
            continue                   # the block form of thousands of signatures: covered at the smaller sizes
        run(eng, w, small_max, c, T, want=want)
    run(eng, w, 0, c, T, dist=False, want=want)   # challenges hashed inside k_batch_prepare
    return want


@pytest.mark.parametrize("n", [300, 5000])
def test_rneg_pairs_cancel_in_buckets_and_double_on_the_key_side(eng, n):
    w = M.case_rneg_pairs(n, n)
    assert run_forms(eng, w)[0] == 2


def test_two_torsion_points(eng):
    run_forms(eng, M.case_two_torsion())


@pytest.mark.parametrize("m", [2, 29, 58, 181])
def test_small_order_keys_and_r(eng, m):
    run_forms(eng, M.case_small_order(m, 0))


@pytest.mark.parametrize("c", M.HORNER_C)
def test_horner_cancel_identity_and_doubling(eng, c):
    w = M.case_order29(M.HORNER_EVENTS, [("msm", c, 0)])
    run(eng, w, 0, c)


def test_window_sum_and_fold(eng):
    run_forms(eng, M.case_order29(M.WINDOW_EVENTS, [("msm", 0, 0)]))


def test_block_form_buckets_running_sums_terms_and_reduce(eng):
    w = M.case_order29(M.SMALL_EVENTS, [("small", 0, 0)])
    run(eng, w, 2**62)
    run(eng, w, 2**62, dist=False)


def test_segments_cross_and_long_buckets(eng):
    w = M.case_segments()
    want = M.oracle(w)
    run(eng, w, 0, 0, 8, want=want)
    run(eng, w, 0, 0, 8, dist=False, want=want)


@pytest.mark.parametrize("n,zero_e,verdict", [(8, True, 0), (8, False, 2), (300, True, 0)])
def test_whole_batch_identity_from_cancelling_items(eng, n, zero_e, verdict):
    w = M.case_whole_identity(n, zero_e)
    assert w["lhs"] == 0
    assert run_forms(eng, w)[0] == verdict


def _slice(w, lo, hi):
    off = w["off"][lo:hi + 1] - w["off"][lo]
    blob = w["blob"][int(w["off"][lo]):int(w["off"][hi])]
    return w["sigs"][lo:hi], w["pk"][lo:hi], w["inf"][lo:hi], blob, off, w["rand"][lo:hi]


@pytest.mark.parametrize("small_max", [256, 0])
def test_partials_identity_and_opposite(eng, small_max):
    w, na, nb = M.case_partials(64, 9)
    eng.set_batch_small_threshold(small_max)
    want = M.oracle(w)
    n = w["n"]
    for cut in ((0, na, n), (na, na + nb, n)):      # A | B C: A's partial is O;  B | C: opposite partials
        parts = np.stack([eng.batch_partial(*_slice(w, cut[0], cut[1])), eng.batch_partial(*_slice(w, cut[1], cut[2]))])
        got = eng.batch_finish(parts)
        s = _slice(w, cut[0], cut[2])
        want_sub = cref.verify_batch(*s, cref.default_threads())
        _same(got, want_sub)
    _same(eng.verify_batch(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], w["rand"]), want)


def test_two_shards_one_partial_identity():
    import schnorr_sig_b200 as s
    e2 = s.Engine([0, 0])
    try:
        w, _ = M.case_two_shards()                      # shard 0: cancelling pairs, its partial is O
        got = e2.verify_batch(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], w["rand"])
        _same(got, M.oracle(w))
        assert e2.last_batch_points() == 2 * w["n"]
    finally:
        e2.close()


def _registered(eng, keys, idx, w):
    base = w["base"]
    pk = np.stack([base.point(p)[0] for p in keys])
    ks, status = eng.register_keys(pk)
    try:
        eng.set_batch_small_threshold(0)
        eng.set_registered_batch_threshold(0)
        got = eng.verify_batch_registered(ks, w["sigs"], idx, w["blob"], w["off"], w["rand"])
        return got, status
    finally:
        ks.close()


@pytest.mark.parametrize("kind", ["cancel", "double", "zero", "large"])
def test_registered_key_side(eng, kind):
    w, keys, idx = M.case_registered(kind)
    got, status = _registered(eng, keys, idx, w)
    assert (status == 0).all()
    _same(got, M.oracle(w))                             # the oracle on the gathered records
    assert eng.last_batch_points() == w["n"]
    _, ev, plan = M.model_registered(w, keys, idx)
    assert eng.last_batch_plan() == plan
    assert M.REGISTERED_EVENTS[kind] <= ev.seen


def test_registered_set_with_a_torsion_key_takes_the_gathered_path(eng):
    w, keys, idx = M.case_registered("cancel")
    t = np.frombuffer(M.torsion(29), dtype=np.uint8)
    base = w["base"]
    pk = np.stack([base.point(p)[0] for p in keys] + [t])
    ks, status = eng.register_keys(pk)
    try:
        assert list(status) == [0, 0, 0, 1]
        eng.set_batch_small_threshold(0)
        eng.set_registered_batch_threshold(0)
        got = eng.verify_batch_registered(ks, w["sigs"], idx, w["blob"], w["off"], w["rand"])
        _same(got, M.oracle(w))
        assert eng.last_batch_points() == 2 * w["n"]
    finally:
        ks.close()


@pytest.mark.parametrize("n,density", M.LOCATE_SIZES)
def test_locate_flags_an_item_by_its_own_term(eng, n, density):
    """Items whose own term s_i D_i is O (randomiser 0; a torsion-shifted R with an even randomiser) are never flagged,
    whatever their neighbours; a torsion-shifted R with an odd randomiser and a wrong e are.  The batch itself fails
    with the oracle's points, and passes without the items that can fail it."""
    w, kinds, pool, idx = M.case_torsion_culprits(n, density, n)
    want = np.where(np.isin(kinds, [M.TORSION_ODD, M.WRONG_E]), 2, 0)
    assert run_forms(eng, w)[0] == 2
    ok = M.subset(w, np.nonzero(want == 0)[0])
    assert run_forms(eng, ok)[0] == 0
    flags = eng.locate_invalid(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], w["rand"])
    assert list(np.nonzero(flags)[0]) == list(np.nonzero(want)[0])
    assert (flags == want).all()
    for i in np.nonzero(kinds != M.CLEAN)[0][:24]:
        assert M.oracle_item(w, int(i)) == want[i]
    pk = np.stack([w["base"].point(p)[0] for p in pool])
    ks, status = eng.register_keys(pk)
    try:
        assert (status == 0).all()
        flags = eng.locate_invalid_registered(ks, w["sigs"], idx, w["blob"], w["off"], w["rand"])
        assert (flags == want).all()
    finally:
        ks.close()
