"""Single-signature verification on exceptional group elements, on the device, against the model and the oracle.

The cases come from verify_exceptional_model.py.  The hook cases (a given challenge) run through the three point cores
of schnorr_b200_debug_verify_core: the result code must be the model's and R the oracle's whenever it is not
exceptional.  The signature cases (hashed challenges: R = O, planned cancels and doublings in the e*G windows, the
same_h doubling, small-order and mixed keys) run through every kernel of the public API, alone and inside a
1000-signature honest workload: every verdict must be the oracle's, and the number of items the fast path hands to the
exact kernel the model's.  test_verify_exceptional_model.py checks the cases and the model without a GPU.
"""
import numpy as np
import pytest

import cref
import verify_exceptional_model as M
from util import pack_msgs, rand_scalars

pytestmark = pytest.mark.gpu


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


@pytest.mark.parametrize("core", ["exact", "fast", "dist"])
def test_hook_cores_agree_with_the_model(eng, core):
    cases = M.hook_cases()
    pk = np.stack([c.pk96() for c in cases])
    h = np.stack([M._le32(c.h) for c in cases])
    e = np.stack([M._le32(c.e) for c in cases])
    res, r97 = eng.debug_verify_core(core, pk, h, e)
    for i, c in enumerate(cases):
        want, r, tr = M.fast_core(c.a, c.h, c.e, c.base)
        if core == "exact":
            want = M.TF if (M.Q * c.a) % c.base.N == 0 else M.NTF
        assert res[i] == want, (c.name, res[i], want, tr.events[:3])
        if want != M.EXC:
            pt, inf = M.oracle_r(c.base, c.a, c.h, c.e)
            assert r97[i, 96] == inf, c.name
            if not inf:
                assert bytes(r97[i, :96]) == bytes(pt), c.name


def test_hook_rejects_an_unknown_core(eng):
    import schnorr_sig_b200 as s
    z = np.zeros((1, 32), dtype=np.uint8)
    with pytest.raises(s.EngineError):
        eng.debug_verify_core(3, np.zeros((1, 96), dtype=np.uint8), z, z)


# (path, setup): one signature per thread, six lanes, one block, exact only
PATHS = {
    "fast": lambda eng: (eng.set_one_threshold(0), eng.set_dist_threshold(0)),
    "dist": lambda eng: (eng.set_one_threshold(0), eng.set_dist_threshold(2**62)),
    "one": lambda eng: eng.set_one_threshold(2**62),
    "exact": lambda eng: eng.set_exact_only(True),
}
BLOCK_SLOTS = (0, 31, 32, 127)


def embedded(n=1000, seed=11, n_keys=16):
    """The signature cases at threads 0, 31, 32 and 127 of consecutive 128-thread blocks of n honest signatures under
    n_keys keys -> (arrays, the SigCase of every item)."""
    rng = np.random.default_rng(seed)
    sk = rand_scalars(rng, n_keys)
    pk, inf = cref.keygen(sk, cref.default_threads())
    owner = rng.integers(0, n_keys, n)
    msgs = [rng.bytes(8) for _ in range(n)]
    blob, off = pack_msgs(msgs)
    sigs = cref.sign_many(sk[owner], pk[owner], inf[owner], blob, off, rand_scalars(rng, n), cref.default_threads())
    dig = cref.hash_messages(sigs[:, :48], pk[owner], blob, off, cref.default_threads())
    items = [M.SigCase("honest", 1, int.from_bytes(bytes(sk[owner[i]]), "little"), sigs[i], msgs[i],
                       M.o.scalar_from_digest(bytes(dig[i])), M.OK) for i in range(n)]
    cases = M.sig_cases()
    slots = [128 * b + t for b in range(n // 128) for t in BLOCK_SLOTS][:len(cases)]
    assert len(slots) == len(cases)
    for s, c in zip(slots, cases):
        items[s] = c
    return M.case_arrays(items), items


def _check(eng, got, items, arrays, path):
    want = cref.verify_many(*arrays, cref.default_threads())
    assert not (got == 0xFF).any()
    bad = np.nonzero(got != want)[0]
    assert not len(bad), [(items[i].name, got[i], want[i]) for i in bad[:8]]
    assert eng.last_exact_count() == sum(M.expected_handback(c, path) for c in items), path


@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("where", ["alone", "embedded"])
def test_verify_many_on_every_kernel(eng, path, where):
    if where == "alone":
        items = M.sig_cases()
        arrays = M.case_arrays(items)
    else:
        arrays, items = embedded()
    PATHS[path](eng)
    _check(eng, eng.verify_many(*arrays), items, arrays, path)
    keyed = np.ascontiguousarray(np.concatenate([np.stack([cref.compress(p) for p in arrays[1]]), arrays[0]], axis=1))
    _check(eng, eng.verify_keyed_many(keyed, arrays[3], arrays[4]), items, arrays, path)


@pytest.mark.parametrize("where", ["alone", "embedded"])
def test_registered_and_keyed_registered(eng, where):
    """Keys registered in a key set: the registered kernel (k_verify_reg) above 384 signatures, verify_many's kernels
    below.  Small-order and mixed keys have status 1 and never reach the point stage there."""
    if where == "alone":
        items = M.sig_cases()
        arrays = M.case_arrays(items)
        path = "one"
    else:
        arrays, items = embedded()
        path = "reg"
    sigs, pk, inf, blob, off = arrays
    keys, idx = np.unique(pk, axis=0, return_inverse=True)
    ks, status = eng.register_keys(keys, np.zeros(len(keys), dtype=np.uint8))
    try:
        assert set(status.tolist()) <= {0, 1}
        _check(eng, eng.verify_registered_many(ks, sigs, idx.astype(np.uint32).reshape(-1), blob, off), items, arrays,
               path)
        keyed = np.ascontiguousarray(np.concatenate([np.stack([cref.compress(p) for p in pk]), sigs], axis=1))
        _check(eng, eng.verify_keyed_registered_many(ks, keyed, blob, off), items, arrays, path)
    finally:
        ks.close()
