"""The device field core (csrc/fp.cuh) word for word, through the schnorr_b200_debug_fp_core test hook: every op on
inputs built to reach each carry and borrow path of its reductions (tests/fp_core_cases.py), checked against Python
integers and, bit for bit, against the CPU model of the PTX (tests/ptx_model.py).  The model comparison pins the
exact non-canonical representatives and accumulator states, and ties the model's reading of the PTX to the
hardware: a wrong assumption about an instruction, or a miscompile, shows up as a mismatch."""
import numpy as np
import pytest

import fp_core_cases as fc
import ptx_model as pm
from ptx_model import M64, P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    import schnorr_sig_b200 as s
    return s.default_engine(0)


@pytest.fixture(scope="module")
def cases():
    return fc.cases(seed=7, n_random=2)


def run(eng, op, items):
    out = eng.debug_fp_core(op, np.array([fc.pack(op, a) for a in items], dtype=np.uint32))
    return [[int(v) for v in row] for row in out]


@pytest.mark.parametrize("op", fc.OPS)
def test_device_matches_integers_and_model(eng, cases, op):
    core = pm.FpCore()
    items = cases[op]
    wrong, differ = [], []
    for args, got in zip(items, run(eng, op, items)):
        err = fc.check(op, args, got)
        if err:
            wrong.append((args, err))
        want = core.op(op, args)
        if got != want:
            differ.append((args, got, want))
    assert not wrong, "%s: %d of %d results wrong, first: %s" % (op, len(wrong), len(items), wrong[:3])
    assert not differ, "%s: %d of %d results differ from the PTX model, first: %s" % (op, len(differ), len(items),
                                                                                     differ[:3])


def test_long_accumulation_to_the_limit(eng):
    """2^20 products on the device from the exact state 2^20 products short of the documented 2^30 limit."""
    n = 1 << 20
    pairs = [(M64, M64), (P - 1, P - 1), (M64, 2**63), (0xFEDCBA9876543210, 0xFFFFFFFF00000000)]
    items = [(fc.state_after(fc.WIDE_MAX_PRODUCTS - n, a, b), a, b, n) for a, b in pairs]
    for (w, a, b, _), got in zip(items, run(eng, "wide_mac_loop", items)):
        assert tuple(got[:8]) == fc.state_after(fc.WIDE_MAX_PRODUCTS, a, b), (a, b)
        want = fc.WIDE_MAX_PRODUCTS * a * b % P
        assert pm.join(got[8], got[9]) % P == want and pm.join(got[10], got[11]) == want, (a, b)


def test_bad_arguments_are_rejected(eng):
    import schnorr_sig_b200 as s
    x = np.zeros((1, 16), dtype=np.uint32)
    for op in (-1, len(fc.OPS)):
        with pytest.raises(s.EngineError, match=r"\(-1\)"):
            eng.debug_fp_core(op, x)
    assert eng.debug_fp_core("mul", np.zeros((0, 16), dtype=np.uint32)).shape == (0, 16)
