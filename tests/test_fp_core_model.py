"""The inline PTX of the device field core (csrc/fp.cuh), run through a CPU model of its instructions
(tests/ptx_model.py), against Python integers on inputs built to reach every carry and borrow path
(tests/fp_core_cases.py).  The host build the other CPU tests compile replaces these asm blocks with portable
fallbacks, so without this file the CPU suite runs none of the arithmetic the kernels are built on."""
from collections import defaultdict

import pytest

import fp_core_cases as fc
import ptx_model as pm
from ptx_model import M32

OPS = fc.OPS


@pytest.fixture(scope="module")
def cases():
    return fc.cases()


@pytest.mark.parametrize("op", OPS)
def test_model_matches_integers(op, cases):
    core = pm.FpCore()
    bad = []
    for args in cases[op]:
        err = fc.check(op, args, core.op(op, args))
        if err:
            bad.append((args, err))
    assert not bad, "%d of %d cases wrong, first: %s" % (len(bad), len(cases[op]), bad[:3])


def _census(paths):
    seen = defaultdict(int)
    for m, c, k, t in paths:
        seen[(m, c)] += 1
        if k == -1 and t & M32 == M32:
            seen["k=-1, t0 all ones"] += 1
        if k == 1 and t & M32 == 0:
            seen["k=+1, t0 zero"] += 1
    return seen


ALL_PATHS = [(0, 0), (0, 1), (1, 0), (1, 1), "k=-1, t0 all ones"]


@pytest.mark.parametrize("op,need", [
    ("reduce160", ALL_PATHS + ["k=+1, t0 zero"]),
    ("wide_reduce", ALL_PATHS + ["k=+1, t0 zero"]),
    ("mul_nc", ALL_PATHS + ["k=+1, t0 zero"]),
    ("sqr_nc", ALL_PATHS),
    ("reduce96_nc", [(0, 0), (0, 1), "k=+1, t0 zero"]),
    ("mul7_nc", [(0, 0), (0, 1)]),
])
def test_cases_reach_every_path(op, need, cases):
    """Each reduction's borrow m and fold carry c take every combination on the case set, and the corrections
    k = -1 and k = +1 meet the low words of t (all ones, zero) at which their own borrow chain changes."""
    if op == "reduce160":
        paths = [pm.reduce_path(*x) for x in cases[op]]
    elif op == "wide_reduce":
        paths = [pm.reduce_path(*pm.wide_words(w)) for (w,) in cases[op]]
    elif op == "mul_nc":
        paths = [pm.product_path(a, b) for a, b in cases[op]]
    elif op == "sqr_nc":
        paths = [pm.product_path(a, a) for (a,) in cases[op]]
    elif op == "reduce96_nc":
        paths = [pm.reduce_path(*x) for x in cases[op]]
    else:
        paths = [pm.reduce_path(*pm.product_words(a, 7)[:3]) for (a,) in cases[op]]
    seen = _census(paths)
    missing = [p for p in need if seen[p] == 0]
    assert not missing, "%s: no case reaches %s (reached: %s)" % (op, missing, dict(seen))


def test_model_covers_every_asm_block():
    """Every asm block of the device form of fp.cuh is modelled; a new block (or a new instruction in one) fails
    here until ptx_model.py is extended."""
    blocks = pm.asm_blocks()
    assert sorted(blocks) == sorted(pm.MODELLED)
    assert all(len(v) == 1 for v in blocks.values())
    assert pm.count_asm() == len(pm.MODELLED)


def test_model_rejects_what_it_does_not_know():
    with pytest.raises(pm.ModelError, match="not modelled"):
        pm.AsmBlock("f", "add.u64 %0, %1, %2;", [("=r", "d")], [("r", "a"), ("r", "b")])
    with pytest.raises(pm.ModelError, match="carry flag"):
        pm.AsmBlock("f", "addc.u32 %0, %1, 0;", [("=r", "d")], [("r", "a")]).run({"a": 1})
    with pytest.raises(pm.ModelError, match="read before"):
        pm.AsmBlock("f", "add.u32 %0, %0, %1;", [("=r", "d")], [("r", "a")]).run({"a": 1})
