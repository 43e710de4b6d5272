"""CPU checks of verify_exceptional_model.py: the model agrees with the oracle, every case makes the event it is named
after happen, the host build of verify_core_fast returns exactly the model's result, and a census of the events the
cases reach (test_gpu_verify_exceptional.py runs the same cases on the device)."""
import ctypes as C

import numpy as np
import pytest

import cref
import verify_exceptional_model as M


def _r_model(base, r):
    pt, inf = base.point(r)
    return None if inf else bytes(pt)


def _r_oracle(c):
    pt, inf = M.oracle_r(c.base, c.a, c.h, c.e)
    return None if inf else bytes(pt)


@pytest.mark.parametrize("c", M.hook_cases(), ids=lambda c: c.name)
def test_hook_case_model_is_the_oracle_and_the_host_build(hostsim, c):
    res, r, tr = M.fast_core(c.a, c.h, c.e, c.base)
    assert _r_model(c.base, r) == _r_oracle(c), "the model's R times B is h*P + e*G"
    out = np.zeros(96, dtype=np.uint8)
    H, E, P = M._le32(c.h), M._le32(c.e), c.pk96().copy()
    got = hostsim.hs_verify_core_fast(P.ctypes.data_as(C.c_void_p), H.ctypes.data_as(C.c_void_p),
                                      E.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    assert got == res, (got, res, tr.events[:4])
    if res != M.EXC:
        assert bytes(out) == _r_oracle(c)
    if c.name == "G_same_h_low":
        assert tr.events == [("h_sum", 1, "same_h")] and res == M.TF
    kind = c.name.rsplit("_", 1)[-1]
    if c.name.startswith("e") and kind in ("double", "cancel"):
        assert tr.events[0] == ("e", int(c.name[1:].split("_")[0]), kind)


@pytest.mark.parametrize("c", M.sig_cases(), ids=lambda c: c.name)
def test_signature_case_events_and_verdict(c):
    sigs, pk, inf, blob, off = M.case_arrays([c])
    assert cref.verify_many(sigs, pk, inf, blob, off)[0] == c.verdict
    digest = cref.hash_messages(sigs[:, :48], pk, blob, off)[0]
    assert M.o.scalar_from_digest(bytes(digest)) == c.h, "the case's challenge is the oracle's hash"
    res, r, tr = M.fast_core(c.a, c.h, c.e, c.base)
    assert _r_model(c.base, r) == _r_oracle(c)
    kinds = tr.kinds()
    if c.name.startswith("V1_R_identity") and c.name != "V1_R_identity_x_nonzero":
        assert r == 0 and ("e", "cancel") in kinds and res == M.EXC
        assert ("final", "cancel") in M.one_core(c.a, c.h, c.e, c.base)[3].kinds()
    elif c.name.startswith("V2"):
        d = int(c.name.split("_d")[1])
        assert M.top_digit(c.e) == d and ("e", "cancel") in kinds and res == M.EXC
        assert [ev for ev in tr.events if ev[2] == "cancel"][0][1] < 19
    elif c.name.startswith("V3"):
        assert tr.events[-1] == ("e", 19, "double") and res == M.EXC
    elif c.name.startswith("V4"):
        assert ("h_sum", "same_h") in kinds and res == M.TF
        if c.name == "V4_same_h_low":
            assert [b for s, b, k in tr.events if k == "same_h"][0] < 6
    elif c.name.startswith("key_"):
        assert res in (M.NTF, M.EXC)
        if c.name == "key_T181_h_event":
            assert res == M.EXC and any(s.startswith("h_") for s, _, _ in tr.events)
    for core in ("reg", "one"):
        if core == "reg" and c.m > 1:
            continue
        fn = M.reg_core if core == "reg" else M.one_core
        assert fn(c.a, c.h, c.e, c.base)[1] == r


def test_q_side_events_per_order():
    """The q-side stages use the constant digits of q: their events depend on the key's order only.  Prime-order and
    mixed keys G + T_m have none; T_2 fails at the first doubling; T_29 and T_58 collide inside the chain buckets;
    T_181 and T_155833 have none, so their h-side events decide."""
    want = {2: {("chain", "dbl2")}, 29: {("q_chain", "double"), ("q_chain", "cancel")}, 58: {("q_chain", "cancel")},
            181: set(), 155833: set()}
    for m, ev in want.items():
        b = M.base_of(m)
        tm = M.Q * pow(M.Q, -1, m) % b.N
        q_side = {(s, k) for s, _, k in M.fast_core(tm, 0, 1, b)[2].events if s in ("chain", "q_chain", "q_running",
                                                                                      "q_sum", "q_check")}
        assert ev <= q_side and (ev or not q_side), (m, q_side)
        assert not M.fast_core(1, 0, 1, b)[2].events
    assert not M.fast_core(12345, 0, 1, M.base_of(1))[2].events


def test_prime_order_h_side_collisions_are_unreachable():
    """For a key k G of prime order every challenge-side value is k z, z an integer built from the signed digits of h:
    bucket and running sums are sums of +-16^j over distinct j (below q / 2, and zero or equal to another such sum only
    as the same digits), and O - R, O + R have digits of magnitude at most 9 < 16, which cannot sum to zero.  So no chain,
    running or sum addition of the challenge side collides, and the only O == R case is the structural same_h one,
    which the fast path doubles.  Likewise the registered h windows: a partial sum stays below half of the next table
    entry.  Checked here on random and edge challenges, in all three cores."""
    assert sum(16 ** j for j in range(64)) < M.Q // 2
    rng = np.random.default_rng(5)
    b = M.base_of(1)
    hs = [int.from_bytes(rng.bytes(32), "little") % M.Q for _ in range(200)] + [0, 1, M.Q - 1, 0x8888888888888888]
    for h in hs:
        _, _, tr = M.fast_core(7777777, h, 0, b)
        assert {k for _, _, k in tr.events} <= {"same_h", "identity"}
        assert not M.reg_core(7777777, h, 3, b)[2].events
        # k_verify_one tests [q]P == O as 2 O_1 + R_0 with an exact addition (a cancel for every key of prime order),
        # and its O == R aggregation step is the same_h case, resolved by the exact fall-back
        assert M.one_core(7777777, h, 3, b)[3].kinds() <= {("q_final", "cancel"), ("h_sum", "double")}


CENSUS = {
    # (core, stage, kind) the cases must keep reaching
    ("fast", "e", "double"), ("fast", "e", "cancel"), ("fast", "e", "identity"), ("fast", "h_sum", "same_h"),
    ("fast", "chain", "dbl2"), ("fast", "q_chain", "double"), ("fast", "q_chain", "cancel"),
    ("fast", "h_chain", "double"), ("fast", "h_chain", "cancel"), ("fast", "h_running", "double"),
    ("fast", "h_running", "cancel"), ("fast", "h_sum", "double"), ("fast", "h_sum", "cancel"),
    ("reg", "e", "double"), ("reg", "e", "cancel"),
    ("one", "final", "cancel"), ("one", "h_sum", "double"),
}
# reachable only with keys of small order, which the registered core never runs (status KEY_NOT_TORSION_FREE), or never
UNREACHABLE = {("reg", "h_table", "double"), ("reg", "h_table", "cancel"), ("one", "e_stage", "double"),
               ("one", "e_stage", "cancel")}


def census():
    seen = set()
    for c in list(M.hook_cases()) + list(M.sig_cases()):
        seen |= {("fast", s, k) for s, k in M.fast_core(c.a, c.h, c.e, c.base)[2].kinds()}
        seen |= {("one", s, k) for s, k in M.one_core(c.a, c.h, c.e, c.base)[3].kinds()}
        if (M.Q * c.a) % c.base.N == 0:
            seen |= {("reg", s, k) for s, k in M.reg_core(c.a, c.h, c.e, c.base)[2].kinds()}
    return seen


def test_census_of_events():
    seen = census()
    print(sorted(seen))
    assert CENSUS <= seen, CENSUS - seen
    assert not UNREACHABLE & seen
