"""The integer model of k_verify_reg_one's h*P stage (registered_one_model.py), without a GPU: the planned challenge
whose two halves are the same multiple of the key, the signed 8-bit recoding and the tree pairing."""
import numpy as np

import registered_one_model as R

Q = R.Q


def edge_challenges():
    out = [0, 1, 128, 129, 255, 256, Q - 1, (Q - 1) // 2, (1 << 254) - 1]
    out.append(R.from_digits([128] * 31 + [0]))                    # every digit +128
    out.append(R.from_digits([-127] * 31 + [1]))                   # every digit -127, the carry into the top window
    out.append(R.from_digits([0] * 8 + [5] + [0] * 15 + [-3] + [0] * 6 + [1]))   # zero windows
    return [h for h in out if 0 <= h < Q]


def test_planner_halves_agree_mod_q():
    h, H, L = R.plan_same_halves()
    assert 0 < h < Q
    assert (H * (1 << 128) - L) % Q == 0
    assert abs(H) < 1 << 128 and abs(L) < 1 << 128
    lo, hi = R.halves(h)
    assert lo == L and hi == H << 128
    assert R.from_digits(R.recode(h)) == h
    # the last tree addition adds two equal multiples of the key: a doubling
    total, adds = R.tree(R.window_terms(h))
    s, j, left, right = adds[-1]
    assert (s, j) == (16, 0) and (left - right) % Q == 0 and total == h


def test_recoding_and_tree_reproduce_the_challenge():
    rng = np.random.default_rng(5)
    cases = edge_challenges() + [int.from_bytes(rng.bytes(32), "little") % Q for _ in range(500)]
    for h in cases:
        d = R.recode(h)
        assert len(d) == 32 and all(-128 < x <= 128 for x in d)
        assert R.from_digits(d) == h
        total, adds = R.tree(R.window_terms(h))
        assert total == h
        assert len(adds) == 31
        assert [s for s, _, _, _ in adds].count(1) == 16 and adds[-1][:2] == (16, 0)


def test_recoding_edges():
    assert R.recode(128)[:2] == [128, 0]
    assert R.recode(129)[:2] == [-127, 1]
    d = R.recode(R.from_digits([-127] * 31 + [1]))
    assert d[31] == 1 and d[30] == -127


def test_tree_rounds():
    """31 additions; per warp 7 sequential ones, then one round on two warps and the last on one: 9 rounds, and
    windows 0-15 meet windows 16-31 only in the last addition."""
    _, adds = R.tree(list(range(32)))
    per_warp = [[a for a in adds if a[0] < 8 and a[1] // 8 == w] for w in range(4)]
    assert all(len(p) == 7 for p in per_warp)
    cross = [a for a in adds if a[0] >= 8]
    assert [(s, j) for s, j, _, _ in cross] == [(8, 0), (8, 16), (16, 0)]
    assert all((j < 16) == (j + s < 16) for s, j, _, _ in adds[:-1])
