"""The h*P stage of k_verify_reg_one (one_reg.cuh) as integers: the signed 8-bit recoding of a challenge, the tree over
its 32 window terms, and the planner of a challenge whose two halves (windows 0-15 and 16-31) are the same multiple of
the key, which makes the last addition of the tree a doubling.
"""
from fractions import Fraction

import pyref as o

Q = o.Q
KT_W, KT_WINDOWS = 8, 32
WARP_WINDOWS = 8


def recode(h):
    """jf_table_accumulate's recoding: 32 signed digits, -128 < d <= 128, carry into the next window."""
    out, carry = [], 0
    for i in range(KT_WINDOWS):
        raw = ((h >> (KT_W * i)) & 0xFF) + carry
        neg = raw > 128
        carry = 1 if neg else 0
        out.append(raw - 256 if neg else raw)
    assert carry == 0
    return out


def from_digits(d):
    return sum(x << (KT_W * i) for i, x in enumerate(d))


def tree(terms):
    """The pairing of the device tree: stride 1, 2, 4 inside each warp's eight windows, then (0..7 + 8..15) and
    (16..23 + 24..31), then their sum -> (total, [(stride, j, left, right)] of every addition, in order)."""
    v = list(terms)
    adds = []
    s = 1
    while s < KT_WINDOWS:
        for j in range(0, KT_WINDOWS, 2 * s):
            adds.append((s, j, v[j], v[j + s]))
            v[j] = v[j] + v[j + s]
        s <<= 1
    return v[0], adds


def window_terms(h):
    """The integer multiple of the key that window i contributes: d_i 2^(8 i)."""
    return [d << (KT_W * i) for i, d in enumerate(recode(h))]


def halves(h):
    """(windows 0-15, windows 16-31) of h's recoding as integers."""
    t = window_terms(h)
    return sum(t[:16]), sum(t[16:])


def convergents(x):
    """Continued-fraction convergents p / r of a Fraction x."""
    p0, p1, r0, r1 = 0, 1, 1, 0
    while True:
        a = x.numerator // x.denominator
        p0, p1 = p1, a * p1 + p0
        r0, r1 = r1, a * r1 + r0
        yield p1, r1
        frac = x - a
        if frac == 0:
            return
        x = 1 / frac


def plan_same_halves():
    """A challenge h < q whose windows 0-15 sum to L and windows 16-31 to H 2^128 with H 2^128 = L (mod q): small H, L
    from a convergent p / r of 2^128 / q (r 2^128 - p q is small), so both halves are L * P.  -> (h, H, L)."""
    best = None
    for p, r in convergents(Fraction(1 << 128, Q)):
        L = r * (1 << 128) - p * Q
        for H, L_ in ((r, L), (-r, -L)):
            h = H * (1 << 128) + L_
            if 0 < h < Q and halves(h) == (L_, H << 128):
                best = (h, H, L_)
        if r > 1 << 127:
            break
    assert best is not None
    return best
