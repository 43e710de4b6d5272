"""Inputs for the device field core (csrc/fp.cuh), built to reach every carry and borrow path of its reductions.

Random operands almost never reach the rare corrections: a reduction of (x1:x0) - (x4:x3) + x2 (2^32 - 1) borrows
without the fold carrying (k = -1) about once in 2^30 random inputs.  The cases here are solved for each path:
words chosen for a given borrow m and carry c, products a*b congruent to a small s mod 2^64 (their subtraction
borrows), exact multiples of 2^96, and accumulator states at the documented limits.  `cases()` returns
{op: [argument tuple]} in the argument form of ptx_model.FpCore.op, and `pack` lays one item out as the 16 input
words of schnorr_b200_debug_fp_core.  tests/test_fp_core_model.py checks that every path is still reached.
"""
import random

from ptx_model import M32, M64, P, hi, join, lo, reduce_path, wide_state, wide_value, wide_words

# the ops of schnorr_b200_debug_fp_core, in the order of its enum
OPS = ("sub", "add", "neg", "dbl", "reduce96_nc", "reduce96", "reduce160_nc", "reduce160", "canon_sel", "canon",
       "mul_nc", "sqr_nc", "mul", "sqr", "mul7_nc", "mul_small", "sqr_n", "inv",
       "wide_mac", "wide_mac_sqr", "wide_add64", "wide_double", "wide_reduce", "wide_mac_loop")

EDGE_WORDS = (0, 1, 2**31, 2**32 - 2, 2**32 - 1)
EDGE_X4 = (0, 1, 2**30, 2**31 - 1)
NONCANON = (P, P + 1, P + 2, 2**64 - 2, 2**64 - 1, 0xFFFFFFFF00000000 + 2**31, (P + 2**64) // 2)
EDGE64 = (0, 1, 2, 7, 2**32 - 1, 2**32, 2**32 + 1, 2**48, 2**63, 2**63 - 1, P - 1, P - 2, P - 2**32,
          0xFFFFFFFF00000000, 0xFFFFFFFEFFFFFFFF, 0x8000000080000000, 0x7FFFFFFF7FFFFFFF, 2**64 - 1, P, P + 1)
CANON_SEL = (P - 1, P, P + 1, 2**64 - 1, 0xFFFFFFFF00000000, 0xFFFFFFFEFFFFFFFF)

# products far above 2^30 terms overflow the accumulator; these are the documented limits
WIDE_MAX_PRODUCTS = 1 << 30


def solve_reduce160(rng, m, c, t=None, x2=None, x4_max=2**31 - 1, tries=4000):
    """Words x0..x4 (x4 <= x4_max) whose reduction takes borrow m and carry c and folds to t (random if None)."""
    for _ in range(tries):
        y2 = rng.getrandbits(32) if x2 is None else x2
        if rng.random() < 0.3:
            y2 = rng.getrandbits(rng.choice((1, 4, 16)))
        sub = (rng.randint(0, x4_max) << 32) | rng.getrandbits(32)
        tt = rng.getrandbits(64) if t is None else t
        low = tt + (c << 64) - y2 * M32 + sub - (m << 64)
        if 0 <= low <= M64:
            x = (lo(low), hi(low), y2, lo(sub), hi(sub))
            got = reduce_path(*x)
            if got[:2] == (m, c) and got[3] == tt:
                return x
    return None


def reduce160_cases(rng, n_random=400):
    out = [(a, b, c, d, e) for a in EDGE_WORDS for b in EDGE_WORDS for c in EDGE_WORDS for d in EDGE_WORDS
           for e in EDGE_X4]
    for m in (0, 1):
        for c in (0, 1):
            for _ in range(60):
                x = solve_reduce160(rng, m, c)
                if x:
                    out.append(x)
    for _ in range(60):
        # k = -1 with the low word of t all ones: the correction's low subtraction does not borrow
        x = solve_reduce160(rng, 1, 0, t=(rng.getrandbits(32) << 32) | M32)
        if x:
            out.append(x)
        # k = +1 with the low word of t zero: the correction's low subtraction borrows
        x = solve_reduce160(rng, 0, 1, t=rng.getrandbits(32) << 32)
        if x:
            out.append(x)
        # k = -1 / +1 near the ends of the range of t
        for m, c, t in ((1, 0, 2**64 - 2**31 - rng.getrandbits(20)), (0, 1, 2**64 - 2**33 - rng.getrandbits(8)),
                        (1, 0, 2**64 - (2**63 - 1) + rng.getrandbits(8))):
            x = solve_reduce160(rng, m, c, t=t)
            if x:
                out.append(x)
    # the extremes of t: k = +1 at t = 2^64 - 2^33 (x1:x0 all ones, x2 = 2^32 - 1) and k = -1 at t = 2^64 - (x4:x3)max
    out += [(M32, M32, M32, 0, 0), (0, 0, 0, M32, 2**31 - 1), (0, 0, 1, M32, 2**31 - 1), (M32 - 1, M32, M32, 0, 0)]
    for _ in range(n_random):
        out.append(tuple(rng.getrandbits(32) for _ in range(4)) + (rng.randint(0, 2**31 - 1),))
    return out


def reduce96_cases(rng, n_random=200):
    out = [(a, b, c) for a in EDGE_WORDS for b in EDGE_WORDS for c in EDGE_WORDS]
    for _ in range(n_random):
        x2 = rng.getrandbits(32)
        low = 2**64 - x2 * M32 + rng.randint(-2**20, 2**20)       # around the fold's carry
        out.append((lo(low), hi(low), x2) if 0 <= low <= M64 else (rng.getrandbits(32), rng.getrandbits(32), x2))
        low = 2**64 - x2 * M32 + (rng.getrandbits(32) << 32)      # carries onto a low word 0
        out.append((lo(low), hi(low), x2) if 0 <= low <= M64 else (0, M32, M32))
        out.append(tuple(rng.getrandbits(32) for _ in range(3)))
    return out


def _sqrt_mod_2_64(s):
    """A square root of s = 1 (mod 8) modulo 2^64 (Hensel lifting)."""
    x = 1
    for i in range(3, 64):
        if ((x * x - s) >> i) & 1:
            x += 1 << (i - 1)
    assert (x * x - s) % 2**64 == 0
    return x & M64


def mul_cases(rng, n_random=600):
    out = [(a, b) for a in EDGE64 for b in EDGE64]
    out += [(a, b) for a in NONCANON for b in EDGE64 + NONCANON]
    # a*b = s (mod 2^64) with a small s: (p1:p0) - p3 borrows
    for bits in (0, 1, 8, 20, 32, 40, 64):
        for _ in range(60):
            a = rng.getrandbits(64) | 1
            s = rng.getrandbits(bits) if bits else 0
            out.append((a, s * pow(a, -1, 2**64) % 2**64))
    # k = -1 needs p2 = p1 = 0 and p0 < p3: exact multiples u 2^96 (u = 1: the low word of t is all ones)
    for j in range(33, 64):
        out.append((1 << j, 1 << (96 - j)))
        u, v = rng.getrandbits(rng.randint(1, 64 - j)) | 1, rng.getrandbits(rng.randint(1, j - 32)) | 1
        out.append((u << j, v << (96 - j)))
    # k = +1 with the low word of t zero: a = 2^64 - 1, b = (b1:b0) with 2 b0 + b1 = 1 (mod 2^32), b0 > b1
    for _ in range(40):
        b0 = rng.randint(2**31 + 2**30, M32)
        out.append((M64, ((1 - 2 * b0) & M32) << 32 | b0))
    for _ in range(n_random):
        out.append((rng.getrandbits(64), rng.getrandbits(64)))
        out.append((rng.randrange(P), rng.randrange(P)))
    return out


def sqr_cases(rng, n_random=400):
    out = list(EDGE64) + list(NONCANON)
    for s in range(1, 2**12, 8):                 # a^2 = s (mod 2^64): borrows
        r = _sqrt_mod_2_64(s)
        out += [r, 2**64 - r, r ^ (1 << 63)]
    for _ in range(100):                         # a = 2^32 h + l with a small l
        out.append((rng.getrandbits(32) << 32) | rng.getrandbits(rng.choice((1, 4, 8))))
    out += [u << 48 for u in range(1, 2**16, 97)]  # a^2 = u^2 2^96: k = -1 (u = 1: the low word of t is all ones)
    out += [rng.getrandbits(64) for _ in range(n_random)] + [rng.randrange(P) for _ in range(n_random)]
    return out


def sub_cases(rng, n_random=300):
    minuends = list(EDGE64) + list(NONCANON) + [rng.getrandbits(64) for _ in range(20)]
    subtrahends = [0, 1, 2, 2**32 - 1, 2**32, P - 2, P - 1, P] + [rng.randrange(P + 1) for _ in range(10)]
    out = [(a, b) for a in minuends for b in subtrahends]
    out += [(rng.randrange(P), rng.randrange(P + 1)) for _ in range(n_random)]
    return out


def canonical(rng, n_random):
    return [x for x in EDGE64 if x < P] + [rng.randrange(P) for _ in range(n_random)]


# ---- accumulator states --------------------------------------------------------------------------------------------
def state_after(n, a=M64, b=M64):
    """The exact state after n products a*b from zero: E and O are plain sums."""
    a0, a1, b0, b1 = lo(a), hi(a), lo(b), hi(b)
    return wide_state(n * (a0 * b0 + (a1 * b1 << 64)), n * (a0 * b1 + a1 * b0))


def random_state(rng, e4_bits=29, o3_bits=30):
    return tuple(rng.getrandbits(32) for _ in range(4)) + (rng.getrandbits(e4_bits),) + \
        (rng.getrandbits(32), rng.getrandbits(32), rng.getrandbits(o3_bits))


def wide_states(rng, n_random=150):
    """States every accumulator op may start from: each still takes one more product without leaving its limits."""
    out = [(0,) * 8, state_after(1), state_after(WIDE_MAX_PRODUCTS // 2), state_after(WIDE_MAX_PRODUCTS - 1),
           state_after(WIDE_MAX_PRODUCTS - 1, P - 1, P - 1), state_after(12345, 2**64 - 1, 2**63)]
    # the reduce160 words as states (o = 0): wide_reduce sees exactly these x0..x4
    for x in reduce160_cases(rng, n_random=0)[::7]:
        if x[4] < 2**30:
            out.append(x + (0, 0, 0))
    # carries of E >> 32 + O across every word
    for e in ((M32, M32, M32), (M32, M32, 0), (0, M32, M32)):
        for o in ((1, 0, 0), (M32, M32, 2**30), (M32, 0, 0), (0, 0, 1)):
            out.append((M32,) + e + (2**29,) + o)
    out += [random_state(rng) for _ in range(n_random)]
    return out


def wide_limit_states():
    """States with e4 and o3 at their largest reachable values, for wide_double and wide_reduce."""
    top = [state_after(WIDE_MAX_PRODUCTS), state_after(WIDE_MAX_PRODUCTS, P - 1, P - 1),
           # x4 = e4 + the carry of E >> 32 + O reaches 2^31 - 1
           (M32, M32, M32, M32, 2**31 - 2, M32, M32, 2**31 - 1), (0, M32, M32, M32, 2**31 - 2, 1, 0, 0)]
    half = [state_after(WIDE_MAX_PRODUCTS // 2), state_after(WIDE_MAX_PRODUCTS // 2, P - 1, P - 1),
            (M32, M32, M32, M32, 2**30 - 2, M32, M32, 2**30 - 1)]   # doubled: x4 = 2^31 - 2
    return top, half


def cases(seed=20261022, n_random=1):
    """{op: [args]} for every op of schnorr_b200_debug_fp_core.  n_random scales the random cases."""
    rng = random.Random(seed)
    r = lambda k: int(k * n_random)
    red160 = reduce160_cases(rng, r(400))
    red96 = reduce96_cases(rng, r(200))
    mul = mul_cases(rng, r(600))
    sqr = sqr_cases(rng, r(400))
    canon_in = canonical(rng, r(200))
    states = wide_states(rng, r(150))
    top, half = wide_limit_states()
    ops64 = list(EDGE64) + list(NONCANON) + [rng.getrandbits(64) for _ in range(r(40))]
    c = {
        "sub": sub_cases(rng, r(300)),
        "add": [(a, b) for a, b in sub_cases(rng, r(300)) if b < P],
        "neg": [(a,) for a in canon_in],
        "dbl": [(a,) for a in canon_in],
        "reduce96_nc": red96, "reduce96": red96,
        "reduce160_nc": red160, "reduce160": red160,
        "canon_sel": [(a,) for a in list(CANON_SEL) + list(EDGE64) + list(NONCANON)] +
                     [(rng.getrandbits(64),) for _ in range(r(200))],
        "canon": [(a,) for a in list(CANON_SEL) + list(EDGE64) + list(NONCANON)],
        "mul_nc": mul, "mul": mul,
        "sqr_nc": [(a,) for a in sqr], "sqr": [(a,) for a in sqr],
        "mul7_nc": [(a,) for a in ops64] + [(2**64 - k,) for k in range(1, 40)] + [(-(-2**64 // 7) + k,) for k in range(-3, 4)],
        "mul_small": [(a, k) for a in ops64 for k in (0, 1, 7, 2**31, M32)] + [(rng.getrandbits(64), rng.getrandbits(32)) for _ in range(r(200))],
        "sqr_n": [(a, n) for a in list(EDGE64[:12]) + list(NONCANON[:3]) for n in (0, 1, 5, 64)],
        "inv": [(a,) for a in list(EDGE64) + list(NONCANON)] + [(rng.randrange(P),) for _ in range(r(20))],
        "wide_reduce": [(w,) for w in states + top + half],
        "wide_double": [(w,) for w in states + half],
    }
    pairs = [(a, b) for a, b in mul[::5]]
    c["wide_mac"] = [(w, a, b) for w, (a, b) in zip(states * 4, pairs)] + \
        [(w, M64, M64) for w in (state_after(WIDE_MAX_PRODUCTS - 1), state_after(WIDE_MAX_PRODUCTS - 1, P - 1, P - 1))]
    c["wide_mac_sqr"] = [(w, a) for w, a in zip(states * 4, sqr)] + [(state_after(WIDE_MAX_PRODUCTS - 1), M64)]
    c["wide_add64"] = [(w, v) for w in states for v in (0, 1, M64, P, rng.getrandbits(64))]
    # repeated products up to the 2^30-product limit, from the exact state 2^10 products before it
    c["wide_mac_loop"] = [(state_after(WIDE_MAX_PRODUCTS - 1024), M64, M64, 1024),
                          (state_after(WIDE_MAX_PRODUCTS - 1024, P - 1, P - 1), P - 1, P - 1, 1024),
                          (state_after(WIDE_MAX_PRODUCTS - 3, M64, 2**63), M64, 2**63, 3),
                          ((0,) * 8, M64, M64, 1000), ((0,) * 8, 0x1234567890ABCDEF, P - 5, 777)]
    return c


def pack(op, args):
    """The 16 input words of one item of schnorr_b200_debug_fp_core."""
    w = [0] * 16
    if op.startswith("wide_"):
        w[0:8] = args[0]
        if len(args) > 1:
            w[8], w[9] = lo(args[1]), hi(args[1])
        if len(args) > 2:
            w[10], w[11] = lo(args[2]), hi(args[2])
        if len(args) > 3:
            w[12] = args[3]
    elif op.startswith("reduce"):
        w[:len(args)] = args
    else:
        w[0], w[1] = lo(args[0]), hi(args[0])
        if len(args) > 1:
            b = args[1]
            w[2], w[3] = lo(b), hi(b)
    return w


# ---- what each op must return, from Python integers --------------------------------------------------------------
def wide_result(op, args):
    """The exact (E, O) after an accumulator op."""
    E, O = wide_value(args[0])
    if op in ("wide_mac", "wide_mac_sqr", "wide_mac_loop"):
        a = args[1]
        b = args[1] if op == "wide_mac_sqr" else args[2]
        n = args[3] if op == "wide_mac_loop" else 1
        E += n * (lo(a) * lo(b) + (hi(a) * hi(b) << 64))
        O += n * (lo(a) * hi(b) + hi(a) * lo(b))
    elif op == "wide_add64":
        E += args[1]
    elif op == "wide_double":
        E, O = 2 * E, 2 * O
    return E, O


def expected(op, args):
    """(residue mod p, canonical?) of an op's result.  canonical = the result must be < p; otherwise any 64-bit
    representative is allowed."""
    if op.startswith("wide_"):
        E, O = wide_result(op, args)
        return (E + (O << 32)) % P, None
    x = args
    v = {
        "sub": lambda: (x[0] - x[1]) % P, "add": lambda: (x[0] + x[1]) % P, "neg": lambda: -x[0] % P,
        "dbl": lambda: 2 * x[0] % P,
        "reduce96_nc": lambda: (x[0] | x[1] << 32 | x[2] << 64) % P,
        "reduce160_nc": lambda: sum(w << (32 * i) for i, w in enumerate(x)) % P,
        "canon_sel": lambda: x[0] % P, "canon": lambda: x[0] % P,
        "mul_nc": lambda: x[0] * x[1] % P, "sqr_nc": lambda: x[0] * x[0] % P, "mul7_nc": lambda: 7 * x[0] % P,
        "mul_small": lambda: x[0] * x[1] % P, "sqr_n": lambda: pow(x[0], 2**x[1], P),
        "inv": lambda: pow(x[0], P - 2, P),
    }
    v["reduce96"], v["reduce160"], v["mul"], v["sqr"] = v["reduce96_nc"], v["reduce160_nc"], v["mul_nc"], v["sqr_nc"]
    nc = op.endswith("_nc") or (op == "sub" and x[0] >= P) or (op == "add" and x[0] >= P)
    return v[op](), not nc


def sub_representative(a, b):
    """The exact 64-bit value fp_sub returns (its host form): a - b, plus p when it borrows."""
    d = (a - b) & M64
    return (d - 0xFFFFFFFF) & M64 if a < b else d


def check(op, args, out):
    """Checks the 16 output words of one item against Python integers; returns None or a description."""
    if op.startswith("wide_"):
        E, O = wide_result(op, args)
        assert E < 2**160 and O < 2**96, "case outside the accumulator's limits"
        assert wide_words(wide_state(E, O))[4] < 2**31, "case outside the reduction's limits"
        if tuple(out[0:8]) != wide_state(E, O):
            return "state %s != %s" % (out[0:8], wide_state(E, O))
        want = (E + (O << 32)) % P
        nc, cn = join(out[8], out[9]), join(out[10], out[11])
        if nc % P != want or cn != want:
            return "reductions %#x %#x != %#x" % (nc, cn, want)
        return None
    if any(out[2:]):
        return "unused words written"
    r = join(out[0], out[1])
    want, canonical = expected(op, args)
    if r % P != want:
        return "%#x = %#x mod p, want %#x" % (r, r % P, want)
    if canonical and r >= P:
        return "%#x is not canonical" % r
    if op == "sub" and r != sub_representative(*args):
        return "representative %#x, want %#x" % (r, sub_representative(*args))
    if op == "add" and r != sub_representative(args[0], (P - args[1]) % 2**64):
        return "representative %#x" % r
    return None
