"""A catalogue of adversarial wire encodings, built from seeds with the big-integer oracle (oracle/pyref.py).

Every byte of a compressed point (49 B: x limbs || flag byte), a signature record (81 B: x || flag || e) and a key
record (96 B: x || y) comes from the caller, and the decoding rules of pyref.decompress / pyref.f6_from_bytes decide
the verdict before any group arithmetic runs.  The rows below sit on each edge of those rules:

  honest     subgroup points with their flag, and with the sign bit flipped (decodes to -P)
  identity   0x80 with x = 0 (decodes); 0xC0, 0x80 with a non-zero or non-canonical limb (do not)
  reserved   each of the bits 0x01 .. 0x20 on an honest x, alone and with 0x40 / 0x80
  limbs      an honest x with limb k at p - 1, p, p + 1, 2^63, 2^64 - 1 under 0x00 and 0x80, and a decodable x with a
             small limb k written as limb + p (a non-canonical alias of a point on the curve)
  offcurve   canonical x with x^3 + x + B a non-square, and x = 0 without the identity flag (B is a non-square)
  torsion2   T2 = KAT * (n / 2), y = 0, under 0x00 and 0x40 (both decode to T2)
  subfield   x = x0 + x1 u with x^3 + x + B in Fp3: the root y in Fp3 (c5 = 0, the only points whose sign is decided
             at c4 or lower) or in u Fp3, the two sub-branches of the Fp3 case of the square root

Fp6 = Fp3[u] / (u^2 - v), v^3 = 7: coefficient 2i is the i-th coefficient of the Fp3 part, 2i + 1 that of the u part.
"""
import functools

import numpy as np

import pyref as o

P, Q = o.P, o.Q
SEED = 0x31BE
CATEGORIES = ("honest", "identity", "reserved", "limbs", "offcurve", "torsion2", "subfield")
LIMB_VALUES = (("p-1", P - 1), ("p", P), ("p+1", P + 1), ("2^63", 2**63), ("2^64-1", 2**64 - 1))


def enc(x, flag):
    """49-byte compressed encoding of six 64-bit limbs (any values) and a flag byte"""
    return b"".join(int(c).to_bytes(8, "little") for c in x) + bytes([flag])


def rhs(x):
    return o.f6_add(o.f6_add(o.f6_mul(o.f6_sqr(x), x), x), o.CURVE_B)


def in_fp3(a):
    return a[1] == a[3] == a[5] == 0


def in_u_fp3(a):
    return a[0] == a[2] == a[4] == 0


def _fp(seed, domain, i):
    return int.from_bytes(o.prf(seed, domain, i, 8), "little") % P


def _fp6(seed, domain, i):
    return tuple(_fp(seed, domain, 6 * i + k) for k in range(6))


@functools.lru_cache(maxsize=None)
def honest_keys():
    """three subgroup points and their secret keys"""
    sks = [o.synth_scalar(SEED, "wire-honest", i) for i in range(3)]
    return [(sk, o.pt_mul(o.generator(), sk)) for sk in sks]


@functools.lru_cache(maxsize=None)
def t2():
    return o.pt_mul((o.KAT_X, o.KAT_Y), o.COFACTOR * Q // 2)


@functools.lru_cache(maxsize=None)
def subfield_points():
    """[(kind, (x, y))]: at least two points with y in Fp3 ("fp3") and two with y in u Fp3 ("ufp3").
    x1 (x1 u, the u part of x) is drawn; the u part of x^3 + x + B, x1 (3 x0^2 + v x1^2 + 1) + 1, vanishes for
    x0^2 = (-1/x1 - v x1^2 - 1) / 3, which has a root in Fp3 for about half of the draws."""
    inv3 = pow(3, P - 2, P)
    got = {"fp3": [], "ufp3": []}
    i = 0
    while len(got["fp3"]) < 2 or len(got["ufp3"]) < 2:
        x1 = tuple(_fp(SEED, "wire-subfield", 3 * i + k) for k in range(3))
        i += 1
        if x1 == (0, 0, 0):
            continue
        vx1 = o._f3_mulv(o._f3_sqr(x1))
        t = tuple((-a - b - c) * inv3 % P for a, b, c in zip(o._f3_inv(x1), vx1, (1, 0, 0)))
        r = o.f6_sqrt((t[0], 0, t[1], 0, t[2], 0))
        if r is None or not in_fp3(r):
            continue                                   # x0^2 = t has no root in Fp3
        x0 = (r[0], r[2], r[4])
        x = (x0[0], x1[0], x0[1], x1[1], x0[2], x1[2])
        a = rhs(x)
        assert in_fp3(a)
        y = o.f6_sqrt(a)
        assert y is not None                           # every element of Fp3 is a square in Fp6
        kind = "fp3" if in_fp3(y) else "ufp3"
        assert kind == "fp3" or in_u_fp3(y)
        if len(got[kind]) < 2:
            got[kind].append((x, y))
    return [(k, pt) for k in ("fp3", "ufp3") for pt in got[k]]


@functools.lru_cache(maxsize=None)
def nonsquare_xs():
    """two canonical x whose x^3 + x + B is a non-square"""
    out, i = [], 0
    while len(out) < 2:
        x = _fp6(SEED, "wire-offcurve", i)
        i += 1
        if not o.f6_is_square(rhs(x)):
            out.append(x)
    return out


@functools.lru_cache(maxsize=None)
def alias_points():
    """for k = 0..5: an x on the curve whose limb k is below 2^32 - 1, so that limb k + p still fits in 64 bits"""
    out, i = [], 0
    for k in range(6):
        while True:
            x = list(_fp6(SEED, "wire-alias", i))
            i += 1
            x[k] %= 2**32 - 1
            x = tuple(x)
            if o.f6_is_square(rhs(x)):
                out.append(x)
                break
    return out


@functools.lru_cache(maxsize=None)
def points():
    """[(name, 49 bytes, category)]"""
    rows = []
    add = lambda name, b, cat: rows.append((name, bytes(b), cat))     # noqa: E731
    hon = honest_keys()
    for j, (_, pt) in enumerate(hon):
        b = o.compress(pt)
        add("honest%d" % j, b, "honest")
        add("honest%d_flipped" % j, b[:48] + bytes([b[48] ^ 0x40]), "honest")
    hx = hon[0][1][0]
    zero = (0,) * 6
    add("identity", enc(zero, 0x80), "identity")
    add("identity_C0", enc(zero, 0xC0), "identity")
    for k in range(6):
        add("identity_limb%d" % k, enc(tuple(1 if i == k else 0 for i in range(6)), 0x80), "identity")
    add("identity_noncanonical", enc((P, 0, 0, 0, 0, 0), 0x80), "identity")
    for bit in range(6):
        for extra in (0, 0x40, 0x80):
            add("reserved_%02x_%02x" % (1 << bit, extra), enc(hx, (1 << bit) | extra), "reserved")
    for k in range(6):
        for vname, v in LIMB_VALUES:
            x = list(hx)
            x[k] = v
            for flag in (0x00, 0x80):
                add("limb%d_%s_%02x" % (k, vname, flag), enc(x, flag), "limbs")
    for k, x in enumerate(alias_points()):
        a = list(x)
        a[k] += P
        add("alias_limb%d" % k, enc(a, 0x00), "limbs")
    for j, x in enumerate(nonsquare_xs()):
        for flag in (0x00, 0x40):
            add("nonsquare%d_%02x" % (j, flag), enc(x, flag), "offcurve")
    for flag in (0x00, 0x40):
        add("x0_%02x" % flag, enc(zero, flag), "offcurve")
    for flag in (0x00, 0x40):
        add("t2_%02x" % flag, enc(t2()[0], flag), "torsion2")
    for j, (kind, (x, _)) in enumerate(subfield_points()):
        for flag in (0x00, 0x40):
            add("subfield_%s%d_%02x" % (kind, j % 2, flag), enc(x, flag), "subfield")
    return rows


# ---- 81-byte signature and 96-byte key records ---------------------------------------------------------------------
MESSAGE = b"wire cases"


@functools.lru_cache(maxsize=None)
def honest_record():
    """(sk, pk point, 81-byte signature over MESSAGE) for honest key 0"""
    sk, pk = honest_keys()[0]
    r49, e = o.sign(sk, pk, MESSAGE, o.synth_scalar(SEED, "wire-nonce", 0))
    return sk, pk, r49 + e.to_bytes(32, "little")


def _e_values():
    qtop = Q >> 192
    return (("e_q-1", Q - 1), ("e_q", Q), ("e_q+1", Q + 1), ("e_2^256-1", 2**256 - 1),
            ("e_top_gt_q", (qtop + 1) << 192), ("e_top_eq_q_low0", qtop << 192))


@functools.lru_cache(maxsize=None)
def records():
    """[(name, 81-byte signature, 96-byte key, pk_inf, category)], category "key", "sig" or "e"; the first row is the
    honest record"""
    _, pk, sig = honest_record()
    pk96 = o.f6_to_bytes(pk[0]) + o.f6_to_bytes(pk[1])
    rows = [("honest", sig, pk96, 0, "honest")]
    three = [v for v in LIMB_VALUES if v[0] in ("p-1", "p", "2^64-1")]
    for k in range(12):
        for vname, v in three:
            key = pk96[:8 * k] + v.to_bytes(8, "little") + pk96[8 * k + 8:]
            for inf in (0, 1):
                rows.append(("key_limb%d_%s_inf%d" % (k, vname, inf), sig, key, inf, "key"))
    for k in range(6):
        for vname, v in three:
            rows.append(("sig_limb%d_%s" % (k, vname), sig[:8 * k] + v.to_bytes(8, "little") + sig[8 * k + 8:], pk96, 0,
                         "sig"))
    for name, e in _e_values():
        rows.append((name, sig[:49] + e.to_bytes(32, "little"), pk96, 0, "e"))
    return rows


def as_arrays(rows):
    """records() rows -> (sigs [n, 81], pks [n, 96], inf [n]) uint8 arrays"""
    sigs = np.stack([np.frombuffer(r[1], np.uint8) for r in rows])
    pks = np.stack([np.frombuffer(r[2], np.uint8) for r in rows])
    return sigs, pks, np.array([r[3] for r in rows], np.uint8)
