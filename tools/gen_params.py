#!/usr/bin/env python3
"""Generate params/params.json and include/cheetah_params.h from the big-int oracle.

Every constant carries a provenance tag (SURVEY.md Appendix A):
  REF          read from the reference repo
  VERIFIED     derived/checked by computation from REF data
  SPEC-DERIVED produced by a published algorithm (Rescue-Prime ePrint 2020/1143)
  RECALLED     memory of the un-vendored upstream crates, NOT checkable here
  PLACEHOLDER  stand-in reproducible from REF data (the true upstream value is unknown)
  DERIVED      pure function of the other constants (helper tables for the kernels)
This file is the single place to swap in true upstream values (cheetah / hash crates).
Run:  python tools/gen_params.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyref as o  # noqa: E402

P, Q = o.P, o.Q


def limbs64(x, n):
    return [(x >> (64 * i)) & (2**64 - 1) for i in range(n)]


def limbs32(x, n):
    return [(x >> (32 * i)) & (2**32 - 1) for i in range(n)]


def wnaf(k, w):
    """width-w NAF, least-significant digit first."""
    out = []
    while k:
        if k & 1:
            d = k % (1 << w)
            if d >= (1 << (w - 1)):
                d -= 1 << w
            k -= d
        else:
            d = 0
        out.append(d)
        k >>= 1
    return out


def fold_top(digits, w, top):
    """Rewrite the two most significant digits of a width-w NAF so that no digit sits above bit `top`: the verification
    kernels walk ONE doubling chain for the subgroup check and for the challenge product, whose last 4-bit window starts
    at bit 252 -- a digit of q at bit 255 would cost three doublings nobody else needs.  The digit set (odd, |d| < 2^(w-1))
    and the number of non-zero digits are unchanged; only the non-adjacency of the top pair is given up, which the bucket
    method does not rely on."""
    d = list(digits)
    while len(d) - 1 > top:
        nz = [i for i, x in enumerate(d) if x]
        i1, i2 = nz[-2], nz[-1]
        m = d[i1] + (d[i2] << (i2 - i1))
        lim = 1 << (w - 1)
        for s in range(1, top - i1 + 1):
            cands = [(a, b) for b in range(-lim + 1, lim, 2) for a in [m - (b << s)] if a & 1 and abs(a) < lim]
            if cands and not any(d[i1 + 1:i1 + s + 1]):
                a, b = cands[0]
                d[i1], d[i2] = a, 0
                d[i1 + s] = b
                break
        else:
            raise ValueError("cannot fold the top digits below bit %d" % top)
        while d and d[-1] == 0:
            d.pop()
    return d


def main():
    G = o.generator()
    ark = o.rescue_round_constants()
    mds = o.rescue_mds()

    # Fp helpers: 2^32-th root of unity for Tonelli-Shanks in Fp, cube root of unity for the
    # Fp3 Frobenius.  7 is a generator of Fp^* for Goldilocks [VERIFIED below].
    for f in (2, 3, 5, 17, 257, 65537):
        assert pow(7, (P - 1) // f, P) != 1
    root32 = pow(7, (P - 1) >> 32, P)            # order 2^32
    assert pow(root32, 1 << 31, P) == P - 1
    omega3 = pow(7, (P - 1) // 3, P)             # v^p = omega3 * v in Fp3 = Fp[v]/(v^3-7)
    assert omega3 != 1 and pow(omega3, 3, P) == 1
    # u^p = 7^((p-1)/6) * u  (Frobenius on Fp6 = Fp[u]/(u^6-7))
    frob6 = [pow(7, ((P - 1) // 6) * i, P) for i in range(6)]

    # quadratic non-residue of Fp3 used by the Fp3 Tonelli-Shanks: any Fp non-square that stays
    # a non-square in Fp3 (odd-degree extension keeps quadratic character) -> 7.
    assert pow(7, (P - 1) // 2, P) == P - 1

    # scalar field Montgomery constants, R = 2^256
    R = 1 << 256
    q_inv32 = (-pow(Q, -1, 1 << 32)) % (1 << 32)
    r2 = (R * R) % Q

    q_wnaf5 = fold_top(wnaf(Q, 5), 5, 251)
    assert sum(d << i for i, d in enumerate(q_wnaf5)) == Q and len(q_wnaf5) == 252
    assert all(d == 0 or (d & 1 and abs(d) < 16) for d in q_wnaf5) and sum(1 for d in q_wnaf5 if d) == 44

    params = {
        "_about": "constants of the Cheetah/Rescue Schnorr path with provenance tags; see tools/gen_params.py",
        "p": {"value": hex(P), "tag": "REF README.md:4"},
        "fp6_nonresidue": {"value": 7, "tag": "REF README.md:8 (u^6 = 7)"},
        "curve_a": {"value": 1, "tag": "REF README.md:4-5"},
        "curve_b": {"value": [395, 1, 0, 0, 0, 0], "tag": "REF README.md:4-5 (u + 395)"},
        "q": {"value": hex(Q), "tag": "VERIFIED (SURVEY App. A)"},
        "cofactor": {"value": str(o.COFACTOR), "tag": "VERIFIED (SURVEY App. A)"},
        "kat_point": {"x": [hex(c) for c in o.KAT_X], "y": [hex(c) for c in o.KAT_Y],
                      "tag": "REF src/signature.rs:387-404"},
        "generator": {"x": [hex(c) for c in G[0]], "y": [hex(c) for c in G[1]],
                      "tag": ("REF (dumped from the cheetah crate: params/upstream_dump.json)" if o.upstream_dump() is not None
                              else "PLACEHOLDER = [cofactor]*kat_point; true cheetah generator unknown")},
        "compressed_flags": {"infinity_bit": 7, "sign_bit": 6,
                             "tag": "bit 7 REF src/public.rs:95-101; bit 6 + lexicographic rule RECALLED"},
        "rescue": {
            "width": 12, "rate": 8, "digest": 4, "alpha": 7, "inv_alpha": hex(o.INV_ALPHA),
            "rounds": o.RESCUE_ROUNDS,
            "mds_first_row": list(o.MDS_FIRST_ROW),
            "ark": [[hex(c) for c in row] for row in ark],
            "tag": "shape INFERRED from `rescue_64_12_8` (src/signature.rs:22); rounds + circulant MDS "
                   "RECALLED; round constants SPEC-DERIVED (SHAKE256, ePrint 2020/1143); "
                   "absorb/padding rule RECALLED (oracle/pyref.py rescue_hash_field)",
        },
    }
    os.makedirs(os.path.join(ROOT, "params"), exist_ok=True)
    with open(os.path.join(ROOT, "params", "params.json"), "w") as f:
        json.dump(params, f, indent=1)
        f.write("\n")

    def arr64(name, vals, per=3):
        s = "static const uint64_t %s[%d] = {\n" % (name, len(vals))
        for i in range(0, len(vals), per):
            s += "    " + ", ".join("0x%016xULL" % v for v in vals[i:i + per]) + ",\n"
        return s + "};\n"

    def arr32(name, vals, per=8):
        s = "static const uint32_t %s[%d] = {\n" % (name, len(vals))
        for i in range(0, len(vals), per):
            s += "    " + ", ".join("0x%08xu" % v for v in vals[i:i + per]) + ",\n"
        return s + "};\n"

    def arr8(name, vals, per=32, ty="int8_t"):
        s = "static const %s %s[%d] = {\n" % (ty, name, len(vals))
        for i in range(0, len(vals), per):
            s += "    " + ", ".join("%d" % v for v in vals[i:i + per]) + ",\n"
        return s + "};\n"

    h = []
    h.append("/* GENERATED by tools/gen_params.py -- do not edit.  Provenance tags: params/params.json.\n"
             " * Constants of the Cheetah curve / Rescue hash shared by the CPU oracle (oracle/cref.c)\n"
             " * and the CUDA engine (schnorr-sig_b200/csrc).  Plain C, usable from C, C++ and CUDA. */\n"
             "#ifndef CHEETAH_PARAMS_H\n#define CHEETAH_PARAMS_H\n#include <stdint.h>\n\n")
    # value-level provenance: 1 only once EVERY constant below carries a REF / VERIFIED tag (i.e. was dumped from the
    # real cheetah / hash crates, rust/dump_params); the library reports it (schnorr_b200_params_pinned)
    h.append("#define CHEETAH_PARAMS_PINNED 0\n")
    h.append("#define CHEETAH_PARAMS_PROVENANCE \"generator: PLACEHOLDER ([cofactor] * KAT point of src/signature.rs:387-404); "
             "Rescue rounds / MDS / padding: RECALLED; round constants: SPEC-DERIVED (ePrint 2020/1143); y-sign flag bit: "
             "RECALLED; p, Fp6, curve, q, KAT point, encodings: REF / VERIFIED\"\n")
    h.append("#define CHEETAH_P 0xffffffff00000001ULL            /* REF README.md:4 */\n")
    h.append("#define CHEETAH_CURVE_B0 395ULL                    /* B = u + 395, REF README.md:4-5 */\n")
    h.append("#define CHEETAH_CURVE_B1 1ULL\n")
    h.append("#define RESCUE_ROUNDS %d\n" % o.RESCUE_ROUNDS)
    h.append("#define RESCUE_INV_ALPHA 0x%016xULL\n" % o.INV_ALPHA)
    h.append("#define FP_ROOT_OF_UNITY_2_32 0x%016xULL   /* 7^((p-1)/2^32) */\n" % root32)
    h.append("#define FP_OMEGA3 0x%016xULL               /* 7^((p-1)/3): v^p = OMEGA3*v */\n" % omega3)
    h.append("#define SCALAR_QINV32 0x%08xu                     /* -q^-1 mod 2^32 */\n\n" % q_inv32)
    h.append("/* subgroup order q, little-endian limbs [VERIFIED] */\n")
    h.append(arr64("CHEETAH_Q64", limbs64(Q, 4), 4))
    h.append(arr32("CHEETAH_Q32", limbs32(Q, 8)))
    h.append("/* 2^512 mod q (Montgomery R^2, R = 2^256) */\n")
    h.append(arr32("SCALAR_R2_32", limbs32(r2, 8)))
    h.append("/* generator [%s] */\n" % ("REF: params/upstream_dump.json" if o.upstream_dump() is not None
                                          else "PLACEHOLDER = cofactor * KAT point"))
    h.append(arr64("CHEETAH_GX", list(G[0])))
    h.append(arr64("CHEETAH_GY", list(G[1])))
    h.append("/* off-subgroup known-answer point, REF src/signature.rs:387-404 */\n")
    h.append(arr64("CHEETAH_KAT_X", list(o.KAT_X)))
    h.append(arr64("CHEETAH_KAT_Y", list(o.KAT_Y)))
    h.append("/* width-5 NAF of q, least-significant digit first (uniform addition chain of the subgroup check) */\n")
    h.append("#define CHEETAH_Q_WNAF5_LEN %d\n" % len(q_wnaf5))
    h.append(arr8("CHEETAH_Q_WNAF5", q_wnaf5 + [0] * (256 - len(q_wnaf5))))   # zero-padded: the chain loops index up to 255
    h.append("/* Frobenius: (u^i)^p = FP6_FROB[i] * u^i */\n")
    h.append(arr64("FP6_FROB", frob6))
    # Brace initialisers for constants that the device code keeps in __constant__ memory / constexpr tables: the kernels
    # take them from HERE, so swapping params means regenerating this header and nothing else.
    def init_list(vals, fmt):
        return "{" + ", ".join(fmt % v for v in vals) + "}"
    h.append("/* initialiser lists of the same constants for __constant__ / constexpr tables of the device code */\n")
    h.append("#define CHEETAH_Q32_INIT %s\n" % init_list(limbs32(Q, 8), "0x%08xu"))
    h.append("#define SCALAR_R2_32_INIT %s\n" % init_list(limbs32(r2, 8), "0x%08xu"))
    row = list(o.MDS_FIRST_ROW)
    # the device MDS layer (csrc/rescue.cuh: rescue_mds_ark) needs a CIRCULANT matrix with entries below 2^28 (twelve
    # 32-bit x entry products are summed in one 64-bit register without carries)
    assert all(mds[i][j] == row[(j - i) % 12] for i in range(12) for j in range(12)), "MDS matrix is not circulant"
    assert max(row) < (1 << 28), "MDS entries too large for the carry-free accumulation of rescue_mds_ark"
    h.append("#define RESCUE_MDS_ROW_INIT %s\n" % init_list(row, "%du"))
    h.append("#define RESCUE_MDS_MAX_ENTRY %du\n" % max(row))
    h.append("#define RESCUE_MDS_IS_CIRCULANT 1\n\n")
    h.append("/* Rescue circulant MDS first row [RECALLED] and full matrix */\n")
    h.append(arr64("RESCUE_MDS_ROW", list(o.MDS_FIRST_ROW), 6))
    h.append(arr64("RESCUE_MDS", [c for row in mds for c in row], 6))
    h.append("/* Rescue round constants [SPEC-DERIVED], 2*ROUNDS rows of 12 */\n")
    h.append(arr64("RESCUE_ARK", [c for row in ark for c in row]))
    h.append("#endif /* CHEETAH_PARAMS_H */\n")
    os.makedirs(os.path.join(ROOT, "include"), exist_ok=True)
    with open(os.path.join(ROOT, "include", "cheetah_params.h"), "w") as f:
        f.write("".join(h))

    # ---- tables of the windowed Tonelli-Shanks square root in Fp (schnorr-sig_b200/csrc/fp6.cuh: fp_sqrt_or_none) ----
    # p - 1 = 2^32 t, g = 7^t generates the 2-power torsion.  For a != 0: b = a^t = g^e; the discrete log e is read
    # eight bits at a time from b^(2^24), (b g^-e0)^(2^16), ... in the order-256 subgroup (one table lookup each).
    g = root32
    ginv = pow(g, P - 2, P)
    tab_ginv = [pow(ginv, j << (8 * i), P) for i in range(4) for j in range(256)]          # g^(-j 2^(8i))
    tab_half = [pow(ginv, j << (8 * i - 1), P) for i in range(1, 4) for j in range(256)]   # g^(-j 2^(8i-1)), i = 1..3
    g0 = pow(g, 1 << 24, P)                                                                 # order 256
    mu = [pow(g0, j, P) for j in range(256)]
    mult, bits = None, 12
    cand = 0x9E3779B97F4A7C15
    for _ in range(1 << 20):                     # multiplicative hash, injective on the 256 elements
        if len({((v * cand) & (2**64 - 1)) >> (64 - bits) for v in mu}) == 256:
            mult = cand
            break
        cand = (cand * 0xD1342543DE82EF95 + 1) & (2**64 - 1) | 1
    assert mult is not None
    dlog = [0] * (1 << bits)
    for j, v in enumerate(mu):
        dlog[((v * mult) & (2**64 - 1)) >> (64 - bits)] = j
    t = []
    t.append("/* GENERATED by tools/gen_params.py -- do not edit.  Tables of the windowed Tonelli-Shanks square root in the\n"
             " * Goldilocks field (g = FP_ROOT_OF_UNITY_2_32).  Define FP_TABLE_QUAL (e.g. __device__) before including. */\n"
             "#ifndef FP_SQRT_TABLES_H\n#define FP_SQRT_TABLES_H\n#include <stdint.h>\n#ifndef FP_TABLE_QUAL\n#define FP_TABLE_QUAL\n#endif\n\n")
    t.append("#define FP_SQRT_DLOG_MUL 0x%016xULL   /* (v * MUL) >> %d is injective on the order-256 subgroup */\n" % (mult, 64 - bits))
    t.append("#define FP_SQRT_DLOG_SHIFT %d\n\n" % (64 - bits))
    t.append("/* g^(-j 2^(8i)), index 256 i + j */\n")
    t.append(arr64("FP_SQRT_GINV", tab_ginv, 4).replace("static const", "FP_TABLE_QUAL static const"))
    t.append("/* g^(-j 2^(8i-1)) for i = 1..3, index 256 (i-1) + j */\n")
    t.append(arr64("FP_SQRT_HALF", tab_half, 4).replace("static const", "FP_TABLE_QUAL static const"))
    t.append("/* discrete log base g^(2^24) of the order-256 subgroup, indexed by the multiplicative hash */\n")
    t.append(arr8("FP_SQRT_DLOG", dlog, 32, "uint8_t").replace("static const", "FP_TABLE_QUAL static const"))
    t.append("#endif /* FP_SQRT_TABLES_H */\n")
    with open(os.path.join(ROOT, "include", "fp_sqrt_tables.h"), "w") as f:
        f.write("".join(t))
    print("wrote params/params.json, include/cheetah_params.h and include/fp_sqrt_tables.h")


if __name__ == "__main__":
    main()
