"""Instruction mix of k_verify_fast per call-target segment, and an estimate per verification.

usage: sass_mix.py SASS.txt [--kernel k_verify_fast] [--base BASE_SASS.txt]

SASS.txt is `cuobjdump -sass` of the library.  The kernel's code is cut at the targets of its CALL.REL.NOINC
instructions: segment 0 is the kernel body, the others are its out-of-line helpers in address order.  Each segment is
weighted by how often one verification executes it, taken from the ncu capture of the shipped kernel
(profiles/r2_k_verify_fast_hotspots_g11.txt: executed warp instructions / static instructions of the segment).  Those
weights are calls per verification for the straight-line helpers (slope 400, fp6_mul_sub_scaled 400, doubling 249.4,
addition 139.5 -- it skips the scaled subtraction on masked operations) and the trip counts of the
squaring / multiplication loops for the permutation.  They stay valid while a change keeps each helper's control flow,
which field-layer changes do.  With --base, the table of a second build and the change per column are printed too.
"""
import argparse
import collections
import re

# (name, executed warp instructions per verification, static instructions) of the g11 capture, in address order
G11 = [("kernel", 1266352 - 362405 - 167602 - 264284 - 195901 - 260849, 2487),
       ("fp6_slope_nc", 362405, 906),
       ("fp6_mul_sub_scaled", 167602, 419),
       ("permutation", 264284, 3442),
       ("jf_add<true>", 195901, 1404),
       ("jf_dbl<true>", 260849, 1046)]

COLS = ["IMAD.MOV*", "MOV", "moves", "IMAD.X", "IMAD.IADD", "IMAD.SHL", "IADD3(.X)", "IMAD.WIDE*", "IMAD.HI", "total"]


def classify(op):
    out = []
    if op.startswith("IMAD.MOV"):
        out += ["IMAD.MOV*", "moves"]
    elif op == "MOV" or op.startswith("MOV."):
        out += ["MOV", "moves"]
    elif op.startswith("IMAD.X"):
        out.append("IMAD.X")
    elif op.startswith("IMAD.IADD"):
        out.append("IMAD.IADD")
    elif op.startswith("IMAD.SHL"):
        out.append("IMAD.SHL")
    elif op.startswith("IMAD.WIDE"):
        out.append("IMAD.WIDE*")
    elif op.startswith("IMAD.HI"):
        out.append("IMAD.HI")
    elif op.startswith("IADD3"):
        out.append("IADD3(.X)")
    return out + ["total"]


def segments(path, kernel):
    lines = open(path).read().split("\n")
    start = end = None
    for i, l in enumerate(lines):
        if "Function :" in l:
            if start is not None and end is None:
                end = i
            if kernel in l and start is None:
                start = i
    assert start is not None, "kernel %s not found" % kernel
    rx = re.compile(r"^\s+/\*([0-9a-f]+)\*/\s+(.*?);")
    ins = [(int(m.group(1), 16), m.group(2).strip()) for l in lines[start:end] for m in [rx.match(l)] if m]
    targets = sorted({int(m.group(1), 16) for _, s in ins for m in [re.search(r"CALL\.REL\.NOINC\s+(0x[0-9a-f]+)", s)] if m})
    bounds = [0] + targets + [ins[-1][0] + 16]
    segs = []
    for k in range(len(bounds) - 1):
        c = collections.Counter()
        for a, s in ins:
            if bounds[k] <= a < bounds[k + 1]:
                op = re.sub(r"^@!?U?P[T\d]+\s+", "", s).split()[0]
                for col in classify(op):
                    c[col] += 1
        segs.append(c)
    assert len(segs) == len(G11), "expected %d segments (kernel + 5 helpers), found %d" % (len(G11), len(segs))
    return segs


def table(segs, title):
    print("## " + title)
    print()
    print("| segment | calls/verif | " + " | ".join(COLS) + " |")
    print("|---|---|" + "---|" * len(COLS))
    est = collections.Counter()
    for (name, dyn, stat), c in zip(G11, segs):
        wgt = dyn / stat
        print("| %s | %.1f | " % (name, wgt) + " | ".join(str(c[k]) for k in COLS) + " |")
        for k in COLS:
            est[k] += c[k] * wgt
    tot = collections.Counter()
    for c in segs:
        tot.update(c)
    print("| **static, whole kernel** | | " + " | ".join(str(tot[k]) for k in COLS) + " |")
    print("| **per verification (est.)** | | " + " | ".join("%.0f" % est[k] for k in COLS) + " |")
    print()
    return est


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("sass")
    ap.add_argument("--kernel", default="k_verify_fast")
    ap.add_argument("--base")
    a = ap.parse_args()
    if a.base:
        eb = table(segments(a.base, a.kernel), "base: " + a.base)
    e = table(segments(a.sass, a.kernel), a.sass)
    if a.base:
        print("| change per verification | " + " | ".join(COLS) + " |")
        print("|---|" + "---|" * len(COLS))
        print("| | " + " | ".join("%+.1f %%" % (100.0 * (e[k] - eb[k]) / eb[k]) if eb[k] else "-" for k in COLS) + " |")


if __name__ == "__main__":
    main()
