"""Failed-batch localisation against batch verification on the same inputs, on one device and on a multi-device context.

For each context and each culprit pattern, the host wall time (the calls end in a device synchronise) of
  verify_batch / verify_batch_seeded           the batch that fails (or passes, with no culprit)
  locate_invalid / locate_invalid_seeded       the culprits of that batch
warmed up, median of --reps with min / max, every run's verdict and flags checked.  Patterns: no culprit (one whole
check), one culprit (deep bisection), 16 spread, and 1 in 40 (every item through the per-item check).  Contexts:
  single     a single-device context, n = 2^size_log2 and, for comparison, every n the multi contexts run
  multi      every GPU of the machine listed once, n = 2^size_log2 x the GPU count
  repeat     on a machine with one GPU only, that GPU listed --repeat times (n = 2^size_log2 x --repeat): independent
             contexts sharing one GPU, so these numbers measure the cost of the sharded path, not scaling
Prints one JSON line (card name, power limit and SM clocks read in the same run).

    python tools/locate_bench.py [--size-log2 20] [--reps 5] [--out locate.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from registered_batch_bench import card   # noqa: E402


def stats(ts):
    return {"median_ms": float(np.median(ts)), "min_ms": float(min(ts)), "max_ms": float(max(ts))}


def culprits(n, pattern):
    if pattern == "none":
        return []
    if pattern == "one":
        return [n // 3 + 17]
    if pattern == "spread16":
        return [int(i) for i in np.linspace(5, n - 5, 16).astype(np.int64)]
    return list(range(7, n, 40))


def measure(eng, w, pattern, reps):
    n = w["sigs"].shape[0]
    bad = culprits(n, pattern)
    sigs = w["sigs"].copy()
    sigs[bad, 49] ^= 1
    args = (sigs, w["pk"], w["inf"], w["blob"], w["off"])
    seed = os.urandom(32)
    rand = eng.batch_randomizers(n, seed)
    want_v = 2 if bad else 0
    calls = {
        "verify_batch": lambda: eng.verify_batch(*args, rand)[0] == want_v,
        "verify_batch_seeded": lambda: eng.verify_batch_seeded(*args, seed)[0] == want_v,
        "locate_invalid": lambda: list(np.nonzero(eng.locate_invalid(*args, rand))[0]) == bad,
        "locate_invalid_seeded": lambda: list(np.nonzero(eng.locate_invalid_seeded(*args, seed))[0]) == bad,
    }
    for name, fn in calls.items():        # warm-up, and the arena grown to this shape
        assert fn(), name
    ts = {k: [] for k in calls}
    for _ in range(reps):                 # alternated, so drift on the card touches every call alike
        for name, fn in calls.items():
            t0 = time.perf_counter()
            ok = fn()
            ts[name].append(1e3 * (time.perf_counter() - t0))
            assert ok, name
    return {"pattern": pattern, "culprits": len(bad), **{k: stats(v) for k, v in ts.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size-log2", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--repeat", type=int, default=2, help="listings of the only GPU on a one-GPU machine")
    ap.add_argument("--patterns", default="none,one,spread16,one_in_40")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("locate_bench needs a CUDA device")
    g = torch.cuda.device_count()
    res = {"tool": "locate_bench", "gpus": g, "cards": [card(k) for k in range(g)], "size_log2": a.size_log2,
           "reps": a.reps, "runs": []}
    base = 1 << a.size_log2
    single = s.Engine(0)
    if g > 1:
        contexts = [("multi", list(range(g)), base * g)]
    else:
        contexts = [("repeat", [0] * a.repeat, base * a.repeat)]
    sizes = sorted({base} | {n for _, _, n in contexts})
    patterns = a.patterns.split(",")
    work = {n: s.synth.signed_workload(single, s.synth.DEFAULT_SEED + 7, n) for n in sizes}
    for n in sizes:
        for p in patterns:
            r = {"context": "single", "devices": [0], "n": n, **measure(single, work[n], p, a.reps)}
            res["runs"].append(r)
            print(json.dumps(r), file=sys.stderr)
    for label, devs, n in contexts:
        eng = s.Engine(devs)
        for p in patterns:
            r = {"context": label, "devices": devs, "n": n, **measure(eng, work[n], p, a.reps)}
            res["runs"].append(r)
            print(json.dumps(r), file=sys.stderr)
        eng.close()
    single.close()
    res["cards_after"] = [card(k) for k in range(g)]
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
