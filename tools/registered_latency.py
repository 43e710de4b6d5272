#!/usr/bin/env python3
"""Latency of small calls against a registered key set (profiles/r11_registered_one.md):

  host   KeySet.verify_signature, KeySet.verify_keyed (one signature), Engine.verify_registered_many and
         Engine.verify_keyed_registered_many at n = 1, 4, 16,
         128, 384, 512: mean ± sd of 20 host-clock calls (each ends in a synchronise), in the style of latency_probe.py.
         With --other TREE the same measurement runs in a subprocess from that source tree (built first), and the two
         trees alternate, round by round, in this one job.
  device CUDA-event time of the registered kernels (last_kernel_ms) for n = 1 ... 4096 with the block-per-signature
         kernel forced (set_one_threshold(SIZE_MAX)) against the per-thread kernel (set_one_threshold(0)).

The card name, power limit and SM clock are read with nvidia-smi in the same run.  Results go to --out (JSON) and, as a
markdown table, to stdout.  Needs a GPU: without one the engine raises and nothing is measured.

    python tools/registered_latency.py --out r11_registered_one.json [--other PARENT_TREE] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SIZES = (1, 4, 16, 128, 384, 512)
DEVICE_SIZES = (1, 2, 4, 8, 16, 32, 64, 128, 256, 296, 384, 512, 768, 1024, 2048, 4096)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = "unavailable (%s)" % e
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if "," in out else {"nvidia-smi": out}


def timeit(fn, reps=20):
    import numpy as np
    fn()
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)) * 1e3, float(np.std(ts)) * 1e3


def workload(eng, n, n_keys=16, seed=5):
    import numpy as np
    import schnorr_sig_b200 as sb
    rng = np.random.default_rng(seed)
    sk = sb.synth.scalars(seed, 1, n_keys)
    pk, inf = eng.keygen(sk)
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    msgs = [rng.bytes(80) for _ in range(n)]
    blob = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()
    off = np.arange(n + 1, dtype=np.uint64) * 80
    sigs = eng.sign_many(sk[idx], pk[idx], inf[idx], blob, off, sb.synth.scalars(seed, 2, n))
    rec = np.ascontiguousarray(np.concatenate([eng.compress(pk[idx], inf[idx]), sigs], axis=1))
    return dict(sk=sk, pk=pk, inf=inf, idx=idx, msgs=msgs, blob=blob, off=off, sigs=sigs, rec=rec)


def measure_host():
    """One round of the host-API latencies of the tree this process imports -> {case: [mean, sd]}."""
    import numpy as np
    import schnorr_sig_b200 as sb
    eng = sb.default_engine(0)
    w = workload(eng, max(HOST_SIZES))
    ks, status = eng.register_keys(w["pk"], w["inf"])
    assert not status.any()
    keys = [sb.PublicKey.from_bytes(bytes(b)) for b in eng.compress(w["pk"], w["inf"])]
    api_set = sb.KeySet(keys)
    sig = sb.Signature.from_bytes(bytes(w["sigs"][0]))
    keyed = bytes(w["rec"][0])
    msg = w["msgs"][0]
    k0 = int(w["idx"][0])
    assert api_set.verify_signature(k0, sig, msg).is_ok() and api_set.verify_keyed(keyed, msg).is_ok()
    out = {"KeySet.verify_signature": timeit(lambda: api_set.verify_signature(k0, sig, msg)),
           "KeySet.verify_keyed": timeit(lambda: api_set.verify_keyed(keyed, msg))}
    for n in HOST_SIZES:
        off = w["off"][:n + 1]
        blob = w["blob"][:int(off[-1])]
        args = (ks, w["sigs"][:n], w["idx"][:n], blob, off)
        assert (eng.verify_registered_many(*args) == 0).all()
        out["verify_registered_many n=%d" % n] = timeit(lambda: eng.verify_registered_many(*args))
        kargs = (ks, w["rec"][:n], blob, off)
        assert (eng.verify_keyed_registered_many(*kargs) == 0).all()
        out["verify_keyed_registered_many n=%d" % n] = timeit(lambda: eng.verify_keyed_registered_many(*kargs))
    return {k: list(v) for k, v in out.items()}


def measure_device(reps=20):
    """CUDA-event time of the registered kernels (block form forced against the per-thread form) -> {n: {...}}."""
    import numpy as np
    import schnorr_sig_b200 as sb
    eng = sb.default_engine(0)
    w = workload(eng, max(DEVICE_SIZES), seed=9)
    ks, _ = eng.register_keys(w["pk"], w["inf"])
    out = {}
    for n in DEVICE_SIZES:
        off = w["off"][:n + 1]
        args = (ks, w["sigs"][:n], w["idx"][:n], w["blob"][:int(off[-1])], off)
        row = {}
        for name, thr in (("block", 2**62), ("thread", 0)):
            eng.set_one_threshold(thr)
            assert (eng.verify_registered_many(*args) == 0).all()
            ms = []
            for _ in range(reps):
                eng.verify_registered_many(*args)
                ms.append(eng.last_kernel_ms())
            row[name] = [float(np.mean(ms)), float(np.std(ms))]
        eng.set_one_threshold(512)
        out[n] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--other", help="another source tree (e.g. the parent commit) to alternate with")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        sys.path.insert(0, os.getcwd())
        json.dump(measure_host(), sys.stdout)
        return
    trees = {"tree": ROOT}
    if a.other:
        trees["other"] = os.path.abspath(a.other)
    for t in trees.values():
        subprocess.check_call([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=t)
    res = {"card_before": card(), "host": {k: [] for k in trees}}
    for _ in range(a.rounds):
        for name, t in trees.items():
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--out", "-"], cwd=t,
                               capture_output=True, text=True, check=True)
            res["host"][name].append(json.loads(p.stdout))
    sys.path.insert(0, ROOT)
    res["device"] = measure_device()
    res["card_after"] = card()
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("card: %s" % res["card_before"])
    cases = list(res["host"]["tree"][0])
    print("| case | " + " | ".join("%s round %d ms" % (k, r) for r in range(a.rounds) for k in trees) + " |")
    print("|---|" + "---|" * (a.rounds * len(trees)))
    for c in cases:
        cells = ["%.3f ± %.3f" % tuple(res["host"][k][r][c]) for r in range(a.rounds) for k in trees]
        print("| %s | %s |" % (c, " | ".join(cells)))
    print()
    print("| n | block kernel ms | per-thread kernel ms |")
    print("|---|---|---|")
    for n, row in res["device"].items():
        print("| %d | %.3f ± %.3f | %.3f ± %.3f |" % (n, *row["block"], *row["thread"]))


if __name__ == "__main__":
    main()
