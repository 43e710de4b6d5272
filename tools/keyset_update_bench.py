"""In-place updates of registered key sets (schnorr_b200_keyset_append / _replace / _remove) on one GPU.

  - replace of m keys in sets of K keys, with the block-per-key registration kernel and with the per-thread kernels,
    alternated, warm, median of --reps host wall times per call (every update synchronises before it returns);
  - the per-kernel device time of a 1-key replace with either kernel (torch.profiler, in a pass of its own);
  - append of 1 and 1024 keys at the largest K, with a growth of the buffers (the first append after keyset_create)
    and without;
  - remove of 1 and 1024 keys;
  - keyset_create at several K, this tree against --parent-lib (the library of the parent commit), alternated;
  - verify_registered_many_dev over 2^log2n device-resident signatures on an updated set against a fresh set of the
    same records: equal verdicts, CUDA-event times alternated.
Prints one JSON line (card name, power limit and SM clocks read before and after in the same run).

    python tools/keyset_update_bench.py [--keys 64,1024,16384] [--m 1,8,64,512,4096] [--parent-lib SO] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from registered_batch_bench import card, timed  # noqa: E402

SIZE_MAX = 2**64 - 1


def wall(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3


def med(xs):
    return round(statistics.median(xs), 4)


def create_times(lib, ctx, pk, reps):
    """keyset_create + destroy through a raw library handle -> ms per create (the destroy is not timed)."""
    out = []
    for _ in range(reps):
        h = C.c_void_p()
        t = time.perf_counter()
        rc = lib.schnorr_b200_keyset_create(ctx, pk.shape[0], pk.ctypes.data_as(C.c_void_p), None, None, C.byref(h))
        out.append((time.perf_counter() - t) * 1e3)
        assert rc == 0
        lib.schnorr_b200_keyset_destroy(h)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keys", default="64,1024,16384")
    ap.add_argument("--m", default="1,8,64,512,4096")
    ap.add_argument("--create-keys", default="1,64,1024,16384")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--parent-lib", default=None, help="libschnorr_b200.so of the parent commit (keyset_create A/B)")
    ap.add_argument("--create-reps", type=int, default=3, help="repeats of keyset_create above 1024 keys")
    ap.add_argument("--parts", default="replace,breakdown,append,remove,create,verify")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    parts = set(a.parts.split(","))
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("keyset_update_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"tool": "keyset_update_bench", "card_before": card(0), "torch_device": torch.cuda.get_device_name(0),
           "reps": a.reps, "default_block_threshold": 512, "replace": [], "breakdown_1key": {}, "append": [],
           "remove": [], "create": [], "verify_updated": {}}
    eng = s.Engine(0)
    keys = [int(k) for k in a.keys.split(",")]
    kmax = max(keys)
    pool = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED ^ 0x77, kmax + 4096)
    pk, inf = pool["pk"], pool["inf"]
    rng = np.random.default_rng(1)

    # ---- replace of m keys in a set of K, both kernels alternated
    for K in (keys if "replace" in parts else []):
        ks, _ = eng.register_keys(pk[:K], inf[:K])
        for m in [int(x) for x in a.m.split(",") if int(x) <= K]:
            t = {"block": [], "thread": []}
            for r in range(a.reps + 1):
                for mode, thr in (("block", SIZE_MAX), ("thread", 0)):
                    eng.set_keyset_block_threshold(thr)
                    idx = rng.choice(K, m, replace=False).astype(np.uint32)
                    src = kmax + (r % 2) * (4096 - m if m < 4096 else 0)
                    ms = wall(lambda: eng.keyset_replace(ks, idx, pk[src:src + m], inf[src:src + m]))
                    if r:                       # the first round warms the scratch of this m
                        t[mode].append(ms)
            res["replace"].append({"K": K, "m": m, "block_ms": med(t["block"]), "thread_ms": med(t["thread"]),
                                   "block_all": [round(x, 4) for x in t["block"]],
                                   "thread_all": [round(x, 4) for x in t["thread"]]})
            print(json.dumps(res["replace"][-1]), file=sys.stderr)
        ks.close()
    eng.set_keyset_block_threshold(512)

    # ---- device time per kernel of a 1-key replace (profiled pass)
    from torch.profiler import profile, ProfilerActivity
    ks, _ = eng.register_keys(pk[:64], inf[:64])
    for mode, thr in ((("block", SIZE_MAX), ("thread", 0)) if "breakdown" in parts else ()):
        eng.set_keyset_block_threshold(thr)
        for _ in range(3):
            eng.keyset_replace(ks, [5], pk[kmax:kmax + 1], inf[kmax:kmax + 1])
        calls = 10
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                eng.keyset_replace(ks, [5], pk[kmax:kmax + 1], inf[kmax:kmax + 1])
        per = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA":
                name = ev.name.split("(")[0].replace("void ", "")
                per[name] = per.get(name, 0.0) + ev.device_time / 1e3 / calls
        res["breakdown_1key"][mode] = {k: round(v, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}
    ks.close()
    eng.set_keyset_block_threshold(512)

    # ---- append at the largest K: with a growth (first append after create) and without
    for m in ((1, 1024) if "append" in parts else ()):
        grow, nogrow = [], []
        for r in range(3):
            ks, _ = eng.register_keys(pk[:kmax], inf[:kmax])
            grow.append(wall(lambda: eng.keyset_append(ks, pk[kmax:kmax + m], inf[kmax:kmax + m])))
            for _ in range(2 if r == 0 else 3):                    # the grown buffers hold 1.5 x kmax slots
                nogrow.append(wall(lambda: eng.keyset_append(ks, pk[kmax:kmax + m], inf[kmax:kmax + m])))
            ks.close()
        res["append"].append({"K": kmax, "m": m, "with_growth_ms": med(grow), "without_growth_ms": med(nogrow[1:]),
                              "with_growth_all": [round(x, 3) for x in grow]})
    # ---- remove
    ks, _ = eng.register_keys(pk[:kmax] if "remove" in parts else pk[:1], inf[:kmax] if "remove" in parts else inf[:1])
    for m in ((1, 1024) if "remove" in parts else ()):
        t = []
        for r in range(a.reps + 1):
            idx = rng.choice(kmax, m, replace=False).astype(np.uint32)
            ms = wall(lambda: eng.keyset_remove(ks, idx))
            if r:
                t.append(ms)
        res["remove"].append({"K": kmax, "m": m, "ms": med(t)})
    ks.close()

    # ---- keyset_create: this tree against the parent's library, alternated
    libs = [("tree", eng._L, eng._h)]
    if a.parent_lib:
        P = C.CDLL(os.path.abspath(a.parent_lib))
        P.schnorr_b200_keyset_create.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        P.schnorr_b200_keyset_destroy.argtypes = [C.c_void_p]
        pctx = C.c_void_p()
        assert P.schnorr_b200_create(0, C.byref(pctx)) == 0
        libs.append(("parent", P, pctx))
    for K in ([int(k) for k in a.create_keys.split(",")] if "create" in parts else []):
        row = {"K": K}
        t = {name: [] for name, _, _ in libs}
        reps = a.reps if K <= 1024 else a.create_reps
        for r in range(reps + 1):
            for name, L, ctx in (libs if r % 2 else libs[::-1]):      # which library goes first alternates
                x = create_times(L, ctx, np.ascontiguousarray(pk[:K]), 1)[0]
                if r:
                    t[name].append(x)
        for name in t:
            row[name + "_ms"] = med(t[name])
            row[name + "_all"] = [round(x, 3) for x in t[name]]
        res["create"].append(row)
        print(json.dumps(row), file=sys.stderr)

    # ---- verification on an updated set against a fresh set of the same records
    if "verify" not in parts:
        res["card_after"] = card(0)
        print(json.dumps(res))
        if a.out:
            with open(a.out, "w") as f:
                f.write(json.dumps(res) + "\n")
        return
    K, n = 1024, 1 << a.log2n
    ks, _ = eng.register_keys(pk[:K], inf[:K])
    rep = rng.choice(K, 128, replace=False).astype(np.uint32)
    eng.keyset_replace(ks, rep, pk[kmax:kmax + 128], inf[kmax:kmax + 128])
    rem = np.setdiff1d(rng.choice(K, 64, replace=False), rep).astype(np.uint32)
    eng.keyset_remove(ks, rem)
    eng.keyset_append(ks, pk[kmax + 128:kmax + 256], inf[kmax + 128:kmax + 256])
    mpk, minf = pk[:K].copy(), inf[:K].copy()
    mpk[rep], minf[rep] = pk[kmax:kmax + 128], inf[kmax:kmax + 128]
    mpk[rem] = 0xFF
    mpk, minf = np.concatenate([mpk, pk[kmax + 128:kmax + 256]]), np.concatenate([minf, inf[kmax + 128:kmax + 256]])
    fresh, _ = eng.register_keys(mpk, minf)
    w = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED, n)      # the signatures; indices into the set below
    idx = rng.integers(0, len(mpk), n).astype(np.uint32)
    t = [torch.from_numpy(x).to(dev) for x in (w["sigs"], idx.view(np.int32), w["blob"], w["off"].view(np.int64))]
    outs = {name: torch.full((n,), 255, dtype=torch.uint8, device=dev) for name in ("updated", "fresh")}
    times = {name: [] for name in outs}
    torch.cuda.synchronize(dev)
    for r in range(a.reps + 2):
        for name, kset in (("updated", ks), ("fresh", fresh)):
            ms = timed(torch, lambda: (eng.verify_registered_many_dev(kset, n, t[0], t[1], t[2], t[3], outs[name]),
                                       eng.synchronize()))
            if r >= 2:
                times[name].append(ms)
    same = bool(torch.equal(outs["updated"], outs["fresh"]))
    res["verify_updated"] = {"K": len(mpk), "n": n, "verdicts_equal": same,
                             "updated_ms": med(times["updated"]), "fresh_ms": med(times["fresh"]),
                             "updated_all": [round(x, 3) for x in times["updated"]],
                             "fresh_all": [round(x, 3) for x in times["fresh"]],
                             "verdict_counts": np.bincount(outs["fresh"].cpu().numpy(), minlength=4).tolist()}
    res["card_after"] = card(0)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    assert same, "verdicts on the updated set differ from the fresh set"


if __name__ == "__main__":
    main()
