"""Batch verification against a registered key set against verify_batch on one GPU.  For every n x K (8-byte messages,
keys drawn uniformly from a set of K, randomisers from a fixed seed): device-resident times of verify_batch_dev on the
gathered key records and of verify_batch_registered_dev on the same buffers (CUDA events, warmed up, alternated, median
of --reps), the registered call with each path forced (key side summed per key / per-signature points on the gathered
records), the MSM points of the path the default selection took, and the host-API times of both entry points.  The
verdict, lhs and rhs of every variant must be equal.  A profiled run at 2^20 gives the time of the key side alone
(k_keyset_scalar_sum + k_keyset_batch_term + the reduction of the key terms) at K = 1 and 16 384.
Prints one JSON line (card name, power limit and SM clocks read in the same run).

    python tools/registered_batch_bench.py [--sizes 10,12,16,20] [--keys 1,64,1024,16384] [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALWAYS, NEVER = 0, 1 << 62   # set_registered_batch_threshold: sum per key whenever allowed / never
DEFAULT = 64                 # the library's default (REG_BATCH_MIN_PER_KEY)


def card(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(zip(q.split(","), out))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def timed(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def result(res):
    r = res.cpu().numpy()
    return int(r[0]), bytes(r[8:105]), bytes(r[112:209])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="10,12,16,20", help="log2 of the batch sizes")
    ap.add_argument("--keys", default="1,64,1024,16384")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--profile-keys", default="1,16384", help="K of the profiled key-side runs (at the largest size)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("registered_batch_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    eng = s.Engine(0)
    stream = torch.cuda.Stream(dev)          # the engine enqueues on this stream: the events below bracket its work
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    sizes = [1 << int(x) for x in a.sizes.split(",")]
    nmax = max(sizes)
    seed = s.synth.DEFAULT_SEED
    blob, off = s.synth.messages(seed, 3, nmax, 8)
    nonce = s.synth.scalars(seed, 2, nmax)
    rand = s.synth.scalars(seed, 5, nmax)
    res = {"tool": "registered_batch_bench", "card": card(0), "torch_device": torch.cuda.get_device_name(0),
           "msg_len": 8, "reps": a.reps, "library": s._lib.library_path().rsplit("/", 1)[-1], "points": [],
           "key_side": []}
    t_blob = torch.from_numpy(blob).to(dev)
    t_off = torch.from_numpy(off.view(np.int64)).to(dev)
    t_rand = torch.from_numpy(rand).to(dev)
    profile_keys = {int(k) for k in a.profile_keys.split(",")}
    for K in [int(k) for k in a.keys.split(",")]:
        keys = s.synth.signed_workload(eng, seed ^ K, K)
        ks, status = eng.register_keys(keys["pk"], keys["inf"])
        assert not status.any()
        idx = np.random.default_rng(K).integers(0, K, nmax).astype(np.uint32)
        sigs = eng.sign_many(keys["sk"][idx], keys["pk"][idx], keys["inf"][idx], blob, off, nonce)
        pk, inf = keys["pk"][idx], keys["inf"][idx]
        t_sig, t_idx = torch.from_numpy(sigs).to(dev), torch.from_numpy(idx.view(np.int32)).to(dev)
        t_pk, t_inf = torch.from_numpy(pk).to(dev), torch.from_numpy(inf).to(dev)
        outs = {v: torch.zeros(216, dtype=torch.uint8, device=dev) for v in ("batch", "reg", "reg_sum", "reg_gather")}
        for n in sizes:
            def batch():
                eng.verify_batch_dev(n, t_sig, t_pk, t_inf, t_blob, t_off, t_rand, outs["batch"])

            def reg(variant="reg", threshold=None):
                if threshold is not None:
                    eng.set_registered_batch_threshold(threshold)
                eng.verify_batch_registered_dev(ks, n, t_sig, t_idx, t_blob, t_off, t_rand, outs[variant])
                if threshold is not None:
                    eng.set_registered_batch_threshold(DEFAULT)
            variants = {"batch": batch, "reg": reg, "reg_sum": lambda: reg("reg_sum", ALWAYS),
                        "reg_gather": lambda: reg("reg_gather", NEVER)}
            reg()
            torch.cuda.synchronize(dev)
            points = eng.last_batch_points()
            for f in variants.values():               # warm-up
                f()
            torch.cuda.synchronize(dev)
            ms = {v: [] for v in variants}
            for _ in range(a.reps):                   # alternated
                for v, f in variants.items():
                    ms[v].append(timed(torch, f))
            want = result(outs["batch"])
            assert want[0] == 0
            for v in variants:
                assert result(outs[v]) == want, (K, n, v)
            # host API (copies in, kernels, copy back, synchronise)
            hb, hr = [], []
            for _ in range(a.host_reps):
                t0 = time.perf_counter()
                rb = eng.verify_batch(sigs[:n], pk[:n], inf[:n], blob[:8 * n], off[:n + 1], rand[:n])
                hb.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                rr = eng.verify_batch_registered(ks, sigs[:n], idx[:n], blob[:8 * n], off[:n + 1], rand[:n])
                hr.append(time.perf_counter() - t0)
                assert (rb[0], bytes(rb[1]), bytes(rb[2])) == want and (rr[0], bytes(rr[1]), bytes(rr[2])) == want
            med = {v: float(np.median(t)) for v, t in ms.items()}
            res["points"].append({
                "n": n, "K": K, "points": points, "path": {0: "block", n: "sum_per_key", 2 * n: "gathered"}.get(points),
                "verify_batch_dev_ms": med["batch"], "registered_dev_ms": med["reg"],
                "registered_sum_forced_ms": med["reg_sum"], "registered_gathered_forced_ms": med["reg_gather"],
                "speedup": med["batch"] / med["reg"],
                "spread_ms": {v: [float(min(t)), float(max(t))] for v, t in ms.items()},
                "verify_batch_host_ms": 1e3 * float(np.median(hb)), "registered_host_ms": 1e3 * float(np.median(hr)),
                "outputs_equal": True})
            print(json.dumps(res["points"][-1]), file=sys.stderr)
        if K in profile_keys:                          # the key side alone, in a profiled run of its own
            from torch.profiler import ProfilerActivity, profile
            n = nmax
            eng.set_registered_batch_threshold(ALWAYS)
            eng.verify_batch_registered_dev(ks, n, t_sig, t_idx, t_blob, t_off, t_rand, outs["reg_sum"])
            torch.cuda.synchronize(dev)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    eng.verify_batch_registered_dev(ks, n, t_sig, t_idx, t_blob, t_off, t_rand, outs["reg_sum"])
                torch.cuda.synchronize(dev)
            eng.set_registered_batch_threshold(DEFAULT)
            kern = {}
            for e in prof.key_averages():
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                kern[e.key] = kern.get(e.key, 0.0) + t / 1e3 / 3      # ms per batch
            pick = lambda tag: sum(v for k, v in kern.items() if tag in k)   # noqa: E731
            total = sum(kern.values())
            res["key_side"].append({
                "n": n, "K": K, "scalar_sum_ms": pick("k_keyset_scalar_sum"), "key_terms_ms": pick("k_keyset_batch_term"),
                "key_term_reduce_ms": pick("k_batch_small_reduce"), "msm_segment_sum_ms": pick("k_msm_segment_sum"),
                "all_kernels_ms": total})
        ks.close()
        del t_sig, t_idx, t_pk, t_inf
        torch.cuda.empty_cache()
    res["card_after"] = card(0)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
