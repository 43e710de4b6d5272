"""Batch verification over KeyedSignature wire records on one GPU.  For every n x K x miss fraction (8-byte messages, keys
drawn uniformly from a set of K, the given fraction of the records under 16 keys outside the set, randomisers from a
fixed seed), device-resident times (CUDA events, warmed up, the variants alternated, median of --reps with min / max)
of:
  batch        verify_batch_dev on the decoded keys: what a caller pays today after decompressing the keys (the
               decompression itself is the separate column decompress_host_ms, a host call with its copies)
  keyed        verify_batch_keyed_dev
  keyed_reg    verify_batch_keyed_registered_dev (MSM planned for 2n points)
  registered   verify_batch_registered_dev on the lookup indices (0 misses only: the floor of keyed_reg)
and the host-API times of verify_batch_keyed and verify_batch_keyed_registered (the latter plans n + m points).  The
verdict, lhs and rhs of every variant must be equal.  Prints one JSON line (card name, power limit and SM clocks read in
the same run).

    python tools/keyed_batch_bench.py [--sizes 16,20] [--keys 1,64,1024,16384] [--misses 0,0.0009765625,0.0625,0.5]
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

from registered_batch_bench import card, result, timed   # noqa: E402

OUTSIDE = 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="16,20", help="log2 of the batch sizes")
    ap.add_argument("--keys", default="1,64,1024,16384")
    ap.add_argument("--misses", default="0,0.0009765625,0.0625,0.5")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("keyed_batch_bench needs a CUDA device")
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
    res = {"tool": "keyed_batch_bench", "card": card(0), "torch_device": torch.cuda.get_device_name(0), "msg_len": 8,
           "reps": a.reps, "points": []}
    t_blob = torch.from_numpy(blob).to(dev)
    t_off = torch.from_numpy(off.view(np.int64)).to(dev)
    t_rand = torch.from_numpy(rand).to(dev)
    for K in [int(k) for k in a.keys.split(",")]:
        keys = s.synth.signed_workload(eng, seed ^ K, K + OUTSIDE)
        ks, status = eng.register_keys(keys["pk"][:K], keys["inf"][:K])
        assert not status.any()
        enc = eng.compress(keys["pk"], keys["inf"])
        for f in [float(x) for x in a.misses.split(",")]:
            rng = np.random.default_rng(K)
            owner = rng.integers(0, K, nmax)
            out = rng.random(nmax) < f
            owner[out] = K + rng.integers(0, OUTSIDE, int(out.sum()))
            sigs = eng.sign_many(keys["sk"][owner], keys["pk"][owner], keys["inf"][owner], blob, off, nonce)
            rec = np.ascontiguousarray(np.concatenate([enc[owner], sigs], axis=1))
            pk, inf = keys["pk"][owner], keys["inf"][owner]
            idx = eng.keyset_lookup(ks, rec[:, :49])
            t_rec, t_sig = torch.from_numpy(rec).to(dev), torch.from_numpy(sigs).to(dev)
            t_pk, t_inf = torch.from_numpy(pk).to(dev), torch.from_numpy(inf).to(dev)
            t_idx = torch.from_numpy(idx.view(np.int32)).to(dev)
            outs = {v: torch.zeros(216, dtype=torch.uint8, device=dev) for v in ("batch", "keyed", "keyed_reg", "registered")}
            for n in sizes:
                m = int((idx[:n] == 0xFFFFFFFF).sum())
                variants = {
                    "batch": lambda: eng.verify_batch_dev(n, t_sig, t_pk, t_inf, t_blob, t_off, t_rand, outs["batch"]),
                    "keyed": lambda: eng.verify_batch_keyed_dev(n, t_rec, t_blob, t_off, t_rand, outs["keyed"]),
                    "keyed_reg": lambda: eng.verify_batch_keyed_registered_dev(ks, n, t_rec, t_blob, t_off, t_rand,
                                                                               outs["keyed_reg"]),
                }
                if m == 0:
                    variants["registered"] = lambda: eng.verify_batch_registered_dev(ks, n, t_sig, t_idx, t_blob, t_off,
                                                                                     t_rand, outs["registered"])
                for fn in variants.values():           # warm-up
                    fn()
                torch.cuda.synchronize(dev)
                ms = {v: [] for v in variants}
                for _ in range(a.reps):                # alternated
                    for v, fn in variants.items():
                        ms[v].append(timed(torch, fn))
                want = result(outs["batch"])
                assert want[0] == 0
                for v in variants:
                    assert result(outs[v]) == want, (K, f, n, v)
                hk, hr, hd = [], [], []
                for _ in range(a.host_reps):
                    t0 = time.perf_counter()
                    rk = eng.verify_batch_keyed(rec[:n], blob[:8 * n], off[:n + 1], rand[:n])
                    hk.append(time.perf_counter() - t0)
                    t0 = time.perf_counter()
                    rr = eng.verify_batch_keyed_registered(ks, rec[:n], blob[:8 * n], off[:n + 1], rand[:n])
                    hr.append(time.perf_counter() - t0)
                    host_points = eng.last_batch_points()
                    t0 = time.perf_counter()
                    eng.decompress(rec[:n, :49])
                    hd.append(time.perf_counter() - t0)
                    for r in (rk, rr):
                        assert (r[0], bytes(r[1]), bytes(r[2])) == want
                med = {v: float(np.median(t)) for v, t in ms.items()}
                res["points"].append({
                    "n": n, "K": K, "miss_fraction": f, "misses": m, "host_points": host_points,
                    "batch_dev_ms": med["batch"], "keyed_dev_ms": med["keyed"], "keyed_reg_dev_ms": med["keyed_reg"],
                    "registered_dev_ms": med.get("registered"),
                    "spread_ms": {v: [float(min(t)), float(max(t))] for v, t in ms.items()},
                    "keyed_host_ms": 1e3 * float(np.median(hk)), "keyed_reg_host_ms": 1e3 * float(np.median(hr)),
                    "decompress_host_ms": 1e3 * float(np.median(hd)), "outputs_equal": True})
                print(json.dumps(res["points"][-1]), file=sys.stderr)
            del t_rec, t_sig, t_pk, t_inf, t_idx
            torch.cuda.empty_cache()
        ks.close()
    res["card_after"] = card(0)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
