"""KeyedSignature records against a registered key set against verify_keyed_many on one GPU.  2^20 device-resident
records (8-byte messages, one invalid signature per 1024), keys drawn from a set of K; a fraction of the records is
signed under keys outside the set (the misses).  For every K x miss fraction: CUDA-event times, warmed up, alternated,
median of --reps, of verify_keyed_many_dev, verify_keyed_registered_many_dev, verify_registered_many_dev on the
indices of a lookup (the floor: the registered path without the keyed front end) and keyset_lookup_dev alone; then
the host forms of the first two.  The verdicts of every keyed variant must be equal (and the floor's at 0 misses).
Registration time per key is measured for every K.  Prints one JSON line (card name, power limit and SM clocks read
in the same run).

    python tools/keyed_registered_bench.py [--log2n 20] [--keys 1,64,1024,16384] [--miss 0,1/1024,1/16,1/2,1] [--out FILE]
"""
import argparse
import json
import os
import sys
import time
from fractions import Fraction

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from registered_batch_bench import card, timed  # noqa: E402

OUTSIDE = 64     # keys outside the set that sign the misses


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--keys", default="1,64,1024,16384")
    ap.add_argument("--miss", default="0,1/1024,1/16,1/2,1")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("keyed_registered_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    eng = s.Engine(0)
    stream = torch.cuda.Stream(dev)          # the engine enqueues on this stream: the events below bracket its work
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    n = 1 << a.log2n
    seed = s.synth.DEFAULT_SEED
    blob, off = s.synth.messages(seed, 3, n, 8)
    nonce = s.synth.scalars(seed, 2, n)
    misses = [Fraction(m) for m in a.miss.split(",")]
    res = {"tool": "keyed_registered_bench", "card": card(0), "torch_device": torch.cuda.get_device_name(0),
           "n": n, "msg_len": 8, "reps": a.reps, "points": [], "registration": []}
    t_blob = torch.from_numpy(blob).to(dev)
    t_off = torch.from_numpy(off.view(np.int64)).to(dev)
    outside = s.synth.signed_workload(eng, seed ^ 0x5A5A, OUTSIDE)
    for K in [int(k) for k in a.keys.split(",")]:
        keys = s.synth.signed_workload(eng, seed ^ K, K)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        ks, status = eng.register_keys(keys["pk"], keys["inf"])
        reg_s = time.perf_counter() - t0
        assert not status.any()
        res["registration"].append({"K": K, "ms": 1e3 * reg_s, "us_per_key": 1e6 * reg_s / K})
        rng = np.random.default_rng(K)
        idx_in = rng.integers(0, K, n)
        order = rng.permutation(n)
        sk_all = np.concatenate([keys["sk"], outside["sk"]])
        pk_all = np.concatenate([keys["pk"], outside["pk"]])
        inf_all = np.concatenate([keys["inf"], outside["inf"]])
        for m in misses:
            owner = idx_in.copy()
            n_miss = int(m * n)
            owner[order[:n_miss]] = K + rng.integers(0, OUTSIDE, n_miss)
            sigs = eng.sign_many(sk_all[owner], pk_all[owner], inf_all[owner], blob, off, nonce)
            sigs[512::1024, 49] ^= 1                          # one invalid signature per 1024
            rec = np.ascontiguousarray(np.concatenate([eng.compress(pk_all, inf_all)[owner], sigs], axis=1))
            t_rec = torch.from_numpy(rec).to(dev)
            t_key = torch.from_numpy(np.ascontiguousarray(rec[:, :49])).to(dev)
            t_sig = torch.from_numpy(np.ascontiguousarray(sigs)).to(dev)
            t_idx = torch.zeros(n, dtype=torch.int32, device=dev)
            outs = {v: torch.zeros(n, dtype=torch.uint8, device=dev) for v in ("keyed", "keyed_reg", "floor")}
            eng.keyset_lookup_dev(ks, n, t_key, t_idx)
            variants = {
                "keyed": lambda: eng.verify_keyed_many_dev(n, t_rec, t_blob, t_off, outs["keyed"]),
                "keyed_reg": lambda: eng.verify_keyed_registered_many_dev(ks, n, t_rec, t_blob, t_off, outs["keyed_reg"]),
                "floor": lambda: eng.verify_registered_many_dev(ks, n, t_sig, t_idx, t_blob, t_off, outs["floor"]),
                "lookup": lambda: eng.keyset_lookup_dev(ks, n, t_key, t_idx),
            }
            for f in variants.values():                   # warm-up
                f()
            torch.cuda.synchronize(dev)
            ms = {v: [] for v in variants}
            for _ in range(a.reps):                       # alternated
                for v, f in variants.items():
                    ms[v].append(timed(torch, f))
            want = outs["keyed"].cpu().numpy()
            assert np.array_equal(outs["keyed_reg"].cpu().numpy(), want), (K, m)
            assert (t_idx.cpu().numpy().view(np.uint32) == 0xFFFFFFFF).sum() == n_miss
            if n_miss == 0:
                assert np.array_equal(outs["floor"].cpu().numpy(), want), K
            hk, hr = [], []
            for _ in range(a.host_reps):
                t0 = time.perf_counter()
                vk = eng.verify_keyed_many(rec, blob, off)
                hk.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                vr = eng.verify_keyed_registered_many(ks, rec, blob, off)
                hr.append(time.perf_counter() - t0)
                assert np.array_equal(vk, want) and np.array_equal(vr, want)
            med = {v: float(np.median(t)) for v, t in ms.items()}
            res["points"].append({
                "K": K, "miss": str(m), "misses": n_miss,
                "keyed_many_dev_ms": med["keyed"], "keyed_registered_dev_ms": med["keyed_reg"],
                "registered_floor_dev_ms": med["floor"], "lookup_dev_ms": med["lookup"],
                "speedup": med["keyed"] / med["keyed_reg"],
                "spread_ms": {v: [float(min(t)), float(max(t))] for v, t in ms.items()},
                "keyed_many_host_ms": 1e3 * float(np.median(hk)), "keyed_registered_host_ms": 1e3 * float(np.median(hr)),
                "verdicts_equal": True, "invalid": int((want == 2).sum())})
            print(json.dumps(res["points"][-1]), file=sys.stderr)
            del t_rec, t_key, t_sig, t_idx, outs
        ks.close()
        torch.cuda.empty_cache()
    res["card_after"] = card(0)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
