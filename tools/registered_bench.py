"""Registered key sets against verify_many on one GPU: 2^20 signatures with 8-byte messages, one invalid signature in
1024, keys drawn uniformly from a set of K.  Per K: device-resident rates of verify_many_dev and
verify_registered_many_dev on the same device buffers (CUDA events, warmed up, the two alternated), the host-API rate
of both, the registration time per key, the challenge-hash kernel on the same inputs (the part of a registered
verification that is not table additions), and whether the key tables fit the 126 MB L2.  The verdicts of both paths
must be equal.  A small-call sweep compares the two at the sizes where verify_many switches to its latency kernels.
Prints one JSON line (card name, power limit and SM clocks read in the same run).

    python tools/registered_bench.py [--keys 1,64,1024,16384] [--log2n 20] [--reps 5] [--out FILE]
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

import cost_model  # noqa: E402

L2_BYTES = 126 * 2**20


def card(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(zip(q.split(","), out))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def timed(torch, fn, reps):
    """median ms of fn() over reps runs, CUDA events on the current stream"""
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keys", default="1,64,1024,16384")
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--small", default="1,128,512,2048,8192")
    ap.add_argument("--kt-w", type=int, default=8, help="KT_W the library was built with (table size per key)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    table_bytes_per_key = (255 // a.kt_w + 1) * ((1 << (a.kt_w - 1)) + 1) * 96
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("registered_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    eng = s.Engine(0)
    # the engine enqueues on a torch stream of its own so that the events below bracket its kernels (a null handle,
    # torch's default stream, would select the engine's private stream)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    n = 1 << a.log2n
    seed = s.synth.DEFAULT_SEED
    blob, off = s.synth.messages(seed, 3, n, 8)
    nonce = s.synth.scalars(seed, 2, n)
    peak, _ = eng.imad_peak()
    res = {"tool": "registered_bench", "card": card(0), "torch_device": torch.cuda.get_device_name(0), "n": n,
           "msg_len": 8, "invalid_every": 1024, "library": s._lib.library_path().rsplit("/", 1)[-1],
           "imad_peak_w_per_s": peak, "w_executed_fast_L8": cost_model.W_EXECUTED_FAST_L8,
           "w_executed_reg_L8": cost_model.W_EXECUTED_REG_L8, "per_K": []}
    t_blob = torch.from_numpy(blob).to(dev)
    t_off = torch.from_numpy(off.view(np.int64)).to(dev)
    for K in [int(k) for k in a.keys.split(",")]:
        keys = s.synth.signed_workload(eng, seed ^ K, K)     # K key pairs (their own messages are unused)
        rng = np.random.default_rng(K)
        idx = rng.integers(0, K, n).astype(np.uint32)
        sigs = eng.sign_many(keys["sk"][idx], keys["pk"][idx], keys["inf"][idx], blob, off, nonce)
        bad = np.arange(512, n, 1024)
        sigs[bad, 49] ^= 1                                   # e +- 1: one invalid signature in 1024
        pk, inf = keys["pk"][idx], keys["inf"][idx]
        torch.cuda.synchronize(dev)
        free0 = torch.cuda.mem_get_info(dev)[0]
        t0 = time.perf_counter()
        ks, status = eng.register_keys(keys["pk"], keys["inf"])
        reg_s = time.perf_counter() - t0
        set_bytes = free0 - torch.cuda.mem_get_info(dev)[0]   # tables, records and registration scratch
        assert not status.any()
        t_sig, t_idx = torch.from_numpy(sigs).to(dev), torch.from_numpy(idx.view(np.int32)).to(dev)
        t_pk, t_inf = torch.from_numpy(pk).to(dev), torch.from_numpy(inf).to(dev)
        out_vm = torch.full((n,), 255, dtype=torch.uint8, device=dev)
        out_rg = torch.full((n,), 255, dtype=torch.uint8, device=dev)
        digests = torch.empty((n, 32), dtype=torch.uint8, device=dev)
        rx = t_sig[:, :48].contiguous()
        vm = lambda: eng.verify_many_dev(n, t_sig, t_pk, t_inf, t_blob, t_off, out_vm)        # noqa: E731
        rg = lambda: eng.verify_registered_many_dev(ks, n, t_sig, t_idx, t_blob, t_off, out_rg)  # noqa: E731
        hs = lambda: eng.hash_messages_dev(n, rx, t_pk, t_blob, t_off, digests)                # noqa: E731
        for f in (vm, rg, hs):                               # warm-up
            f()
        torch.cuda.synchronize(dev)
        ms_vm, ms_rg = [], []
        for _ in range(a.reps):                              # alternated
            ms_vm.append(timed(torch, vm, 1))
            ms_rg.append(timed(torch, rg, 1))
        ms_hash = timed(torch, hs, a.reps)
        v_vm, v_rg = out_vm.cpu().numpy(), out_rg.cpu().numpy()
        assert np.array_equal(v_vm, v_rg), "verdicts differ"
        assert (v_rg == 2).sum() == len(bad) and (v_rg == 0).sum() == n - len(bad)
        # host API (copies in, kernels, copy back, synchronise)
        eng.verify_many(sigs, pk, inf, blob, off)
        eng.verify_registered_many(ks, sigs, idx, blob, off)
        h_vm, h_rg = [], []
        for _ in range(max(2, a.reps // 2)):
            t0 = time.perf_counter(); hv = eng.verify_many(sigs, pk, inf, blob, off); h_vm.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); hr = eng.verify_registered_many(ks, sigs, idx, blob, off); h_rg.append(time.perf_counter() - t0)
        assert np.array_equal(hv, v_vm) and np.array_equal(hr, v_vm)
        mvm, mrg = float(np.median(ms_vm)), float(np.median(ms_rg))
        rate_rg = n / (mrg * 1e-3)
        res["per_K"].append({
            "K": K, "kt_w": a.kt_w, "table_bytes": K * table_bytes_per_key, "device_bytes_allocated": set_bytes,
            "tables_fit_l2": K * table_bytes_per_key <= L2_BYTES,
            "verify_many_dev_ms": mvm, "registered_dev_ms": mrg, "hash_kernel_ms": ms_hash,
            "verify_many_dev_rate": n / (mvm * 1e-3), "registered_dev_rate": rate_rg, "speedup_dev": mvm / mrg,
            "verify_many_host_ms": 1e3 * float(np.median(h_vm)), "registered_host_ms": 1e3 * float(np.median(h_rg)),
            "registered_host_over_dev": 1e3 * float(np.median(h_rg)) / mrg,
            "registration_s": reg_s, "registration_us_per_key": 1e6 * reg_s / K,
            "frac_executed_reg": cost_model.W_EXECUTED_REG_L8 * rate_rg / peak,
            "verdicts_equal": True})
        ks.close()
        del t_sig, t_idx, t_pk, t_inf, out_vm, out_rg, digests, rx
        torch.cuda.empty_cache()
    # small calls: verify_many picks its latency kernels below 10 241 signatures
    K = 64
    keys = s.synth.signed_workload(eng, seed ^ 7, K)
    ks, _ = eng.register_keys(keys["pk"], keys["inf"])
    small = []
    for m in [int(x) for x in a.small.split(",")]:
        idx = np.random.default_rng(m).integers(0, K, m).astype(np.uint32)
        sigs = eng.sign_many(keys["sk"][idx], keys["pk"][idx], keys["inf"][idx], blob[:8 * m], off[:m + 1], nonce[:m])
        t_sig, t_idx = torch.from_numpy(sigs).to(dev), torch.from_numpy(idx.view(np.int32)).to(dev)
        t_pk, t_inf = torch.from_numpy(keys["pk"][idx]).to(dev), torch.from_numpy(keys["inf"][idx]).to(dev)
        o1 = torch.empty(m, dtype=torch.uint8, device=dev)
        o2 = torch.empty(m, dtype=torch.uint8, device=dev)
        vm = lambda: eng.verify_many_dev(m, t_sig, t_pk, t_inf, t_blob, t_off, o1)          # noqa: E731
        rg = lambda: eng.verify_registered_many_dev(ks, m, t_sig, t_idx, t_blob, t_off, o2)  # noqa: E731
        vm(); rg()
        torch.cuda.synchronize(dev)
        a1, a2 = [], []
        for _ in range(10):
            a1.append(timed(torch, vm, 1))
            a2.append(timed(torch, rg, 1))
        assert torch.equal(o1, o2) and int(o1.sum()) == 0
        small.append({"n": m, "verify_many_dev_ms": float(np.median(a1)), "registered_dev_ms": float(np.median(a2))})
    res["small_calls"] = small
    res["card_after"] = card(0)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
