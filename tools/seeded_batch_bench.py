"""Batch randomisers made on the device from a 32-byte seed against randomisers made on the host, on one GPU:
  generator    device time of k_batch_randomizers (batch_randomizers_dev, CUDA events, warmed up, median of --reps
               with min / max) at each --gen-sizes
  facade       wall time of the Python facade's verify_batch(signatures, public_keys, messages) at --facade-size, with
               rng (OsRng: one os.urandom call and one Python big-integer reduction per signature) and with seed=
  host_forms   wall time at --size of the host entry points verify_batch and verify_batch_registered (64 keys), three
               ways alternated in one process (median of --reps with min / max):
                 pregenerated  rand32 made before the timed call (what the engine costs with the randomisers given)
                 host_rand     rand32 made inside the timed call by a vectorised host method: os.urandom(32 n) with the
                               top two bits of every randomiser cleared (uniform below 2^254 < q, as the C++ facade does)
                 seeded        the _seeded entry point with one os.urandom(32)
The verdicts are checked (an all-valid batch: 0 everywhere), and the seeded forms' lhs / rhs are checked against the
rand32 forms fed with batch_randomizers(seed).  Prints one JSON line (card name, power limit and SM clocks read in the
same run).

    python tools/seeded_batch_bench.py [--size-log2 20] [--gen-sizes 16,20,21] [--facade-size-log2 16]
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

from registered_batch_bench import card, timed   # noqa: E402


def stats(ts):
    return {"median_ms": float(np.median(ts)), "min_ms": float(min(ts)), "max_ms": float(max(ts))}


def host_rand(n):
    r = np.frombuffer(os.urandom(32 * n), dtype=np.uint8).reshape(n, 32).copy()
    r[:, 31] &= 0x3F
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size-log2", type=int, default=20)
    ap.add_argument("--gen-sizes", default="16,20,21", help="log2 of the generator sizes")
    ap.add_argument("--facade-size-log2", type=int, default=16)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--facade-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import schnorr_sig_b200 as s
    if not torch.cuda.is_available():
        raise SystemExit("seeded_batch_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    eng = s.Engine(0)
    stream = torch.cuda.Stream(dev)          # the engine enqueues on this stream: the events below bracket its work
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    res = {"tool": "seeded_batch_bench", "card": card(0), "torch_device": torch.cuda.get_device_name(0), "msg_len": 8,
           "reps": a.reps}

    # 1. the generator alone
    seed = np.frombuffer(os.urandom(32), dtype=np.uint8).copy()
    t_seed = torch.from_numpy(seed).to(dev)
    gen = []
    for lg in [int(x) for x in a.gen_sizes.split(",")]:
        n = 1 << lg
        out = torch.empty((n, 32), dtype=torch.uint8, device=dev)
        fn = lambda: eng.batch_randomizers_dev(n, t_seed, 0, out)   # noqa: E731
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        ms = [timed(torch, fn) for _ in range(a.reps)]
        assert np.array_equal(out[:4].cpu().numpy(), eng.batch_randomizers(4, seed.tobytes()))
        gen.append({"n": n, **stats(ms), "bytes_written": 32 * n})
        print(json.dumps(gen[-1]), file=sys.stderr)
        del out
    res["generator"] = gen

    # 2. the Python facade: rng against seed
    nf = 1 << a.facade_size_log2
    w = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED, nf)
    sigs = [s.Signature(bytes(w["sigs"][i, :49]), bytes(w["sigs"][i, 49:])) for i in range(nf)]
    keys = [s.PublicKey(bytes(w["pk"][i]), bool(w["inf"][i])) for i in range(nf)]
    msgs = [bytes(w["blob"][int(w["off"][i]):int(w["off"][i + 1])]) for i in range(nf)]
    assert s.verify_batch(sigs, keys, msgs).is_ok() and s.verify_batch(sigs, keys, msgs, seed=os.urandom(32)).is_ok()
    fr, fs = [], []
    for _ in range(a.facade_reps):
        t0 = time.perf_counter()
        assert s.verify_batch(sigs, keys, msgs).is_ok()
        fr.append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        assert s.verify_batch(sigs, keys, msgs, seed=os.urandom(32)).is_ok()
        fs.append(1e3 * (time.perf_counter() - t0))
    res["facade"] = {"n": nf, "rng": stats(fr), "seed": stats(fs)}
    print(json.dumps(res["facade"]), file=sys.stderr)
    del sigs, keys, msgs

    # 3. the host entry points at --size-log2, three ways alternated
    n = 1 << a.size_log2
    w = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED + 1, n)
    K = 64
    kw = s.synth.signed_workload(eng, s.synth.DEFAULT_SEED + 2, K)
    ks, status = eng.register_keys(kw["pk"], kw["inf"])
    assert not status.any()
    idx = np.random.default_rng(5).integers(0, K, n).astype(np.uint32)
    rsigs = eng.sign_many(kw["sk"][idx], kw["pk"][idx], kw["inf"][idx], w["blob"], w["off"], w["nonce"])
    plain = (w["sigs"], w["pk"], w["inf"], w["blob"], w["off"])
    reg = (ks, rsigs, idx, w["blob"], w["off"])
    forms = {
        "verify_batch": (lambda r: eng.verify_batch(*plain, r), lambda sd: eng.verify_batch_seeded(*plain, sd)),
        "verify_batch_registered": (lambda r: eng.verify_batch_registered(*reg, r),
                                    lambda sd: eng.verify_batch_registered_seeded(*reg, sd)),
    }
    res["host_forms"] = []
    for name, (with_rand, seeded) in forms.items():
        sd = os.urandom(32)
        a1, a2 = seeded(sd), with_rand(eng.batch_randomizers(n, sd))
        assert a1[0] == a2[0] == 0 and bytes(a1[1]) == bytes(a2[1]) and bytes(a1[2]) == bytes(a2[2]), name
        pre = host_rand(n)
        for _ in range(2):                   # warm-up
            with_rand(pre)
            seeded(sd)
        ts = {"pregenerated": [], "host_rand": [], "seeded": []}
        for _ in range(a.reps):
            t0 = time.perf_counter()
            assert with_rand(pre)[0] == 0
            ts["pregenerated"].append(1e3 * (time.perf_counter() - t0))
            t0 = time.perf_counter()
            assert with_rand(host_rand(n))[0] == 0
            ts["host_rand"].append(1e3 * (time.perf_counter() - t0))
            t0 = time.perf_counter()
            assert seeded(os.urandom(32))[0] == 0
            ts["seeded"].append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        for _ in range(a.reps):
            host_rand(n)
        host_rand_ms = 1e3 * (time.perf_counter() - t0) / a.reps
        res["host_forms"].append({"form": name, "n": n, **{k: stats(v) for k, v in ts.items()},
                                  "host_rand_alone_ms": host_rand_ms, "outputs_equal": True})
        print(json.dumps(res["host_forms"][-1]), file=sys.stderr)
    ks.close()
    res["card_after"] = card(0)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
