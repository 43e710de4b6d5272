#!/usr/bin/env python3
"""bench.py -- Schnorr verifications/sec on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2n 20] [--msg-len 8]
                    [--dump-outputs DIR]

Workload (config.workload): independent Signature::verify of 2^20 synthetic signatures per GPU,
8-byte messages (BASELINE.json configs[2]; the metric's own configuration).  A step = one pass of the
hot path over the whole batch.  Signatures/keys are produced by the engine's device signer from a
seeded generator (synthetic), one invalid signature per 1024 injected (SURVEY.md §8d).

 value      whole-job verifications/s with the inputs resident in HBM (device-timed, CUDA events,
            max over ranks)
 e2e        same metric through the public host API (pinned host buffers, H2D + kernels + D2H inside
            the timed region)
 roofline   integer-multiply pipe ("imad"): canonical wide multiplies per verification (SURVEY.md §8d
            cost model v1: 787 338) x verifications per launch / k_verify_fast device time, against the
            peak measured live by the engine's own IMAD.WIDE calibration kernel (K6) -- HBM and tensor
            cores are not the bound of this path; the HBM fraction is reported alongside.
 cpu_baseline / --impl reference
            the reference's Rust crate cannot be built here (no cargo, un-vendored deps): the timed
            CPU path is the C restatement oracle/cref.c ("port") on all host threads, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

import cost_model  # noqa: E402  (single source of the unit counts, SURVEY.md 8(d))
from cost_model import permutations_for, w_per_hash, w_per_verify  # noqa: E402

METRIC = "schnorr_verifications_per_sec"
UNIT = "verifications/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=20, help="signatures per GPU = 2^log2n")
    ap.add_argument("--msg-len", type=int, default=8)
    ap.add_argument("--no-extras", action="store_true", help="skip the hash / batch side measurements")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 2^log2n signatures per GPU (default); strong: 2^log2n signatures in total, split over the GPUs")
    ap.add_argument("--batch-log2n", type=int, default=None,
                    help="signatures per GPU of the batch side measurement (default 16 at 1 GPU = configs[3], "
                         "21 at N > 1 = configs[4]: 2^24 over 8 GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the verdicts of the last timed step of both timed paths to DIR/<name>.npy (float32; "
                         "a fixed sample of rows above 2^22 signatures over all GPUs), so that two builds can be "
                         "compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours (the CPU arm sizes its inputs from the measured host rate)")
    return args


DUMP_MAX_ROWS = 1 << 22      # over all ranks: two float32 outputs per row -> at most 32 MiB (+ file headers) in all


def dump_rows(n, k):
    """The fixed sample of k of n rows that the dump keeps when a rank's output is longer than its share: sorted,
    drawn from seed 0, a function of (n, k) alone (so a reader can recompute which signatures the files hold)."""
    return np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def dump_outputs(path, outputs, rank=0, world=1):
    """Writes each output of this rank (one row per signature) as float32 to path/<name>.npy, or path/<name>_rank<r>.npy
    when world > 1.  Each rank keeps at most DUMP_MAX_ROWS // world rows, the rows dump_rows(n, cap) when it has more,
    so the dump of all ranks together stays under DUMP_MAX_ROWS rows whatever the size and the number of GPUs."""
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(outputs.values())))
    cap = DUMP_MAX_ROWS // world
    rows = dump_rows(n, cap) if n > cap else slice(None)
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, a in outputs.items():
        np.save(os.path.join(path, name + suffix + ".npy"), np.asarray(a)[rows].astype(np.float32))


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_rate(n_target_seconds, msg_len, seed):
    """Times the CPU restatement (oracle/cref.c) on all host threads over a bounded sample."""
    import cref
    cores = cref.default_threads()
    pilot = cref.workload(seed, 16 * cores, msg_len, cores)
    t0 = time.perf_counter()
    v = cref.verify_many_fast(pilot["sigs"], pilot["pk"], pilot["inf"], pilot["blob"], pilot["off"], cores)
    dt = time.perf_counter() - t0
    assert (v == 0).all()
    # the textbook oracle on the same pilot set: the two CPU restatements must agree, and its rate is reported beside
    t0 = time.perf_counter()
    v2 = cref.verify_many(pilot["sigs"], pilot["pk"], pilot["inf"], pilot["blob"], pilot["off"], cores)
    textbook_rate = len(v2) / (time.perf_counter() - t0)
    assert np.array_equal(v, v2)
    rate = len(v) / dt
    n = int(max(16 * cores, min(rate * n_target_seconds, 1 << 17)))
    reps = -(-n // len(v))
    sigs = np.tile(pilot["sigs"], (reps, 1))[:n]
    pk = np.tile(pilot["pk"], (reps, 1))[:n]
    inf = np.tile(pilot["inf"], reps)[:n]
    blob = np.tile(pilot["blob"], reps)[:n * msg_len]
    off = (np.arange(n + 1, dtype=np.uint64) * np.uint64(msg_len))
    return dict(cores=cores, n=n, sigs=sigs, pk=pk, inf=inf, blob=blob, off=off, textbook_rate=textbook_rate)


CPU_PORT_NOTE = ("oracle/cfast.c: optimised C restatement of the reference's CPU path (width-5 NAF subgroup check, "
                 "Straus-Shamir double-base product with a base-point table as src/signature.rs:194-198 describes, one "
                 "reduction per Fp6 coefficient); the Rust crate itself cannot be built here (no cargo, un-vendored git "
                 "dependencies); the textbook oracle oracle/cref.c runs at `textbook_value`")


def run_reference(args):
    """--impl reference: the CPU path on the host cores.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import cref
    per_step = max(1.0, args.cpu_seconds / max(1, args.steps + args.warmup) * 2)
    s = cpu_reference_rate(per_step, args.msg_len, 1234)
    for _ in range(args.warmup):
        cref.verify_many_fast(s["sigs"][:256], s["pk"][:256], s["inf"][:256], s["blob"][:256 * args.msg_len], s["off"][:257], s["cores"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v = cref.verify_many_fast(s["sigs"], s["pk"], s["inf"], s["blob"], s["off"], s["cores"])
    dt = time.perf_counter() - t0
    assert (v == 0).all()
    value = args.steps * s["n"] / dt
    sample = "%d signatures per step (distinct base set of %d tiled), %d-byte messages, %d threads" % (
        s["n"], 16 * s["cores"], args.msg_len, s["cores"])
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (Goldilocks Fp / Fp6, exact)",
            "data": "synthetic",
            "config": {"workload": "independent Signature::verify, %d-byte messages; CPU restatement of the reference "
                                   "(oracle/cfast.c: the Rust crate needs cargo + un-vendored git deps, absent here)" % args.msg_len,
                       "signatures_per_step": s["n"]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": s["cores"], "kind": "port", "sample": sample,
                             "note": CPU_PORT_NOTE, "textbook_value": s["textbook_rate"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def protect_stdout():
    """Libraries (NCCL prints its version banner) must not pollute stdout: fd 1 is pointed at stderr and
    the JSON line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    args = parse_args()
    protect_stdout()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import schnorr_sig_b200 as sb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    eng = sb.Engine(local)
    stream = torch.cuda.Stream(device=dev)
    eng.set_stream(stream.cuda_stream)
    n = (1 << args.log2n) if args.scaling == "weak" else max(128, (1 << args.log2n) // world)
    L = args.msg_len
    seed = sb.synth.DEFAULT_SEED

    # ---- synthetic inputs: host RNG -> device signer (this rank's shard) ---------------------
    hin = sb.synth.host_inputs(seed, n, L, shard=rank)
    with torch.cuda.stream(stream):
        d_sk = torch.from_numpy(hin["sk"]).to(dev)
        d_nonce = torch.from_numpy(hin["nonce"]).to(dev)
        d_blob = torch.from_numpy(hin["blob"]).to(dev) if hin["blob"].size else torch.zeros(16, dtype=torch.uint8, device=dev)
        d_off = torch.from_numpy(hin["off"].view(np.int64)).to(dev)
        d_pk = torch.empty((n, 96), dtype=torch.uint8, device=dev)
        d_inf = torch.zeros(n, dtype=torch.uint8, device=dev)
        d_sigs = torch.empty((n, 81), dtype=torch.uint8, device=dev)
        eng.keygen_dev(n, d_sk, d_pk, d_inf)
        eng.sign_many_dev(n, d_sk, d_pk, d_inf, d_blob, d_off, d_nonce, d_sigs)
        stream.synchronize()
        # invalid-signature injection on the host copy (1 in 1024), pushed back
        w = dict(hin, sigs=d_sigs.cpu().numpy(), pk=d_pk.cpu().numpy(), inf=d_inf.cpu().numpy())
        w = sb.synth.inject_faults(w, every=1024)
        d_sigs.copy_(torch.from_numpy(w["sigs"]))
        d_pk.copy_(torch.from_numpy(w["pk"]))
        d_blob[:w["blob"].size].copy_(torch.from_numpy(w["blob"]))
        d_verdicts = torch.full((n,), 255, dtype=torch.uint8, device=dev)
        stream.synchronize()
    expect = w["expect"]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- HBM-resident timing: `value` --------------------------------------------------------
    def step_dev():
        eng.verify_many_dev(n, d_sigs, d_pk, d_inf, d_blob, d_off, d_verdicts)

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_dev()
        stream.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    launches0 = eng.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    kernel_ms = []
    with torch.cuda.stream(stream):
        ev[0].record(stream)
        for k in range(args.steps):
            step_dev()
            ev[k + 1].record(stream)
            kernel_ms.append(eng.last_kernel_ms())   # waits for this step's k_verify (events on the same stream)
        stream.synchronize()
    barrier()
    launches = eng.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    got = d_verdicts.cpu().numpy()          # the verdicts of the last timed step
    if not np.array_equal(got, expect):
        raise SystemExit("rank %d: verdicts differ from the expected pattern (%d mismatches)" % (rank, int((got != expect).sum())))
    dev_ms = ev[0].elapsed_time(ev[-1])
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * n * args.steps / (total_ms * 1e-3)

    # ---- end to end through the host API: `e2e` -----------------------------------------------
    h_sigs = torch.from_numpy(w["sigs"]).pin_memory()
    h_pk = torch.from_numpy(w["pk"]).pin_memory()
    h_inf = torch.from_numpy(w["inf"]).pin_memory()
    h_blob = torch.from_numpy(w["blob"] if w["blob"].size else np.zeros(16, np.uint8)).pin_memory()
    h_off = torch.from_numpy(hin["off"].view(np.int64)).pin_memory()
    h_out = torch.full((n,), 255, dtype=torch.uint8).pin_memory()
    h2d = n * 81 + n * 96 + n + int(hin["off"][-1]) + (n + 1) * 8
    d2h = n

    def step_e2e():
        eng.verify_many_raw(n, h_sigs, h_pk, h_inf, h_blob, h_off, h_out)   # copies in, kernels, copy out, sync

    step_e2e()
    if not np.array_equal(h_out.numpy(), expect):
        raise SystemExit("rank %d: e2e verdicts differ" % rank)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_e2e()
    e1.record(stream)
    stream.synchronize()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.steps / (float(t.item()) * 1e-3)
    e2e_got = h_out.numpy().copy()          # the verdicts of the last timed step
    if not np.array_equal(e2e_got, expect):
        raise SystemExit("rank %d: e2e verdicts differ" % rank)
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, {"verdicts": got, "e2e_verdicts": e2e_got}, rank, world)

    # ---- roofline of the dominant kernel (k_verify_fast; the exact pass over handed-back items is inside kernel_ms) ----
    peak_w, peak_ms = eng.imad_peak(1 << 15)
    k_ms = float(np.mean(kernel_ms))
    achieved_w = n * w_per_verify(L) / (k_ms * 1e-3)
    executed_w = n * cost_model.w_executed_fast(L) / (k_ms * 1e-3)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_achieved = n * cost_model.hbm_bytes_per_verify(L) / (k_ms * 1e-3) / 1e9
    nominal = cost_model.nominal_peak_w_per_s(148, (clocks or {}).get("sm_max_mhz") or 1965.0)
    # DRAM traffic / instruction counts of one launch come from the ncu capture committed under profiles/; they are only
    # quoted when the capture was taken from the sources this library is built from
    ncu = cost_model.ncu_constants() or {}
    ncu_k = (ncu.get("k_verify_fast") or {}).get(str(args.log2n)) if n == (1 << args.log2n) else None
    ncu_current = bool(ncu) and ncu.get("source_sha256") == cost_model.source_sha256()
    roofline = {"bound": "imad", "achieved": achieved_w / 1e12, "peak": peak_w / 1e12, "unit": "Tmul32x32/s",
                "frac": achieved_w / peak_w, "traffic": (ncu_k or {}).get("dram_bytes") if ncu_current else None,
                "traffic_source": (ncu.get("capture") if ncu_k else None),
                "traffic_capture_matches_sources": ncu_current if ncu_k else None,
                "frac_executed": executed_w / peak_w,
                "frac_vs_nominal": achieved_w / nominal, "frac_executed_vs_nominal": executed_w / nominal,
                "kernel": "k_verify_fast", "kernel_ms": k_ms, "kernel_share_of_step": k_ms * args.steps / dev_ms,
                "peak_source": "measured live: schnorr_b200_imad_peak (K6, IMAD.WIDE.U32 chains, full grid), %.2f ms" % peak_ms,
                "peak_nominal": nominal / 1e12,
                "algorithmic_units": "%d wide multiplies per verification (cost_model.py = SURVEY.md 8d model v1, %d-byte message) x %d per launch" % (w_per_verify(L), L, n),
                "executed_units": "%d wide multiplies per verification actually executed (host-build counter, cost_model.py)" % cost_model.w_executed_fast(L),
                "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}

    # ---- parity evidence gathered in this very run ----------------------------------------------------------------
    parity = {"verdicts_equal_expected_pattern": int(n), "ranks": world}
    if rank == 0:
        import cref
        rng = np.random.default_rng(5)
        bad_idx = np.nonzero(expect)[0][:1024]
        idx = np.unique(np.concatenate([rng.choice(n, min(n, 1024), replace=False), bad_idx]))
        sub_blob = w["blob"].reshape(n, L)[idx].reshape(-1) if L else np.zeros(0, np.uint8)
        sub_off = np.arange(len(idx) + 1, dtype=np.uint64) * np.uint64(L)
        want = cref.verify_many(w["sigs"][idx], w["pk"][idx], w["inf"][idx], sub_blob, sub_off, cref.default_threads())
        if not np.array_equal(want, got[idx]):
            raise SystemExit("verdicts differ from the oracle on the sampled indices")
        parity["verdicts_equal_oracle_on_sample"] = int(len(idx))
        parity["sample"] = "1024 random indices + every injected fault (up to 1024), oracle/cref.c"

    # ---- side measurements (not part of the timed region) --------------------------------------
    extras = {}
    if not args.no_extras:
        extras = side_measurements(args, eng, stream, dev, torch, n, d_sigs, d_pk, d_inf, d_blob, d_off, hin, rank, world, dist, parity)

    # ---- CPU baseline beside it (rank 0, N = 1) -------------------------------------------------
    cpu = None
    if rank == 0 and world == 1:
        import cref
        s = cpu_reference_rate(args.cpu_seconds, L, 1234)
        t0 = time.perf_counter()
        v = cref.verify_many_fast(s["sigs"], s["pk"], s["inf"], s["blob"], s["off"], s["cores"])
        dt = time.perf_counter() - t0
        assert (v == 0).all()
        cpu = {"value": s["n"] / dt, "unit": UNIT, "cores": s["cores"], "kind": "port",
               "sample": "%d signatures (base set of %d tiled), %d-byte messages, oracle/cfast.c on %d threads, %.1f s"
                         % (s["n"], 16 * s["cores"], L, s["cores"], dt),
               "note": CPU_PORT_NOTE, "textbook_value": s["textbook_rate"]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "u64 (Goldilocks Fp / Fp6 on 32-bit IMAD, exact)", "data": "synthetic",
                "config": {"workload": "independent Signature::verify of %s, %d-byte messages, "
                                       "1/1024 invalid injected (BASELINE configs[2])" % (
                                           ("2^%d signatures per GPU" % args.log2n) if args.scaling == "weak"
                                           else ("2^%d signatures in total (%d per GPU)" % (args.log2n, n)), L),
                           "signatures_per_gpu": n, "msg_len": L, "parallelism": "shard%d (no data-path collective)" % world,
                           "l2_policy": "inputs (%.0f MB per GPU) larger than L2; no flush" % (n * (177 + L + 8) / 1e6)},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
                "parity_checked": parity}
        line.update(extras)
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


def side_measurements(args, eng, stream, dev, torch, n, d_sigs, d_pk, d_inf, d_blob, d_off, hin, rank, world, dist, parity):
    """hash_message throughput (configs[1]), batch verification (configs[3]/[4]), strong scaling of configs[2], the
    one-process multi-GPU arm of the C ABI and the small-call latencies; device-timed, outside the headline region."""
    import schnorr_sig_b200 as sb
    out = {}
    L = args.msg_len

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # K1: hash sweep point at n messages
    d_rx = d_sigs[:, :48].contiguous()
    d_dig = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    with torch.cuda.stream(stream):
        eng.hash_messages_dev(n, d_rx, d_pk, d_blob, d_off, d_dig)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng.hash_messages_dev(n, d_rx, d_pk, d_blob, d_off, d_dig)
        b.record(stream)
        stream.synchronize()
    hms = a.elapsed_time(b)
    peak_w, _ = eng.imad_peak(1 << 15)
    out["hash"] = {"metric": "rescue_hash_message_per_sec", "value": world * n / (hms * 1e-3), "n_per_gpu": n, "msg_len": L,
                   "ms": hms, "roofline_frac_imad": (n * w_per_hash(L) / (hms * 1e-3)) / peak_w}

    # K3/K4: one batch of nb signatures per GPU, partial MSM per rank + one small gather + finish on rank 0
    blog = args.batch_log2n if args.batch_log2n is not None else (16 if world == 1 else 21)
    nb = 1 << blog
    bin_ = hin if nb <= n else sb.synth.host_inputs(sb.synth.DEFAULT_SEED + 1, nb, L, shard=rank)

    def device_batch(inputs, count):
        """device-resident keys / signatures / randomisers for `count` signatures of `inputs`"""
        with torch.cuda.stream(stream):
            d_sk = torch.from_numpy(inputs["sk"][:count]).to(dev)
            d_nonce = torch.from_numpy(inputs["nonce"][:count]).to(dev)
            gb = torch.from_numpy(inputs["blob"][:count * L]).to(dev) if L else torch.zeros(16, dtype=torch.uint8, device=dev)
            goff = torch.from_numpy(inputs["off"][:count + 1].view(np.int64)).to(dev)
            gpk = torch.empty((count, 96), dtype=torch.uint8, device=dev)
            ginf = torch.zeros(count, dtype=torch.uint8, device=dev)
            gsig = torch.empty((count, 81), dtype=torch.uint8, device=dev)
            eng.keygen_dev(count, d_sk, gpk, ginf)
            eng.sign_many_dev(count, d_sk, gpk, ginf, gb, goff, d_nonce, gsig)
            d_rand = torch.from_numpy(inputs["rand"][:count]).to(dev)
            stream.synchronize()
        return gsig, gpk, ginf, gb, goff, d_rand

    part = torch.zeros(192, dtype=torch.uint8, device=dev)
    res = torch.zeros(216, dtype=torch.uint8, device=dev)
    allp = torch.zeros((world, 192), dtype=torch.uint8, device=dev)

    def batch_once(bufs, count):
        """this rank's partial -> ONE all_gather of 192 bytes per rank, enqueued on the engine's stream right behind the
        partial kernels (no host synchronisation around it) -> finish on rank 0"""
        gsig, gpk, ginf, gb, goff, d_rand = bufs
        if dist is None:   # one GPU: the whole batch as one enqueue ((sum s e) G runs beside the MSM)
            eng.verify_batch_dev(count, gsig, gpk, ginf, gb, goff, d_rand, res)
            return
        with torch.cuda.stream(stream):
            eng.batch_partial_dev(count, gsig, gpk, ginf, gb, goff, d_rand, part)
            if dist is not None:
                dist.all_gather_into_tensor(allp, part)
                gathered = allp
            else:
                gathered = part.view(1, 192)
            if rank == 0:
                eng.batch_finish_dev(world, gathered, res)

    bufs = device_batch(bin_, nb)
    batch_once(bufs, nb)
    stream.synchronize()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    batch_once(bufs, nb)
    b.record(stream)
    stream.synchronize()
    bms = max_over_ranks(a.elapsed_time(b))
    plan = eng.last_batch_plan()
    verdict = int(res[0].item()) if rank == 0 else None
    # invalid-signature injection (SURVEY.md 8d C4/C5): one corrupted signature on the LAST rank must fail the lot
    if rank == world - 1:
        bufs[0][nb // 2, 49] ^= 1
    batch_once(bufs, nb)
    stream.synchronize()
    torch.cuda.synchronize(dev)
    verdict_bad = int(res[0].item()) if rank == 0 else None
    w_sig = cost_model.w_per_batch_signature(nb, L, plan[:3])
    out["batch"] = {"metric": "schnorr_batch_verified_signatures_per_sec", "value": world * nb / (bms * 1e-3),
                    "signatures_per_gpu": nb, "ms": bms, "verdict": verdict,
                    "verdict_with_one_corrupted_signature_on_last_rank": verdict_bad,
                    "plan": {"window_bits": plan[0], "windows": plan[1], "buckets_per_window": plan[2], "segment_len": plan[3]},
                    "canonical_w_per_signature": w_sig,
                    "roofline_frac_imad": (nb * w_sig / (bms * 1e-3)) / peak_w,
                    "exchange": "one all_gather of 192 B per rank on the compute stream" if world > 1 else "none (1 GPU)"}
    if rank == 0 and (verdict != 0 or verdict_bad != 2):
        raise SystemExit("batch verification returned verdicts %r / %r (expected 0 / 2)" % (verdict, verdict_bad))

    # sharded batch against the oracle (configs[4] in miniature): 4096 signatures cut over the ranks; rank 0's finished
    # points must equal a single-GPU run over the concatenated shards and oracle/cref.c; an invalid signature on the last
    # rank must turn the verdict into Err
    ns = 4096
    small = sb.synth.host_inputs(sb.synth.DEFAULT_SEED + 99, ns, L, shard=0)     # the same inputs on every rank
    lo, hi = (ns * rank) // world, (ns * (rank + 1)) // world
    sl = {k: small[k][lo:hi] for k in ("sk", "nonce", "rand")}
    sl["blob"] = small["blob"][lo * L:hi * L]
    sl["off"] = small["off"][lo:hi + 1] - small["off"][lo]
    sbufs = device_batch(sl, hi - lo)
    batch_once(sbufs, hi - lo)
    stream.synchronize()
    torch.cuda.synchronize(dev)
    if rank == 0:
        import cref
        got = res.cpu().numpy().copy()
        pk_s, inf_s = eng.keygen(small["sk"])
        sig_s = eng.sign_many(small["sk"], pk_s, inf_s, small["blob"], small["off"], small["nonce"])
        v1, l1, r1 = eng.verify_batch(sig_s, pk_s, inf_s, small["blob"], small["off"], small["rand"])
        cv, cl, cr = cref.verify_batch(sig_s, pk_s, inf_s, small["blob"], small["off"], small["rand"], cref.default_threads())
        same = (got[0] == v1 == cv == 0 and np.array_equal(got[8:105], l1) and np.array_equal(got[8:105], cl)
                and np.array_equal(got[112:209], r1) and np.array_equal(got[112:209], cr))
        if not same:
            raise SystemExit("sharded batch over %d ranks differs from the single-GPU run / the oracle" % world)
    if rank == world - 1:
        sbufs[0][(hi - lo) // 2, 49] ^= 1
    batch_once(sbufs, hi - lo)
    stream.synchronize()
    torch.cuda.synchronize(dev)
    if rank == 0:
        if int(res[0].item()) != 2:
            raise SystemExit("sharded batch with an injected invalid signature returned %d" % int(res[0].item()))
        parity["sharded_batch_points_equal_single_gpu_and_oracle"] = {"signatures": ns, "ranks": world, "injected_invalid_verdict": 2}

    # strong scaling of configs[2]: the SAME 2^log2n signatures in total, cut over the ranks (131 072 per GPU at N = 8:
    # 3.46 kernel waves)
    if args.scaling == "weak" and world > 1:
        m = max(128, n // world)
        with torch.cuda.stream(stream):
            v_s = torch.full((m,), 255, dtype=torch.uint8, device=dev)
            eng.verify_many_dev(m, d_sigs, d_pk, d_inf, d_blob, d_off, v_s)
            stream.synchronize()
        if dist is not None:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(args.steps):
            eng.verify_many_dev(m, d_sigs, d_pk, d_inf, d_blob, d_off, v_s)
        b.record(stream)
        stream.synchronize()
        sms = max_over_ranks(a.elapsed_time(b)) / args.steps
        out["strong_scaling"] = {"metric": METRIC, "value": world * m / (sms * 1e-3), "signatures_total": world * m,
                                 "signatures_per_gpu": m, "ms_per_step": sms, "n_gpus": world}

    # one process driving every GPU through the C ABI (schnorr_b200_create_multi): host buffers in, verdicts out.
    # Rank 0 only; the other ranks wait on a HOST-side (gloo) barrier -- an NCCL barrier would keep a spinning kernel on
    # their GPUs, which rank 0's kernels would have to time-slice with.
    cpu_group = None
    if dist is not None:
        torch.cuda.synchronize(dev)
        cpu_group = dist.new_group(backend="gloo")
        dist.barrier(group=cpu_group)
    if rank == 0 and torch.cuda.device_count() >= world:
        me = sb.Engine(list(range(world)))
        try:
            w_sigs, w_pk, w_inf = d_sigs.cpu().numpy(), d_pk.cpu().numpy(), d_inf.cpu().numpy()
            w_blob = d_blob.cpu().numpy()[:n * L]
            reps = world
            hs = torch.from_numpy(np.tile(w_sigs, (reps, 1))).pin_memory()
            hp = torch.from_numpy(np.tile(w_pk, (reps, 1))).pin_memory()
            hi_ = torch.from_numpy(np.tile(w_inf, reps)).pin_memory()
            hb = torch.from_numpy(np.tile(w_blob, reps) if L else np.zeros(16, np.uint8)).pin_memory()
            ho = torch.from_numpy((np.arange(reps * n + 1, dtype=np.uint64) * np.uint64(L)).view(np.int64)).pin_memory()
            hv = torch.full((reps * n,), 255, dtype=torch.uint8).pin_memory()
            me.verify_many_raw(reps * n, hs, hp, hi_, hb, ho, hv)
            ref = hv.numpy()[:n].copy()
            ok = all(np.array_equal(hv.numpy()[k * n:(k + 1) * n], ref) for k in range(reps))
            t0 = time.perf_counter()
            for _ in range(args.steps):
                me.verify_many_raw(reps * n, hs, hp, hi_, hb, ho, hv)
            dt = (time.perf_counter() - t0) / args.steps
            out["e2e_one_process"] = {"value": reps * n / dt, "unit": UNIT, "devices": world, "ms_per_step": dt * 1e3,
                                      "signatures_per_step": reps * n, "verdicts_consistent_across_devices": bool(ok),
                                      "api": "schnorr_b200_create_multi + schnorr_b200_verify_many (pinned host buffers, "
                                             "one host thread per device, copies inside the call, wall clock)"}
        finally:
            me.close()
    if dist is not None:
        dist.barrier(group=cpu_group)

    # small calls through the host API (the reference's own Criterion case is ONE verify, benches/schnorr.rs:60-77):
    # host buffers in, verdicts out, wall clock around the call; rank 0 only
    if rank == 0:
        small_calls = {}
        for ns_ in (1, 1024):
            hs = {k: hin[k] for k in ("sk", "nonce", "blob", "off")}
            pk_s, inf_s = eng.keygen(hs["sk"][:ns_])
            off_s = hs["off"][:ns_ + 1].copy()
            blob_s = hs["blob"][:int(off_s[-1])] if int(off_s[-1]) else np.zeros(0, np.uint8)
            sig_s = eng.sign_many(hs["sk"][:ns_], pk_s, inf_s, blob_s, off_s, hs["nonce"][:ns_])
            v = eng.verify_many(sig_s, pk_s, inf_s, blob_s, off_s)
            if int(v.max()) != 0:
                raise SystemExit("small-call verification failed")
            ts = []
            for _ in range(20):
                t0 = time.perf_counter()
                eng.verify_many(sig_s, pk_s, inf_s, blob_s, off_s)
                ts.append(time.perf_counter() - t0)
            small_calls["n%d_ms" % ns_] = float(np.mean(ts)) * 1e3
        small_calls["kernel"] = "n1: k_verify_one (one thread block per signature); n1024: k_verify_dist (one signature per six lanes)"
        out["small_calls"] = small_calls
        out["criterion_protocol"] = criterion_protocol(eng, sb)
        out["hash_sweep"] = hash_sweep(eng, torch, dev, stream, peak_w)
    return out


def criterion_protocol(eng, sb):
    """The reference's own Criterion cases (benches/schnorr.rs:22-24,67-96) through the host API, wall clock, mean of
    20 samples (sample_size(20), benches/schnorr.rs:113): one Signature::verify for 8 / 80 / 160-byte messages and
    verify_batch of 4 / 16 / 32 / 64 / 128 signatures over one shared 80-byte message."""
    res = {"samples": 20, "verify_ms": {}, "verify_batch_ms": {}}
    for L in (8, 80, 160):
        w = sb.synth.signed_workload(eng, 0xC21 + L, 1, msg_len=L)
        assert int(eng.verify_many(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"])[0]) == 0
        ts = []
        for _ in range(20):
            t0 = time.perf_counter()
            eng.verify_many(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"])
            ts.append(time.perf_counter() - t0)
        res["verify_ms"]["%d_bytes" % L] = float(np.mean(ts)) * 1e3
    for size in (4, 16, 32, 64, 128):
        w = sb.synth.host_inputs(0xBA7 + size, size, 80)
        w["blob"] = np.tile(w["blob"][:80], size)                 # one shared message (benches/schnorr.rs:81)
        pk, inf = eng.keygen(w["sk"])
        sigs = eng.sign_many(w["sk"], pk, inf, w["blob"], w["off"], w["nonce"])
        assert eng.verify_batch(sigs, pk, inf, w["blob"], w["off"], w["rand"])[0] == 0
        ts = []
        for _ in range(20):
            t0 = time.perf_counter()
            eng.verify_batch(sigs, pk, inf, w["blob"], w["off"], w["rand"])
            ts.append(time.perf_counter() - t0)
        res["verify_batch_ms"]["%d_signatures" % size] = float(np.mean(ts)) * 1e3
    return res


def hash_sweep(eng, torch, dev, stream, peak_w):
    """BASELINE configs[1]: hash_message throughput for 2^10 ... 2^22 messages of 8 bytes on one GPU (device-resident
    uniform field elements, CUDA events, second of two launches)."""
    rng = np.random.default_rng(11)
    nmax = 1 << 22
    P = np.uint64(0xFFFFFFFF00000001)
    def felts(k):
        v = rng.integers(0, 2**64, k, dtype=np.uint64)
        return np.where(v >= P, v - P, v).view(np.uint8)
    with torch.cuda.stream(stream):
        d_rx = torch.from_numpy(felts(6 * nmax).reshape(nmax, 48)).to(dev)
        d_pk = torch.from_numpy(felts(12 * nmax).reshape(nmax, 96)).to(dev)
        d_blob = torch.from_numpy(rng.integers(0, 256, nmax * 8, dtype=np.uint8)).to(dev)
        d_off = torch.from_numpy((np.arange(nmax + 1, dtype=np.uint64) * np.uint64(8)).view(np.int64)).to(dev)
        d_out = torch.empty((nmax, 32), dtype=torch.uint8, device=dev)
        stream.synchronize()
    rows = []
    for lg in range(10, 23, 2):
        n = 1 << lg
        with torch.cuda.stream(stream):
            eng.hash_messages_dev(n, d_rx, d_pk, d_blob, d_off, d_out)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            eng.hash_messages_dev(n, d_rx, d_pk, d_blob, d_off, d_out)
            b.record(stream)
            stream.synchronize()
        ms = a.elapsed_time(b)
        rows.append({"log2_messages": lg, "ms": ms, "hashes_per_s": n / (ms * 1e-3),
                     "roofline_frac_imad": n * w_per_hash(8) / (ms * 1e-3) / peak_w})
    return {"msg_len": 8, "points": rows}


if __name__ == "__main__":
    main()
