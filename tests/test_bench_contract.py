"""bench.py contract: the reference arm prints exactly ONE JSON line with the required keys (CPU); --dump-outputs
writes the verdicts of the timed paths (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-seconds", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "schnorr_verifications_per_sec" and d["unit"] == "verifications/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_canonical_work_units_match_the_survey():
    """SURVEY.md 8(d): 787 338 / 843 618 wide multiplies per verification at 8 / 80-byte messages."""
    import importlib.util
    sp = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(sp)
    sp.loader.exec_module(b)
    assert b.w_per_verify(8) == 787338 and b.w_per_verify(80) == 843618 and b.w_per_verify(160) == 871758
    assert [b.permutations_for(L) for L in (0, 8, 21, 22, 80, 160)] == [2, 2, 2, 3, 4, 5]


def test_non_zero_rank_of_the_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _bench_module():
    import importlib.util
    sp = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(sp)
    sp.loader.exec_module(b)
    return b


def test_dump_outputs_writes_float32_and_samples_large_outputs(tmp_path):
    import numpy as np
    b = _bench_module()
    v = np.arange(100, dtype=np.uint8) % 4
    b.dump_outputs(str(tmp_path / "small"), {"verdicts": v, "e2e_verdicts": v})
    assert sorted(os.listdir(tmp_path / "small")) == ["e2e_verdicts.npy", "verdicts.npy"]
    for name in ("verdicts", "e2e_verdicts"):
        a = np.load(tmp_path / "small" / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, v)
    # ranks whose outputs exceed their share: a fixed sample of rows, recomputable from (n, cap) alone
    n = b.DUMP_MAX_ROWS // 2 + 5
    v = (np.arange(n) % 4).astype(np.uint8)
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), {"verdicts": v}, rank=1, world=2)
    a = np.load(tmp_path / "a" / "verdicts_rank1.npy")
    assert a.dtype == np.float32 and len(a) == b.DUMP_MAX_ROWS // 2
    assert np.array_equal(a, v[b.dump_rows(n, len(a))])
    assert np.array_equal(a, np.load(tmp_path / "b" / "verdicts_rank1.npy"))


def test_dump_of_all_ranks_stays_within_64_mb(tmp_path):
    """The budget holds for the whole job, not per process: 2^20 and 2^22 signatures per GPU on 1, 2 and 8 ranks."""
    import numpy as np
    b = _bench_module()
    for log2n, world in ((20, 1), (20, 8), (22, 2), (22, 8)):
        d = tmp_path / ("%d_%d" % (log2n, world))
        v = np.zeros(1 << log2n, dtype=np.uint8)
        for rank in range(world):
            b.dump_outputs(str(d), {"verdicts": v, "e2e_verdicts": v}, rank, world)
        files = os.listdir(d)
        assert len(files) == 2 * world
        assert sum(os.path.getsize(d / f) for f in files) <= 64 * 10**6, (log2n, world)


def test_bench_refuses_meaningless_arguments():
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and out.stdout == "", args


def _run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--log2n", "12", "--no-extras",
                          "--cpu-seconds", "0.5"] + list(args), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    return json.loads(out.stdout)


@pytest.mark.gpu
def test_dump_outputs_holds_the_verdicts_of_the_timed_paths(tmp_path):
    import numpy as np
    import schnorr_sig_b200 as s
    n = 1 << 12
    one = _run_bench("--steps", "1", "--warmup", "1")
    d = _run_bench("--steps", "3", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 3 and d["warmup"] == 0
    # the launches inside the timed region follow --steps (and not --warmup)
    assert one["gpu_launches"] > 0 and d["gpu_launches"] == 3 * one["gpu_launches"]
    w = s.synth.inject_faults(dict(s.synth.host_inputs(s.synth.DEFAULT_SEED, n, 8), sigs=np.zeros((n, 81), np.uint8),
                                   pk=np.zeros((n, 96), np.uint8)), every=1024)
    assert sorted(os.listdir(tmp_path)) == ["e2e_verdicts.npy", "verdicts.npy"]
    for name in ("verdicts", "e2e_verdicts"):
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, w["expect"]), name
