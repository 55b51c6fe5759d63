"""CPU: the benchmark's reference arm (`bench.py --impl reference`) prints exactly one JSON line with the keys the driver reads.
(The GPU arm is exercised on the B200 box; its line carries the same keys plus roofline / clocks / gpu_launches.)"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-sessions", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                       # stdout carries the JSON line and nothing else
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "streams" and d["higher_is_better"] is True
    assert d["metric"] == "real-time G.711 TTS streams (RTF<=1)" and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 1 and d["dtype"] in ("bf16", "f32") and d["data"] == "synthetic"
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "streams", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_non_zero_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_steps_below_one_and_dumps_of_the_cpu_arm_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert p.returncode == 2 and p.stdout == "", (extra, p.stderr[-500:])


def test_dump_outputs_writes_float32_and_samples_rows_beyond_the_budget(tmp_path):
    import numpy as np
    import torch
    import bench
    small = torch.randint(0, 256, (16, 4096), dtype=torch.uint8)
    bench.dump_outputs(str(tmp_path / "a"), {"g711": small})
    a = np.load(tmp_path / "a" / "g711.npy")
    assert a.dtype == np.float32 and np.array_equal(a, small.numpy().astype(np.float32))
    big = torch.arange(8192, dtype=torch.float64)[:, None].expand(8192, 4096)       # 256 MB as float64: row i holds i
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"g711": big}, rank=1, world=2)
    b, c = np.load(tmp_path / "b" / "g711_rank1.npy"), np.load(tmp_path / "c" / "g711_rank1.npy")
    assert (tmp_path / "b" / "g711_rank1.npy").stat().st_size <= 32 << 20
    assert b.dtype == np.float32 and np.array_equal(b, c)                               # the same rows in every run
    rows = b[:, 0]
    assert len(rows) > 1000 and np.all(np.diff(rows) > 0) and np.array_equal(b, np.repeat(rows[:, None], 4096, axis=1))


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    import numpy as np
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--sessions", "8", "--dump-outputs", str(out),
                        "--no-cpu-baseline", "--no-latency", "--no-sessions", "--no-front", "--no-strong"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.strip()][-1])
    assert d["steps"] == 2 and d["per_gpu_stats"][0]["steps"] == 2
    g = np.load(out / "g711.npy")
    assert g.dtype == np.float32 and g.shape == (8, 32 * 128)
    assert np.all(g == np.round(g)) and g.min() >= 0 and g.max() <= 255 and len(np.unique(g)) > 16
