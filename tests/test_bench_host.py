"""Host-side pieces of bench.py that run without a GPU: the reference arm's JSON line (the CPU port of the
reference path) and the clock sampler's bookkeeping."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-batch", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "scenes/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_clock_sampler_reports_only_samples_of_the_timed_region():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler.__new__(bench.ClockSampler)

    class _Proc:
        def terminate(self): pass
        def wait(self, timeout=None): return 0
        def kill(self): pass

    now = time.perf_counter()
    s.proc, s.t0 = _Proc(), now - 0.05
    s.lines = [(now - 1.0, "1200, 1965, 200.0, Not Active, Not Active, Not Active, Not Active\n"),      # before the region
               (now - 0.04, "1965, 1965, 310.5, Not Active, Not Active, Not Active, Active\n"),
               (now - 0.02, "1950, 1965, 305.0, Not Active, Not Active, Not Active, Not Active\n"),
               (now - 0.01, "garbage line\n")]
    r = s.stop()
    assert r["samples_in_timed_region"] == 3 and r["samples"] == 2          # the garbage line does not parse
    assert r["sm_mhz"] == 1957.5 and r["sm_max_mhz"] == 1965.0 and r["power_w_max"] == 310.5
    assert r["reasons"] == ["sw_power_cap"]


def test_dump_outputs_writes_a_fixed_sample(tmp_path):
    """--dump-outputs: float32 (float64 for 64-bit types), shapes kept below the sample size, larger tensors as the same
    seeded sample on every call, and the size cap enforced before anything is written."""
    import numpy as np
    import pytest
    import torch
    sys.path.insert(0, ROOT)
    import bench
    big = torch.arange(bench.DUMP_SAMPLE * 3, dtype=torch.float32)
    tensors = {"loss": torch.tensor(0.5, dtype=torch.bfloat16), "counts": torch.tensor([3, 1 << 40]),
               "binary": torch.ones(2, 3, dtype=torch.uint8), "big": big}
    for d in ("a", "b"):
        bench.dump_outputs(tensors, str(tmp_path / d))
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in tensors}
    assert a["loss"].dtype == np.float32 and a["loss"].shape == () and float(a["loss"]) == 0.5
    assert a["counts"].dtype == np.float64 and a["counts"].tolist() == [3, 1 << 40]
    assert a["binary"].dtype == np.float32 and a["binary"].shape == (2, 3)
    s = a["big"]
    assert s.shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(s) >= 0) and s.max() > 2 * bench.DUMP_SAMPLE
    assert np.array_equal(s, np.load(tmp_path / "b" / "big.npy"))
    many = {f"t{i}": big for i in range(17)}                       # 17 x 4 MB samples > 64 MB
    with pytest.raises(SystemExit):
        bench.dump_outputs(many, str(tmp_path / "c"))
    assert not (tmp_path / "c").exists()


def test_step_outputs_of_the_roadmap_step():
    """What a training step hands its caller: loss, the state left behind, RoadMapBCE's metrics."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from driving_dirty_b200.synthetic import random_roadmap_model
    model = random_roadmap_model(16, 8, 16, 20, dtype="fp32", device="cpu", map_size=8)
    model.last_metrics = {"ts": torch.tensor(0.25), "binary": torch.zeros(1, 8, 8, dtype=torch.uint8)}
    out = bench.step_outputs(model, torch.tensor(0.75))
    assert float(out["loss"]) == 0.75 and float(out["metrics.ts"]) == 0.25
    assert torch.equal(out["metrics.binary"], model.last_metrics["binary"])
    assert {k[len("state."):] for k in out if k.startswith("state.")} == set(model.state_dict())
    assert torch.equal(out["state.fc1.weight"], model.fc1.weight)


def test_bench_rejects_zero_steps_and_unsupported_dumps():
    for extra in (["--steps", "0"], ["--config", "inference", "--dump-outputs", "x"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-500:])


def test_clock_sampler_without_nvidia_smi():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler.__new__(bench.ClockSampler)
    s.proc, s.lines, s.t0 = None, [], None
    assert s.stop()["sm_mhz"] is None
