"""bench.py's reference arm (`--impl reference`: the CPU oracle on the host cores) end to end on the small workload, and
the arithmetic of its roofline helper: the keys the driver parses are there, the faithful rate (every evaluation padded
to ActionSpace samples, meta.go:125-135) sits below the useful-work rate, rank > 0 prints nothing; and, on the GPU, the
search state --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e, timeout=300)


def test_reference_arm_json_line():
    r = _run(["--impl", "reference", "--workload", "C2", "--steps", "3", "--warmup", "3"])
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "mcts_sims_per_sec" and d["unit"] == "sims/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and cb["nproc"] >= cb["cores"]
    assert 0 < d["faithful_sims_per_sec"] < d["value"]           # 81 samples per evaluation instead of 1
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--workload", "C2", "--steps", "2", "--warmup", "3", "--gpus", "2"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_needs_the_b200_arm(tmp_path):
    r = _run(["--impl", "reference", "--workload", "C2", "--steps", "2", "--dump-outputs", str(tmp_path / "d")])
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_after_exactly_the_timed_steps(tmp_path):
    """--dump-outputs writes the search state after warm-up + `--steps` waves, float32/float64 within 64 MB, and the
    same bytes on a repeat run with the same arguments."""
    steps, warmup, games = 7, 3, 16
    dumps = []
    for i in range(2):
        d = tmp_path / str(i)
        r = _run(["--workload", "C2", "--games", str(games), "--steps", str(steps), "--warmup", str(warmup), "--no-e2e",
                  "--no-cpu-baseline", "--no-train", "--no-fast", "--dump-outputs", str(d)])
        assert r.returncode == 0, r.stderr[-500:]
        assert json.loads(r.stdout)["steps"] == steps
        dumps.append({f.stem: np.load(f) for f in d.iterdir()})
    a, b = dumps
    assert set(a) == {"games", "root_visits", "root_value_sum", "root_prior", "board"}
    assert all(x.dtype in (np.float32, np.float64) for x in a.values()) and sum(x.nbytes for x in a.values()) <= 64 << 20
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), k
    assert (a["games"] == np.arange(games)).all() and a["root_visits"].shape == (games, 2, 82)
    # the first warm-up step is the root evaluation, every later one a simulation; a root child is born with one visit
    v = a["root_visits"]
    sims = np.where(v > 0, v - 1, 0).sum(axis=2).max(axis=1)
    assert sims.max() == warmup + steps - 1, sims
    assert (np.abs(a["root_prior"].sum(axis=2).max(axis=1) - 1) < 1e-3).all()


def test_roofline_arithmetic():
    sys.path.insert(0, ROOT)
    import bench
    w = bench.WORKLOADS["C3"]
    assert bench.flops_per_eval(w) == 17065507816      # SURVEY section 8d: 17.07 GFLOP per 19x19 20x256 evaluation
    arm = dict(prof=dict(conv_ms=800.0, conv_launches=1000.0, kernel_kind=4), cnt=dict(evals=25600), dt=1.0, workload="C3")
    r = bench.roofline_of(arm, w, {"bf16_tflops_sustained": 1465.8}, "measured")
    per_launch = 2 * 9 * 256 * 512 * 361 * 25600 * 20 / 1000.0
    assert abs(r["algorithmic_flops_per_launch"] - per_launch) < 1 and abs(r["achieved"] - per_launch * 1000 / 0.8 / 1e12) < 1e-6
    assert abs(r["frac"] - r["achieved"] / 1465.8) < 1e-12 and r["tensor_passes_per_mac"] == 3.0
    assert "halo" in r["kernel"] and r["bound"] == "tensor" and r["unit"] == "TFLOP/s"
