"""bench.py's reference arm runs on the CPU: check the JSON contract of the line it prints (the b200 arm
prints the same keys plus roofline / clocks / gpu_launches; it needs a GPU, and its --dump-outputs is checked by a gpu test)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "3",
                          "--warmup", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().split("\n")[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "LM iterations/s" and line["higher_is_better"] is True
    assert line["vs_baseline"] is None and line["dtype"] == "f64" and line["data"] == "synthetic"
    assert line["value"] > 0 and abs(line["ms_per_step"] * line["value"] - 1e3) < 1e-6 * 1e3
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["config"]["workload"].startswith("cfg1")
    # the arm RUNS what it reports: K iterations inside the timed region, nothing extrapolated
    assert cb["lm_iterations"] == 3 and abs(cb["seconds"] * 1e3 - line["ms_per_step"] * 3) < 1e-6
    assert "nothing extrapolated" in cb["sample"] and "projected" not in line


def test_both_arms_print_the_same_config():
    """bench_config() is the one place the workload description comes from."""
    sys.path.insert(0, ROOT)
    import bench
    import ba_b200

    class A:
        workload, scale, solver = "cfg1", 1.0, "auto"
    p = ba_b200.synthetic.make_config(1)
    c = bench.bench_config(A, bench.WORKLOADS["cfg1"], p, 1, 10)
    assert c["n_obs"] == p.n_obs and c["lm_iterations"] == 10 and "l2" in c and "parallelism" in c


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1", "--gpus", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_stays_under_64_mb_with_a_fixed_sample(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(5)
    points = rng.normal(size=(3000000, 3)).astype(np.float32)
    points[:, 0] = np.arange(points.shape[0])   # row number, to check the sample against
    arrays = {"pose7": rng.normal(size=(10, 7)), "points": points, "intrinsics": np.ones(4)}
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["intrinsics.npy", "points.npy", "pose7.npy"]
    assert sum(np.load(tmp_path / "a" / n).nbytes for n in names) <= 64e6
    pts = np.load(tmp_path / "a" / "points.npy")
    assert pts.dtype == np.float64 and 2500000 < pts.shape[0] < 3000000 and pts.shape[1] == 3
    assert np.array_equal(pts, np.load(tmp_path / "b" / "points.npy"))
    # a sample of whole rows, in their original order
    rows = pts[:, 0].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and np.array_equal(pts, points[rows].astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "a" / "pose7.npy"), arrays["pose7"])


def test_dump_outputs_refused_by_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1",
                          "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_of_two_runs_are_identical(tmp_path):
    """The b200 arm with --dump-outputs: the timed solve runs exactly --steps LM iterations, and two runs with the same
    arguments write the same arrays."""
    lines = []
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "4", "--warmup", "1",
                              "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600,
                             cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads(out.stdout.strip().split("\n")[-1]))
    assert lines[0]["steps"] == 4 and lines[0]["detail"]["lm_iterations"] == 4
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["cost_per_iteration.npy", "intrinsics.npy", "points.npy", "pose7.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and np.array_equal(a, b), n
    pose, pts = np.load(tmp_path / "a" / "pose7.npy"), np.load(tmp_path / "a" / "points.npy")
    assert pose.shape == (7, 7) and pts.shape == (500, 3)
    cost = np.load(tmp_path / "a" / "cost_per_iteration.npy")
    assert cost.shape == (5,) and cost[-1] == lines[0]["final_cost"] and cost[0] == lines[0]["initial_cost"]


def test_committed_gpu_bench_line_keeps_the_contract():
    """The b200 arm needs a GPU; the line it printed at HEAD is committed (profiles/r02_bench_cfg5.log): its keys, the roofline
    object's enum / arithmetic and the phase shares are checked here, and executed_roofline() is re-run on its phase times."""
    sys.path.insert(0, ROOT)
    import bench
    line = None
    for l in open(os.path.join(ROOT, "profiles", "r02_bench_cfg5.log")):
        if l.startswith("{"):
            line = json.loads(l)
    assert line is not None
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "parity_vs_n1"):
        assert key in line, key
    assert line["metric"] == "LM iterations/s" and line["n_gpus"] == 1 and line["dtype"] == "f64" and line["vs_baseline"] is None
    assert abs(line["value"] * line["ms_per_step"] - 1e3) < 1e-6 * 1e3 and line["gpu_launches"] > 0
    assert line["config"]["workload"].startswith("cfg5") and line["config"]["n_obs"] == 8000000
    e = line["e2e"]
    assert 0 < e["value"] < line["value"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    r = line["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and r["limiter"]
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and r["traffic"] and 0 < r["share_of_step"] < 1
    assert abs(r["achieved"] - r["bytes"] / r["ms_per_step"] / 1e6) < 1e-6 * r["achieved"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and cb["lm_iterations"] >= 1
    assert line["clocks"]["reasons"] == [] and line["parity_vs_n1"]["ok"] is True
    shares = sum(v["share_of_step"] for v in line["phase_rooflines"].values())
    assert 0.9 < shares <= 1.0 + 1e-9
    # the same function on the same phase times gives the same dominant phase and fraction

    class Full:
        n_obs, n_pt, n_cam = 8000000, 2000000, 10000
    it = line["steps"]
    roof, table = bench.executed_roofline("cfg5", {k: v * it for k, v in line["phase_ms_per_step"].items()}, it, 4, Full,
                                          line["detail"]["sparse_pairs"], 0, dict(line["sparse_cholesky"]), 0, r["peak"], r["peak_source"])
    assert roof["kernel"] == r["kernel"] and abs(roof["frac"] - r["frac"]) < 1e-9 and set(table) == set(line["phase_rooflines"])
