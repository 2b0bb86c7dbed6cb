"""bench.py's reference arm runs on the CPU, so its JSON contract can be checked here; the committed bench lines of
our own arm (profiles/) are checked for the keys the contract names."""
import glob
import json
import os
import subprocess
import sys

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "gpu_launches"}


def test_reference_arm_prints_one_contract_line():
    # torchrun exports OMP_NUM_THREADS=1 to its children: the CPU arm must still use (and verify) every host core
    env = dict(os.environ, OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-budget", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert BASE_KEYS <= set(j) and j["impl"] == "reference" and j["vs_baseline"] is None
    assert j["metric"] == "Mrays/s" and j["unit"] == "Mrays/s" and j["higher_is_better"] is True and j["value"] > 0
    assert j["config"]["workload"] == "gridsoup1m_1920x1080x256" and j["config"]["baseline_config"] == 4
    cores = len(os.sched_getaffinity(0))
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] == cores and j["cpu_baseline"]["value"] == j["value"]
    assert "%d OpenMP threads verified" % cores in j["cpu_baseline"]["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_at_n_gt_1_is_the_strong_scaled_config5_scene_on_all_cores():
    """rank 0 of a torchrun launch (OMP_NUM_THREADS=1 exported): same workload at every N, every host core."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="4", LOCAL_RANK="0", OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "4", "--steps", "1", "--warmup", "0",
                        "--cpu-budget", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    j = json.loads(p.stdout.strip())
    assert j["config"]["workload"] == "gridsoup1m_3840x2160x64" and j["config"]["height"] == 2160 and j["scaling"] == "strong"
    assert j["n_gpus"] == 4 and j["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))


def test_reference_arm_light_workload_runs_the_unmodified_reference_binary():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "bin", "nodof", "CLSuperPathTracer")):
        import pytest
        pytest.skip("oracle/_ref not built")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--workload", "nodof_512x512x64"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    j = json.loads(p.stdout.strip())
    assert j["cpu_baseline"]["kind"] == "reference" and "%d OpenMP threads" % len(os.sched_getaffinity(0)) in j["cpu_baseline"]["sample"]


def test_reference_arm_runs_the_requested_number_of_steps():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "4", "--warmup", "0",
                        "--cpu-budget", "0.2", "--workload", "nodof_512x512x64"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    j = json.loads(p.stdout.strip())
    assert j["steps"] == 4 and len(j["step_ms"]) == 4 and all(ms > 0 for ms in j["step_ms"])
    assert abs(j["ms_per_step"] - sum(j["step_ms"]) / 4) < 1e-2


def test_bench_refuses_zero_steps_and_dumps_of_the_reference_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert p.returncode == 2 and p.stdout == "" and "error" in p.stderr, extra
    assert not os.path.exists(tmp_path / "out")


def test_dump_outputs_keeps_whole_arrays_below_the_limit_and_the_same_seeded_rows_above_it(tmp_path, monkeypatch):
    import numpy as np
    import bench
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (1024, 256, 4), dtype=np.uint8)
    acc = rng.random((1024, 256, 4), dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "whole"), {"image": img})
    assert sorted(os.listdir(tmp_path / "whole")) == ["image.npy"]
    got = np.load(tmp_path / "whole" / "image.npy")
    assert got.dtype == np.float32 and np.array_equal(got, img)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 << 20)         # image + accum as float32: 8 MiB
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"image": img, "accum": acc})
    d = tmp_path / "a"
    assert sorted(os.listdir(d)) == ["accum.npy", "image.npy", "rows.npy"]
    assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 3 << 20
    rows = np.load(d / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) > 100 and np.all(np.diff(rows) > 0)
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(d / "image.npy"), img[r]) and np.array_equal(np.load(d / "accum.npy"), acc[r])
    for f in os.listdir(d):
        assert (d / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_committed_bench_lines_follow_the_contract():
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r1_2*_bench_*.json")) + glob.glob(os.path.join(ROOT, "profiles", "r1_17_bench_*.json")))
    assert files
    for f in files:
        j = json.loads(open(f).read().strip().splitlines()[-1])
        assert BASE_KEYS <= set(j), f
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(j["e2e"]), f
        assert j["e2e"]["h2d_bytes_per_step"] > 0 and j["e2e"]["d2h_bytes_per_step"] > 0, f
        assert j["gpu_launches"] > 0 and j["warmup"] >= 3, f
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(j["clocks"]), f
        assert not set(j["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}, f
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(j["roofline"]), f
        assert "workload" in j["config"] and "l2" in j["config"], f


def test_committed_round2_lines_headline_config4_parity_and_ray_accounting():
    """round 2: headline = BASELINE config 4 at N = 1, config 5 strong-scaled at N > 1; every line checked what it timed
    (bit-exact row bands vs the oracle, reduced frame == one-GPU frame) and says how rays are counted."""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r2_4[0-9]_bench_n*.json")) + glob.glob(os.path.join(ROOT, "profiles", "r2_37_bench_n1.json")))
    assert len(files) >= 3
    for f in files:
        j = json.loads(open(f).read().strip().splitlines()[-1])
        assert BASE_KEYS <= set(j), f
        n = j["n_gpus"]
        assert j["config"]["workload"] == ("gridsoup1m_1920x1080x256" if n == 1 else "gridsoup1m_3840x2160x64"), f
        assert j["scaling"] == ("weak" if n == 1 else "strong"), f
        assert j["parity_check"]["bit_exact"] is True and j["parity_check"]["mismatching_pixels"] == 0, f
        if n > 1:
            assert j["parity_check"]["multi_gpu"]["identical"] is True, f
            assert len(j["per_rank"]["render_kernel_ms"]["per_rank"]) == n, f
        # rays: the reference's TraceRay calls; the elided dead shadow rays are reported, not hidden
        assert 0 < j["rays_traced_per_step"] < j["rays_per_step"] and "TraceRay calls of the REFERENCE" in j["ray_count"], f
        assert abs(j["value"] - j["rays_per_step"] / 1e3 / j["ms_per_step"]) < 1e-6 * j["value"], f
        assert j["roofline"]["bound"] == "fp32" and 0 < j["roofline"]["frac"] < 1 and j["roofline"]["peak"] > 60, f
        assert not set(j["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}, f
        if n == 1 and "configs" in j:
            for name, c in j["configs"].items():
                assert c["parity_check"]["bit_exact"] is True, (f, name)
                assert c["cpu_baseline"]["value"] > 0 and c["e2e"]["ms_per_step"] >= c["ms_per_step"], (f, name)
