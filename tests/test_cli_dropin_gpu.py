"""The drop-in executables: same argv, scene files from the CWD, stdout lines in the reference's order, and a
result.ppm whose bytes equal what the oracle writes for the printed seeds."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

BIN = os.path.join(ROOT, "opencl_montecarlo_path_tracing_b200", "bin")
DIRS = {"base": "CLSuperPathTracer", "lmem": "CLSuperPathTracer_lmem", "nodof": "CLSuperPathTracer_lmem_NoDoF",
        "grid": "CLSuperPathTracer_trianglegrid"}
EXPECTED_ORDER = {
    "base": ["Usage:", "number of platforms:", "selected platform", "number of devices:", "selected device", "compiling:",
             "=== BUILD LOG ===", "Seeds:", "Processing image", "Cam values:", "Number of triangles:", "Number of lights:",
             "Successfully created render image result.ppm", "rendering :", "read render data :", "Total time:"],
    "grid": ["Usage:", "Seeds:", "Processing image", "Cam values:", "Triangles bounding box values:", "Triangles grid size:",
             "Light 0:", "Number of triangles:", "Number of lights:", "Successfully created", "init triangles grid :",
             "rendering :", "read render data :", "Total time:"],
    "nodof": ["Usage:", "Seeds:", "Light 0:", "Light 1:", "Number of triangles: 1", "Number of lights: 2", "rendering :",
              "reduce img samples :", "read render data :", "Total time:"],
}


@pytest.mark.parametrize("variant,args", [("base", ["256", "192"]), ("lmem", []), ("nodof", ["384", "384"]), ("grid", ["512", "512", "6.5"])])
def test_cli_matches_oracle(scene_dirs, oracle_fma, variant, args):
    exe = os.path.join(BIN, DIRS[variant], "CLSuperPathTracer")
    d = scene_dirs[variant]
    env = dict(os.environ, PT_SEEDS="123456789,42,7,99999")
    p = subprocess.run([exe, *args], cwd=d, env=env, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    out = p.stdout
    pos = 0
    for token in EXPECTED_ORDER.get(variant, EXPECTED_ORDER["base"]):
        k = out.find(token, pos)
        assert k >= 0, "stdout misses %r after offset %d:\n%s" % (token, pos, out)
        pos = k
    seeds = tuple(int(x) for x in re.search(r"Seeds: (\d+), (\d+), (\d+), (\d+)", out).groups())
    assert seeds == (123456789, 42, 7, 99999)
    w = int(args[0]) if args else 512
    h = int(args[1]) if len(args) > 1 else 512
    modifier = float(args[2]) if len(args) > 2 else 3.0
    ref = oracle_fma.render(variant, w, h, seeds, oracle_fma.load_scene_dir(d, variant), want_accum=False, want_rng=False, modifier=modifier)
    tmp = os.path.join(d, "oracle_expected.ppm")
    oracle_fma.save_pam(tmp, ref["image"])
    assert open(os.path.join(d, "result.ppm"), "rb").read() == open(tmp, "rb").read()
    assert ("Processing image %dx%d with data size %d bytes" % (w, h, w * h * 4)) in out


@pytest.mark.parametrize("variant", ["base", "lmem"])
@pytest.mark.parametrize("nlights", [1, 5])
def test_cli_other_light_counts(scene_dirs, oracle_fma, tmp_path, variant, nlights):
    """The executables' default 512x512 frame (AUTO picks the speculative kernel there) with a lights.txt of 1 and 5 lights"""
    from test_spec_kernel_gpu import FIVE_LIGHTS
    d = str(tmp_path / variant)
    shutil.copytree(scene_dirs[variant], d)
    with open(os.path.join(d, "lights.txt"), "w") as f:
        f.write("\n".join("%g" % v for v in FIVE_LIGHTS[:nlights].reshape(-1)))
    exe = os.path.join(BIN, DIRS[variant], "CLSuperPathTracer")
    env = dict(os.environ, PT_SEEDS="123456789,42,7,99999")
    p = subprocess.run([exe], cwd=d, env=env, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert ("Number of lights: %d" % nlights) in p.stdout and "Processing image 512x512" in p.stdout
    osc = oracle_fma.load_scene_dir(d, variant)
    assert np.array_equal(osc["lights"], FIVE_LIGHTS[:nlights])
    ref = oracle_fma.render(variant, 512, 512, (123456789, 42, 7, 99999), osc, want_accum=False, want_rng=False)
    tmp = os.path.join(d, "oracle_expected.ppm")
    oracle_fma.save_pam(tmp, ref["image"])
    assert open(os.path.join(d, "result.ppm"), "rb").read() == open(tmp, "rb").read()


def test_cli_wall_clock_seeds_and_error_convention(scene_dirs, tmp_path):
    exe = os.path.join(BIN, DIRS["base"], "CLSuperPathTracer")
    env = {k: v for k, v in os.environ.items() if k != "PT_SEEDS"}
    p = subprocess.run([exe, "64", "64"], cwd=scene_dirs["base"], env=env, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0
    seeds = [int(x) for x in re.search(r"Seeds: (\d+), (\d+), (\d+), (\d+)", p.stdout).groups()]
    assert all(0 <= s < 2 ** 27 for s in seeds)          # 27-bit mask of the reference
    # a missing scene file is reported ocl_check-style ("<what> - error <n>", exit status 1) instead of crashing
    q = subprocess.run([exe, "64", "64"], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=120)
    assert q.returncode == 1 and " - error " in q.stderr


def test_cli_extra_outputs(scene_dirs):
    """PT_EXTRA_OUTPUT=png,ppm: the same frame as result.ppm (PAM) in PNG and binary P6 (SURVEY.md 8f rank 4)."""
    import zlib
    import opencl_montecarlo_path_tracing_b200 as pt
    exe = os.path.join(BIN, DIRS["lmem"], "CLSuperPathTracer")
    d = scene_dirs["lmem"]
    env = dict(os.environ, PT_SEEDS="1,2,3,4", PT_EXTRA_OUTPUT="png,ppm")
    p = subprocess.run([exe, "96", "64"], cwd=d, env=env, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    pam, _ = pt.load_pam(os.path.join(d, "result.ppm"))
    assert pam.shape == (64, 96, 4)
    raw = open(os.path.join(d, "result_p6.ppm"), "rb").read()
    hdr = b"P6\n96 64\n255\n"
    assert raw.startswith(hdr) and np.array_equal(np.frombuffer(raw[len(hdr):], np.uint8).reshape(64, 96, 3), pam[..., :3])
    png = open(os.path.join(d, "result.png"), "rb").read()
    k = png.index(b"IDAT")
    n = int.from_bytes(png[k - 4:k], "big")
    rows = np.frombuffer(zlib.decompress(png[k + 4:k + 4 + n]), np.uint8).reshape(64, 96 * 4 + 1)
    assert np.array_equal(rows[:, 1:].reshape(64, 96, 4), pam)
