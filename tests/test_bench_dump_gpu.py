"""bench.py --dump-outputs: the dumped frame is what the timed launches computed, byte for byte the frame a plain render of
the same workload returns, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_dumped_image_is_the_timed_frame(renderer, tmp_path):
    out = tmp_path / "out"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "nodof_512x512x64", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    j = json.loads(p.stdout.strip().splitlines()[-1])
    assert j["steps"] == 2 and len(j["step_ms"]) == 2 and j["parity_check"]["bit_exact"] is True
    assert abs(j["ms_per_step"] - sum(j["step_ms"]) / 2) < 1e-3 * j["ms_per_step"] + 1e-3
    assert sorted(os.listdir(out)) == ["image.npy"]
    img = np.load(out / "image.npy")
    assert img.dtype == np.float32 and img.shape == (512, 512, 4)
    import write_scenes
    d = str(tmp_path / "nodof")
    write_scenes.write_variant("nodof", d)
    renderer.set_scene(pt.load_scene_dir(d, "nodof"))
    res = renderer.render("nodof", 512, 512, (1, 2, 3, 4), spp=64, arith="fma")
    assert np.array_equal(img, res.image.astype(np.float32))
