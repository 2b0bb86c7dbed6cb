"""Build-container only: the oracle against the reference itself, run here.  Skipped where /root/reference
or oracle/_ref is absent (the GPU box); tests/golden carries the same pin there."""
import os
import subprocess

import numpy as np
import pytest

from conftest import REF_BUILD, REFERENCE, SEED_SETS

pytestmark = pytest.mark.needs_reference
have_ref = all(os.path.exists(os.path.join(REF_BUILD, "bin", v, e)) for v, e in
               (("base", "CLSuperPathTracer"), ("lmem", "CLSuperPathTracer"), ("nodof", "CLSuperPathTracer"), ("grid", "CLSuperPathTracer"),
                ("bidir", "CLSuperBidirectionalPathTracer")))


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="needs /root/reference")
def test_scene_files_regenerate_byte_identical():
    import write_scenes
    assert write_scenes.verify_against_reference(REFERENCE)


@pytest.mark.skipif(not have_ref, reason="needs oracle/_ref (make -C oracle ref)")
@pytest.mark.parametrize("variant,size", [("base", (256, 384)), ("lmem", (256, 384)), ("nodof", (256, 384)), ("grid", (256, 384)),
                                          ("bidir", (320, 384))])
def test_result_ppm_identical(oracle_sep, scene_dirs, tmp_path, variant, size):
    """Unmodified reference host + kernel (CPU, refrt) vs oracle_render: identical result.ppm bytes."""
    w, h = size
    d = scene_dirs[variant]
    env = dict(os.environ, PT_SEEDS=",".join(str(s) for s in SEED_SETS[1]))
    exe = "CLSuperBidirectionalPathTracer" if variant == "bidir" else "CLSuperPathTracer"
    subprocess.run([os.path.join(REF_BUILD, "bin", variant, exe), str(w), str(h)], cwd=d, env=env, check=True,
                   capture_output=True)
    raw = open(os.path.join(d, "result.ppm"), "rb").read()
    k = raw.index(b"ENDHDR\n") + 7
    ref_img = np.frombuffer(raw[k:], np.uint8).reshape(h, w, 4)
    out = oracle_sep.render(variant, w, h, SEED_SETS[1], oracle_sep.load_scene_dir(d, variant), want_rng=False, want_accum=False)
    assert np.array_equal(out["image"], ref_img)
    oracle_sep.save_pam(os.path.join(str(tmp_path), "o.ppm"), out["image"])
    assert open(os.path.join(str(tmp_path), "o.ppm"), "rb").read() == raw


@pytest.mark.skipif(not have_ref, reason="needs oracle/_ref (make -C oracle ref)")
@pytest.mark.parametrize("variant", ["base", "lmem", "bidir"])
@pytest.mark.parametrize("nlights", [1, 5])
def test_other_light_counts_match_the_reference(oracle_sep, tmp_path, variant, nlights):
    """lights.txt with 1 and with MAX_LIGHTS = 5 entries (one of them zero-intensity: base skips it AFTER drawing its
    random numbers, the lmem family does not skip it): unmodified reference vs oracle, identical result.ppm bytes."""
    import write_scenes
    d = str(tmp_path / "scene")
    write_scenes.write_variant(variant, d)
    lights = [(10, 4, 10, 200), (15, 2, 7, 0), (3, -2, 14, 90), (8, 5, 3, 60), (14, 0, 13.5, 300)][:nlights]
    open(os.path.join(d, "lights.txt"), "w").write("\n".join("\n".join(str(x) for x in l) for l in lights))
    w, h = 256, 352
    env = dict(os.environ, PT_SEEDS=",".join(str(s) for s in SEED_SETS[0]))
    exe = "CLSuperBidirectionalPathTracer" if variant == "bidir" else "CLSuperPathTracer"
    out = subprocess.run([os.path.join(REF_BUILD, "bin", variant, exe), str(w), str(h)], cwd=d, env=env, check=True,
                         capture_output=True, text=True).stdout
    assert "Number of lights: %d" % nlights in out
    raw = open(os.path.join(d, "result.ppm"), "rb").read()
    k = raw.index(b"ENDHDR\n") + 7
    ref_img = np.frombuffer(raw[k:], np.uint8).reshape(h, w, 4)
    sc = oracle_sep.load_scene_dir(d, variant)
    assert sc["lights"].shape[0] == nlights
    got = oracle_sep.render(variant, w, h, SEED_SETS[0], sc, want_rng=False, want_accum=False)
    assert np.array_equal(got["image"], ref_img)
