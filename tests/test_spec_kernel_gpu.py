"""PT_KERNEL_SPEC (pt_spec.cuh): light pixels thread-per-pixel, pixels that see the mesh warp-per-pixel with 32 samples traced
at once from SPECULATED offsets into the pixel's RNG stream.  Bar: bit-exact against the CPU oracle — image, float sums,
final RNG state of every pixel (the stream position the speculation must reproduce) and the work counters (only accepted
samples may count) — on whole frames, both brute-force variants, both arithmetic policies, sample counts that are not a
multiple of the batch of 32, and on pixels where hit and sky samples alternate (every batch mispredicts).
Follows CLSuperPathTracer/pathtracer.ocl:139-241 and CLSuperPathTracer_lmem/pathtracer.ocl:138-254."""
import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import SEED_SETS

pytestmark = pytest.mark.gpu
COUNTERS = ("samples", "rays", "shadow_rays", "tri_tests", "prim_tests")
FIVE_LIGHTS = np.array([[10, 4, 10, 200], [15, 2, 7, 0], [3, -2, 14, 90], [8, 5, 3, 60], [14, 0, 13.5, 300]], np.float32)


def _same(res, ref, H, W, rows, what):
    r0, r1 = rows
    assert np.array_equal(res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]), what + ": RNG state"
    assert np.array_equal(res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)), what + ": float sums"
    assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), what + ": image"
    for k in COUNTERS:
        assert res.counters[k] == ref["counters"][k], (what, k, res.counters[k], ref["counters"][k])


@pytest.mark.parametrize("variant", ["base", "lmem"])
@pytest.mark.parametrize("arith", ["fma", "separate"])
def test_spec_full_frame_bit_exact(renderer, scene_dirs, oracle_fma, oracle_sep, variant, arith):
    o = oracle_fma if arith == "fma" else oracle_sep
    d = scene_dirs[variant]
    renderer.set_scene(pt.load_scene_dir(d, variant))
    osc = o.load_scene_dir(d, variant)
    W = H = 512
    for seeds in SEED_SETS:
        res = renderer.render(variant, W, H, seeds, kernel="spec", arith=arith, want_accum=True, want_rng=True)
        ref = o.render(variant, W, H, seeds, osc)
        _same(res, ref, H, W, (0, H), "%s/%s/%s" % (variant, arith, seeds))
        assert res.counters["tri_tests_executed"] < res.counters["tri_tests"]


@pytest.mark.parametrize("spp", [1, 7, 32, 33, 100])
def test_spec_sample_counts_and_scene_memories(renderer, scene_dirs, oracle_fma, spp):
    """Sample counts that cut the last batch or window short, with the scene's two lights and with 1 and 5 (odd counts
    place the window-mode candidates one RNG pair apart instead of two)"""
    d = scene_dirs["torus"]
    scene = pt.load_scene_dir(d, "base")
    osc = oracle_fma.load_scene_dir(d, "base")
    W, H, rows = 512, 512, (140, 172)
    for lights in (scene.lights, FIVE_LIGHTS[:1], FIVE_LIGHTS):
        scene.lights = osc["lights"] = lights
        renderer.set_scene(scene)
        ref = oracle_fma.render("base", W, H, SEED_SETS[0], osc, spp=spp, rows=rows)
        for mem in ("smem", "const"):
            res = renderer.render("base", W, H, SEED_SETS[0], rows=rows, spp=spp, kernel="spec", scene_mem=mem, want_accum=True, want_rng=True)
            _same(res, ref, H, W, rows, "torus spp %d %s %d lights" % (spp, mem, len(lights)))


def test_spec_mispredicting_pixels(renderer, oracle_fma):
    """A sparse cloud of big triangles in view and above the horizon, against the sky: along its silhouette hit and sky
    samples alternate inside one pixel, so batches are cut at the first surprise and redone; rows through the silhouette
    must still be bit-exact."""
    from test_light_counts_gpu import silhouette_triangles
    tris = silhouette_triangles()
    sph, sq = np.zeros(9, np.int32), np.zeros(9, np.int32)
    lights = np.array([[10, 4, 10, 400], [15, 2, 7, 300]], np.float32)
    scene = pt.Scene(sph, sq, tris, lights)
    osc = {"spheres": sph, "squares": sq, "triangles": tris, "lights": lights}
    renderer.set_scene(scene)
    W, H = 256, 256
    full = renderer.render("base", W, H, SEED_SETS[0], kernel="mega", want_accum=True)
    spec = renderer.render("base", W, H, SEED_SETS[0], kernel="spec", want_accum=True, want_rng=True)
    assert np.array_equal(full.accum.view(np.uint32), spec.accum.view(np.uint32))
    # rows where the mesh is visible against the sky (alpha-independent: colour differs from pure sky rows)
    ref = oracle_fma.render("base", W, H, SEED_SETS[0], osc)
    _same(spec, ref, H, W, (0, H), "silhouette scene")
    sky = oracle_fma.render("base", W, H, SEED_SETS[0], dict(osc, triangles=tris[:0]), want_accum=False, want_rng=False)
    assert (ref["image"] != sky["image"]).any()                             # the triangles are in view
    # SPEC threw speculation away: triangle tests the megakernel never ran
    assert spec.counters["tri_tests_executed"] > full.counters["tri_tests_executed"] > 0


def test_spec_tiles_stripes_and_culls(renderer, scene_dirs):
    """Row windows, interleaved stripes and the conservative culls compose exactly as with the megakernel."""
    d = scene_dirs["base"]
    renderer.set_scene(pt.load_scene_dir(d, "base"))
    W, H = 640, 360
    whole = renderer.render("base", W, H, SEED_SETS[1], kernel="mega", want_accum=True, want_rng=True)
    spec = renderer.render("base", W, H, SEED_SETS[1], kernel="spec", want_accum=True, want_rng=True)
    assert np.array_equal(whole.accum.view(np.uint32), spec.accum.view(np.uint32)) and np.array_equal(whole.rng_state, spec.rng_state)
    for k in COUNTERS:
        assert whole.counters[k] == spec.counters[k], k
    acc = np.zeros_like(whole.accum)
    for rank in range(3):
        acc += renderer.render("base", W, H, SEED_SETS[1], kernel="spec", want_accum=True, interleave=8, rank=rank, nranks=3).accum
    assert np.array_equal(acc.view(np.uint32), whole.accum.view(np.uint32))
    nocull = renderer.render("base", W, H, SEED_SETS[1], kernel="spec", want_accum=True, cull=False)
    assert np.array_equal(nocull.accum.view(np.uint32), whole.accum.view(np.uint32))
