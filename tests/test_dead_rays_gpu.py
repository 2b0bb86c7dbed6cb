"""Dead shadow-ray elision (pt_render_params.dead_rays, the library default): a sample whose camera ray hits a triangle
returns the facing ratio and ignores the illumination (CLSuperPathTracer/pathtracer.ocl:203-205,
CLSuperPathTracer_trianglegrid/pathtracer.ocl:268-270), so its shadow rays are not traced; only their RNG pairs are drawn
(pathtracer.ocl:168).  Bar: image bytes, float accumulation buffer and the final RNG state of every work-item stay
BIT-EXACT against the CPU oracle (which traces everything); `samples` equals the oracle's count, the ray / cell / test
counters drop to what was really traced.  tests/conftest.py runs every other GPU test in TRACE mode (counters == oracle)."""
import os
import subprocess

import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import ROOT, SEED_SETS

pytestmark = pytest.mark.gpu

WINDOWS = {"sky+mesh+sphere+square": (112, 144), "floor+sphere+shadow": (340, 372)}


def _same_bits(res, ref, rows, W, H, what):
    r0, r1 = rows
    a, b = res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]
    assert np.array_equal(a, b), "%s: RNG state differs in %d pixels" % (what, int((a != b).any(axis=2).sum()))
    a, b = res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)
    assert np.array_equal(a, b), "%s: accumulation differs in %d pixels" % (what, int((a != b).any(axis=2).sum()))
    assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), what
    assert res.counters["samples"] == ref["counters"]["samples"], what


@pytest.mark.parametrize("variant,mesh", [("base", "base"), ("lmem", "lmem"), ("grid", "grid"), ("base", "torus")])
@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("kernel", ["auto", "mega", "spec", "grid_queue", "grid_async"])
def test_elided_frames_keep_every_bit(renderer, scene_dirs, oracle_fma, oracle_sep, variant, mesh, arith, kernel):
    if kernel == "spec" and variant == "grid":
        pytest.skip("PT_KERNEL_SPEC is for the brute-force variants")
    if kernel.startswith("grid_") and variant != "grid":
        pytest.skip("%s is a trianglegrid kernel" % kernel)
    o = oracle_fma if arith == "fma" else oracle_sep
    d = scene_dirs[mesh]
    scene = pt.load_scene_dir(d, variant)
    renderer.set_scene(scene)
    osc = o.load_scene_dir(d, variant)
    if variant == "grid":
        renderer.build_grid(pt.grid_dims(scene))
    W = H = 512
    saved = 0
    for name, rows in WINDOWS.items():
        what = "%s/%s/%s/%s/%s" % (variant, mesh, arith, kernel, name)
        ref = o.render(variant, W, H, SEED_SETS[0], osc, rows=rows)
        el = renderer.render(variant, W, H, SEED_SETS[0], rows=rows, arith=arith, kernel=kernel, want_accum=True, want_rng=True, dead_rays="elide")
        tr = renderer.render(variant, W, H, SEED_SETS[0], rows=rows, arith=arith, kernel=kernel, want_accum=True, want_rng=True, dead_rays="trace")
        _same_bits(el, ref, rows, W, H, what + " elide")
        _same_bits(tr, ref, rows, W, H, what + " trace")
        for k in ("rays", "shadow_rays", "tri_tests", "prim_tests"):
            assert tr.counters[k] == ref["counters"][k], (what, k)
            assert el.counters[k] <= tr.counters[k], (what, k)
        assert el.counters["rays"] - el.counters["shadow_rays"] == tr.counters["rays"] - tr.counters["shadow_rays"], what
        saved += tr.counters["shadow_rays"] - el.counters["shadow_rays"]
    if mesh != "torus":                                 # the default mesh is inside the first window: rays were really saved
        assert saved > 0


def test_full_frames_elide_equals_trace(renderer, scene_dirs):
    """whole 512x512 frames, second seed set: identical accumulation buffers with and without the elision"""
    for variant in ("base", "lmem", "grid"):
        scene = pt.load_scene_dir(scene_dirs[variant], variant)
        renderer.set_scene(scene)
        if variant == "grid":
            renderer.build_grid(pt.grid_dims(scene))
        a = renderer.render(variant, 512, 512, SEED_SETS[1], want_accum=True, want_rng=True, dead_rays="elide")
        b = renderer.render(variant, 512, 512, SEED_SETS[1], want_accum=True, want_rng=True, dead_rays="trace")
        assert np.array_equal(a.accum.view(np.uint32), b.accum.view(np.uint32)), variant
        assert np.array_equal(a.rng_state, b.rng_state), variant
        assert np.array_equal(a.image, b.image), variant
        assert a.counters["rays"] < b.counters["rays"], variant


def test_no_cull_implies_trace(renderer, scene_dirs):
    scene = pt.load_scene_dir(scene_dirs["base"], "base")
    renderer.set_scene(scene)
    a = renderer.render("base", 256, 256, SEED_SETS[0], cull=False, dead_rays="elide")
    b = renderer.render("base", 256, 256, SEED_SETS[0], cull=False, dead_rays="trace")
    assert a.counters == b.counters


def test_soup1m_config4_window_elided(oracle_fma):
    """the benchmark's own default: config-4 scene (1 M triangles, 128^3 grid), big-grid megakernel, elision on"""
    import gen_mesh
    tris = gen_mesh.soup(1 << 20)
    lo, hi = gen_mesh.bbox_like_reference(tris)
    sph = np.array([1024, 0, 0, 0, 145, 0, 0, 2048, 0], np.int32)
    sq = np.array([4096, 0, 0, 0, 0, 0, 129, 0, 8192], np.int32)
    lights = np.array([[10, 4, 10, 400], [15, 2, 7, 300]], np.float32)
    scene = pt.Scene(sph, sq, tris, lights, lo, hi)
    osc = {"spheres": sph, "squares": sq, "triangles": tris, "lights": lights, "box_min": lo, "box_max": hi}
    with pt.Renderer(device=0) as r:
        r.set_scene(scene)
        g = pt.grid_dims(scene)
        r.build_grid(g)
        res, cell = np.array(g.res[:], np.int32), np.array(g.cell_size[:], np.float32)
        grid = {"box_min": lo, "box_max": hi, "res": res, "cell_size": cell, "csr": oracle_fma.build_grid(tris, lo, res, cell)}
        W, H, spp = 1920, 1080, 256
        for rows in [(420, 424), (700, 704)]:
            ref = oracle_fma.render("grid", W, H, SEED_SETS[0], osc, spp=spp, rows=rows, grid=grid)
            el = r.render("grid", W, H, SEED_SETS[0], rows=rows, spp=spp, want_accum=True, want_rng=True, dead_rays="elide")
            _same_bits(el, ref, rows, W, H, "config 4 rows %s elide" % (rows,))
            assert el.counters["rays"] < ref["counters"]["rays"]
            assert el.counters["cells_visited"] < ref["counters"]["cells_visited"]


def test_config4_window_trace_and_elide_legs():
    """config-4 scene (1 M triangles, 128^3 grid), one window: the elide and trace legs of the default kernel and of the
    grid_queue / grid_async kernels (which honour the elision too) give the same bits; elide traces fewer rays"""
    import gen_mesh
    tris = gen_mesh.soup(1 << 20)
    lo, hi = gen_mesh.bbox_like_reference(tris)
    sph = np.array([1024, 0, 0, 0, 145, 0, 0, 2048, 0], np.int32)
    sq = np.array([4096, 0, 0, 0, 0, 0, 129, 0, 8192], np.int32)
    lights = np.array([[10, 4, 10, 400], [15, 2, 7, 300]], np.float32)
    with pt.Renderer(device=0) as r:
        r.set_scene(pt.Scene(sph, sq, tris, lights, lo, hi))
        r.build_grid(pt.grid_dims(r._scene))
        W, H, spp, rows = 1920, 1080, 64, (540, 548)
        tr = r.render("grid", W, H, SEED_SETS[0], rows=rows, spp=spp, want_accum=True, want_rng=True, dead_rays="trace")
        for kernel in ("auto", "grid_queue", "grid_async"):
            el = r.render("grid", W, H, SEED_SETS[0], rows=rows, spp=spp, kernel=kernel, want_accum=True, want_rng=True, dead_rays="elide")
            r0, r1 = rows
            assert np.array_equal(el.accum[r0:r1].view(np.uint32), tr.accum[r0:r1].view(np.uint32)), kernel
            assert np.array_equal(el.rng_state.reshape(H, W, 4)[r0:r1], tr.rng_state.reshape(H, W, 4)[r0:r1]), kernel
            assert np.array_equal(el.image[r0:r1], tr.image[r0:r1]), kernel
            assert el.counters["samples"] == tr.counters["samples"], kernel
            assert el.counters["rays"] < tr.counters["rays"], kernel


@pytest.mark.parametrize("variant,dirname", [("base", "CLSuperPathTracer"), ("grid", "CLSuperPathTracer_trianglegrid")])
def test_cli_default_is_elide_and_bytes_match_oracle(scene_dirs, oracle_fma, variant, dirname):
    """the drop-in executable with its defaults (PT_DEAD_RAYS unset -> elide) writes the oracle's result.ppm bytes"""
    exe = os.path.join(ROOT, "opencl_montecarlo_path_tracing_b200", "bin", dirname, "CLSuperPathTracer")
    d = scene_dirs[variant]
    env = {k: v for k, v in os.environ.items() if k != "PT_DEAD_RAYS"}
    env["PT_SEEDS"] = "1,2,3,4"
    p = subprocess.run([exe, "320", "256"], cwd=d, env=env, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    ref = oracle_fma.render(variant, 320, 256, (1, 2, 3, 4), oracle_fma.load_scene_dir(d, variant), want_accum=False, want_rng=False)
    tmp = os.path.join(d, "oracle_expected_elide.ppm")
    oracle_fma.save_pam(tmp, ref["image"])
    assert open(os.path.join(d, "result.ppm"), "rb").read() == open(tmp, "rb").read()
