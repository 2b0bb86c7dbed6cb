"""Diffuse bounces with Russian roulette (include/ptcuda.h pt_set_bounces, DESIGN.md 5b) on the GPU, against the path oracle.

Bar: image bytes, float accumulation buffer (as uint32), the final RNG state of every pixel and the work counters equal
oracle_render_bounces' under both arithmetic policies, with dead_rays "trace" and "elide" each set explicitly (elide: the
same bits, fewer shadow rays).  Every case also checks that the oracle frame reaches what it is meant to test: bounce rays,
hits refused by the bounce rays' lower bound, Russian-roulette terminations.  Then progressive ranges, row stripes, the
refusals, switching B on one context and the drop-in executables with PT_BOUNCES."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import ROOT, SEED_SETS
from test_light_counts_gpu import build_scene, set_scene
from test_spec_kernel_gpu import FIVE_LIGHTS

pytestmark = pytest.mark.gpu

W = H = 512
SEEDS = SEED_SETS[0]
SPP = 8
BRUTE_COUNTERS = ("samples", "rays", "shadow_rays", "tri_tests", "prim_tests")
GRID_COUNTERS = ("samples", "rays", "shadow_rays", "cells_visited", "tri_tests")
# case: (variant, scene, render keywords)
CASES = {
    "base-smem": ("base", "default", {"scene_mem": "smem"}),
    "base-const": ("base", "default", {"scene_mem": "const"}),
    "lmem-smem": ("lmem", "default", {"scene_mem": "smem"}),
    "lmem-const": ("lmem", "default", {"scene_mem": "const"}),
    "base-cluster-cull": ("base", "default", {"cluster_cull": "on"}),
    "grid": ("grid", "default", {}),
    "grid-soup": ("grid", "soup", {}),
}
# row windows: mesh, sky and spheres / floor, spheres, squares and shadows
WINDOWS = {"default": ((112, 128), (340, 356)), "soup": ((250, 258), (420, 428))}


@pytest.fixture(scope="module")
def rend():
    r = pt.Renderer(device=0)
    yield r
    r.close()


@pytest.fixture(scope="module")
def poracle():
    from oracle.pyoracle import cpu_has_fma
    from oracle_paths.pypaths import PathOracle
    out = {"separate": PathOracle(contract=0)}
    if cpu_has_fma():
        out["fma"] = PathOracle(contract=1)
    return out


@pytest.fixture(scope="module")
def frames():
    return {}


def oracle_frame(cache, poracle, arith, variant, scene, lset, osc, rows, bounces, **kw):
    if arith not in poracle:
        pytest.skip("host CPU lacks FMA")
    key = (variant, scene, lset, arith, rows, bounces, tuple(sorted(kw.items())))
    if key not in cache:
        cache[key] = poracle[arith].render_bounces(variant, W, H, SEEDS, osc, bounces, spp=SPP, rows=rows, **kw)
    return cache[key]


def same_bits(res, ref, rows, what):
    r0, r1 = rows
    a, b = res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]
    assert np.array_equal(a, b), "%s: RNG state differs in %d pixels" % (what, int((a != b).any(axis=-1).sum()))
    a, b = res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)
    assert np.array_equal(a, b), "%s: accumulation differs in %d pixels" % (what, int((a != b).any(axis=2).sum()))
    assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), "%s: image bytes" % what


def scene_of(scene_dirs, variant, scene, lights=None):
    """-> (pt.Scene, oracle scene dict); lights None: those of the variant's scene files"""
    if lights is None:
        lights = pt.load_scene_dir(scene_dirs[variant], variant).lights
    return build_scene(scene_dirs, variant, scene, lights)


@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("bounces", [1, 2, 5])
@pytest.mark.parametrize("case", list(CASES))
def test_bounces_bit_exact(rend, scene_dirs, poracle, frames, case, bounces, arith):
    variant, scene, kw = CASES[case]
    s, osc = scene_of(scene_dirs, variant, scene)
    set_scene(rend, variant, s)
    counters = GRID_COUNTERS if variant == "grid" else BRUTE_COUNTERS
    reach = {"bounce_rays": 0, "tmin_rejections": 0, "rr_terminations": 0}
    saved = 0
    for rows in WINDOWS[scene]:
        ref = oracle_frame(frames, poracle, arith, variant, scene, "scene", osc, rows, bounces)
        for k in reach:
            reach[k] += ref["path_counters"][k]
        rc = ref["counters"]
        assert rc["rays"] - rc["samples"] - rc["shadow_rays"] == ref["path_counters"]["bounce_rays"]
        what = "%s/B=%d/%s rows %s" % (case, bounces, arith, rows)
        res = rend.render(variant, W, H, SEEDS, spp=SPP, rows=rows, arith=arith, want_accum=True, want_rng=True,
                          dead_rays="trace", bounces=bounces, **kw)
        assert rend.last_kernel() == "mega"
        same_bits(res, ref, rows, what)
        for k in counters:
            assert res.counters[k] == rc[k], (what, k, res.counters[k], rc[k])
        el = rend.render(variant, W, H, SEEDS, spp=SPP, rows=rows, arith=arith, want_accum=True, want_rng=True,
                         dead_rays="elide", bounces=bounces, **kw)
        same_bits(el, ref, rows, what + " elide")
        assert el.counters["samples"] == rc["samples"]
        assert el.counters["shadow_rays"] <= rc["shadow_rays"], what
        assert el.counters["rays"] - el.counters["shadow_rays"] == rc["rays"] - rc["shadow_rays"], what
        saved += rc["shadow_rays"] - el.counters["shadow_rays"]
    assert reach["bounce_rays"] > 0 and reach["tmin_rejections"] > 0, (case, reach)
    if bounces >= 5:
        assert reach["rr_terminations"] > 0, (case, reach)
    assert saved > 0, case                                   # the mesh window has triangle hits, whose shadow rays are dead


@pytest.mark.parametrize("nl", [0, 2, 5])
def test_bounces_light_counts(rend, scene_dirs, poracle, frames, nl):
    """0, 2 and 5 lights at B = 2 (base, shared-memory scene): the light pairs come before the roulette and disk pairs"""
    lights = FIVE_LIGHTS[:nl]
    s, osc = scene_of(scene_dirs, "base", "default", lights)
    rend.set_scene(s)
    arith = "fma" if "fma" in poracle else "separate"
    for rows in WINDOWS["default"]:
        ref = oracle_frame(frames, poracle, arith, "base", "default", "five%d" % nl, osc, rows, 2)
        assert ref["path_counters"]["bounce_rays"] > 0
        if nl:
            assert ref["counters"]["shadow_rays"] > 0
        res = rend.render("base", W, H, SEEDS, spp=SPP, rows=rows, arith=arith, want_accum=True, want_rng=True,
                          dead_rays="trace", bounces=2, scene_mem="smem")
        same_bits(res, ref, rows, "%d lights rows %s" % (nl, rows))
        for k in BRUTE_COUNTERS:
            assert res.counters[k] == ref["counters"][k], (nl, rows, k)


def test_bounces_progressive(rend, scene_dirs):
    """A chain [0, 1) [1, 15) [15, 48) at B = 2 equals one launch; a saved state resumes it; another B or a new scene is refused"""
    s, _ = scene_of(scene_dirs, "lmem", "default")
    rend.set_scene(s)
    kw = dict(spp=48, rows=(330, 350), dead_rays="trace", bounces=2)
    one = rend.render("lmem", W, H, SEEDS, want_accum=True, want_rng=True, **kw)
    for b, e in ((0, 1), (1, 15), (15, 48)):
        last = rend.render("lmem", W, H, SEEDS, samples=(b, e), want_accum=True, want_rng=True, **kw)
        if e == 15:
            cp = last
    assert np.array_equal(last.image, one.image)
    assert np.array_equal(last.accum.view(np.uint32), one.accum.view(np.uint32))
    assert np.array_equal(last.rng_state, one.rng_state)
    rend.set_render_state("lmem", W, H, SEEDS, 15, cp.accum, cp.rng_state, **{k: v for k, v in kw.items() if k != "dead_rays"})
    res = rend.render("lmem", W, H, SEEDS, samples=(15, 48), want_accum=True, want_rng=True, **kw)
    assert np.array_equal(res.accum.view(np.uint32), one.accum.view(np.uint32)) and np.array_equal(res.image, one.image)
    # another B continues no progression of B = 2
    rend.render("lmem", W, H, SEEDS, samples=(0, 15), **kw)
    with pytest.raises(pt.PtError):
        rend.render("lmem", W, H, SEEDS, samples=(15, 48), **dict(kw, bounces=3))
    rend.render("lmem", W, H, SEEDS, samples=(0, 15), **kw)
    rend.set_scene(s)
    with pytest.raises(pt.PtError):
        rend.render("lmem", W, H, SEEDS, samples=(15, 48), **kw)


@pytest.mark.parametrize("variant", ["base", "grid"])
def test_bounces_stripes(rend, scene_dirs, variant):
    """Ranks 0..2 of row_interleave = 8, rendered on one device and summed, equal the full frame"""
    s, _ = scene_of(scene_dirs, variant, "default")
    set_scene(rend, variant, s)
    rows = (96, 144)
    kw = dict(spp=SPP, rows=rows, dead_rays="trace", bounces=2, want_accum=True)
    full = rend.render(variant, W, H, SEEDS, **kw)
    acc = np.zeros_like(full.accum)
    for rank in range(3):
        acc += rend.render(variant, W, H, SEEDS, interleave=8, rank=rank, nranks=3, **kw).accum
    assert np.array_equal(acc.view(np.uint32), full.accum.view(np.uint32))


def test_bounces_multi_gpu(scene_dirs, poracle):
    """pt_multi over 2 GPUs (row stripes + NCCL reduce) with B = 2 equals the oracle frame"""
    L = pt._lib.cuda_lib()
    if L.pt_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s, osc = scene_of(scene_dirs, "base", "default")
    arith = "fma" if "fma" in poracle else "separate"
    rows = (330, 346)
    ref = poracle[arith].render_bounces("base", W, H, SEEDS, osc, 2, spp=SPP, rows=rows)
    m = L.pt_multi_create(2)
    assert m
    try:
        cs = s.to_c()
        assert L.pt_multi_set_scene(m, C.byref(cs)) == 0
        assert L.pt_multi_set_bounces(m, 2) == 0
        p = pt.make_params("base", W, H, SEEDS, spp=SPP, rows=rows, arith=arith)
        cam = pt.camera()
        e = L.pt_multi_launch_pathtracer(m, C.byref(cam), C.byref(p))
        assert e, L.pt_last_error().decode()
        ptr = L.pt_multi_map_render(m, None)
        img = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(H, W, 4)).copy()
        L.pt_release_event(e)
    finally:
        L.pt_multi_destroy(m)
    assert np.array_equal(img[rows[0]:rows[1]], ref["image"][rows[0]:rows[1]])


def test_bounces_refusals(rend, scene_dirs):
    s, _ = scene_of(scene_dirs, "base", "default")
    rend.set_scene(s)
    for b in (-1, 16):
        with pytest.raises(pt.PtError, match="pt_set_bounces"):
            rend.set_bounces(b)
    kw = dict(rows=(0, 8), spp=SPP)
    with pytest.raises(pt.PtError, match="bounces"):
        rend.render("nodof", W, H, SEEDS, bounces=1, rows=(0, 8))
    rend.light_tracer(SEEDS, n_vlp=64)
    with pytest.raises(pt.PtError, match="bounces"):
        rend.render("bidir", W, H, SEEDS, bounces=1, **kw)
    lo, hi = rend.vlp_bounds()
    rend.build_vlp_grid(pt.vlp_grid_dims(lo, hi, 64 * 2))
    with pytest.raises(pt.PtError, match="bounces"):
        rend.render("vlpgrid", W, H, SEEDS, bounces=1, **kw)
    for kernel in ("spec", "persistent", "wavefront"):
        with pytest.raises(pt.PtError, match="per-pixel kernel"):
            rend.render("base", W, H, SEEDS, bounces=1, kernel=kernel, **kw)
    rend.render("base", W, H, SEEDS, bounces=1, kernel="auto", **kw)
    assert rend.last_kernel() == "mega"
    sg, _ = scene_of(scene_dirs, "grid", "default")
    set_scene(rend, "grid", sg)
    for kernel in ("grid_tma", "grid_stream", "grid_pool", "grid_queue", "grid_async", "persistent", "wavefront"):
        with pytest.raises(pt.PtError, match="per-pixel kernel"):
            rend.render("grid", W, H, SEEDS, bounces=2, kernel=kernel, **kw)
    rend.render("grid", W, H, SEEDS, bounces=2, kernel="auto", **kw)
    assert rend.last_kernel() == "mega"
    # B = 0 keeps every flavour
    rend.render("grid", W, H, SEEDS, bounces=0, kernel="grid_queue", **kw)
    assert rend.last_kernel() == "grid_queue"


@pytest.mark.parametrize("variant", ["base", "grid"])
def test_bounces_then_zero_is_a_fresh_context(rend, scene_dirs, variant):
    """B = 3 and then B = 0 on one renderer: the second frame has the bytes of a fresh context's"""
    s, _ = scene_of(scene_dirs, variant, "default")
    set_scene(rend, variant, s)
    kw = dict(spp=SPP, rows=(112, 144), want_accum=True, want_rng=True)
    b3 = rend.render(variant, W, H, SEEDS, bounces=3, **kw)
    b0 = rend.render(variant, W, H, SEEDS, bounces=0, **kw)
    with pt.Renderer(device=0) as fresh:
        set_scene(fresh, variant, s)
        f = fresh.render(variant, W, H, SEEDS, **kw)
        k_fresh = fresh.last_kernel()
    assert not np.array_equal(b3.accum, f.accum)
    assert np.array_equal(b0.image, f.image) and np.array_equal(b0.accum.view(np.uint32), f.accum.view(np.uint32))
    assert np.array_equal(b0.rng_state, f.rng_state)
    assert rend.last_kernel() == k_fresh


@pytest.mark.parametrize("variant,args", [("base", ["256", "192"]), ("grid", ["512", "256", "6.5"])])
def test_cli_bounces(scene_dirs, poracle, tmp_path, variant, args):
    """PT_BOUNCES=2 with the drop-ins: the reference's stdout lines, result.ppm == the oracle frame"""
    from test_cli_dropin_gpu import BIN, DIRS, EXPECTED_ORDER
    d = str(tmp_path / variant)
    shutil.copytree(scene_dirs[variant], d)
    exe = os.path.join(BIN, DIRS[variant], "CLSuperPathTracer")
    arith = "fma" if "fma" in poracle else "separate"
    env = dict(os.environ, PT_SEEDS="123456789,42,7,99999", PT_BOUNCES="2", PT_SPP=str(SPP), PT_ARITH=arith)
    p = subprocess.run([exe, *args], cwd=d, env=env, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    pos = 0
    for token in EXPECTED_ORDER[variant]:
        k = p.stdout.find(token, pos)
        assert k >= 0, "stdout misses %r:\n%s" % (token, p.stdout)
        pos = k
    w, h = int(args[0]), int(args[1])
    o = poracle[arith]
    osc = o.load_scene_dir(d, variant)
    grid = None
    if variant == "grid":
        res, cell = o.grid_dims(osc["box_min"], osc["box_max"], osc["triangles"].shape[0], float(args[2]))
        grid = {"box_min": osc["box_min"], "box_max": osc["box_max"], "res": res, "cell_size": cell}
    ref = o.render_bounces(variant, w, h, (123456789, 42, 7, 99999), osc, 2, spp=SPP, grid=grid)
    assert ref["path_counters"]["bounce_rays"] > 0
    tmp = os.path.join(d, "oracle_expected.ppm")
    o.save_pam(tmp, ref["image"])
    assert open(os.path.join(d, "result.ppm"), "rb").read() == open(tmp, "rb").read()
