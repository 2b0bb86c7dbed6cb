"""Progressive rendering (include/ptcuda.h, pt_launch_pathtracer_range / pt_set_render_state): a frame rendered as a chain
of sample ranges, each continuing from the state the previous range left or from a saved checkpoint, equals the frame of
one launch bit for bit — image bytes, accumulation buffer (as uint32) and the RNG state of every pixel — and the ranges'
work counters add up to the one launch's."""
import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import SEED_SETS
from test_vlpgrid import GOLDEN, _golden_grid

pytestmark = pytest.mark.gpu

W = H = 512
ROWS = (112, 144)                       # mesh, spheres, floor and sky of the default view
SEEDS = SEED_SETS[1]
PLANS = [[64], [1, 63], [16] * 4, [5, 27, 32], [1] * 64]
SUMMED = ("samples", "rays", "shadow_rays", "tri_tests", "cells_visited", "prim_tests", "vpl_evals")
# scene -> (variant, kernels)
SCENES = {"base": ("base", ("auto", "mega", "spec")), "lmem": ("lmem", ("auto", "mega", "spec")), "torus": ("base", ("auto", "mega")),
          "grid": ("grid", ("auto", "mega")), "gridsoup": ("grid", ("auto", "mega")), "bidir": ("bidir", ("auto", "mega")),
          "vlpgrid": ("vlpgrid", ("auto", "mega"))}


def soup_scene(scene_dirs):
    """20 000 triangles (> 16 384: the big-grid megakernel) around the eye"""
    import gen_mesh
    s = pt.load_scene_dir(scene_dirs["grid"], "grid")
    tris = gen_mesh.soup(20000, seed=9, box_size=20.0)
    lo, hi = gen_mesh.bbox_like_reference(tris)
    return pt.Scene(s.spheres, s.squares, tris, s.lights, lo, hi)


def setup(r, scene_dirs, name, arith="fma"):
    """puts scene `name` (with its grid, VPL buffer, VLP grid) into Renderer r; -> variant"""
    variant = SCENES[name][0]
    if name == "gridsoup":
        scene = soup_scene(scene_dirs)
    else:
        scene = pt.load_scene_dir(scene_dirs["bidir" if variant in ("bidir", "vlpgrid") else name], variant)
    r.set_scene(scene)
    if variant == "grid":
        r.build_grid(pt.grid_dims(scene))
    if variant == "bidir":
        r.light_tracer(SEEDS, 512, arith=arith)
    if variant == "vlpgrid":
        vpl = GOLDEN["bidir_vpl"].view(np.float32)
        r.set_vpls(vpl)
        lo, hi = r.vlp_bounds()
        r.build_vlp_grid(pt.vlp_grid_dims(lo, hi, vpl.shape[0], 3.0))
    return variant


def one_launch(r, variant, w=W, h=H, **kw):
    return r.render(variant, w, h, SEEDS, want_accum=True, want_rng=True, **kw)


def progress(r, variant, plan, w=W, h=H, per_range=None, **kw):
    """renders the frame in ranges of the lengths in `plan` (per_range[k]: extra keywords of range k); -> (result of the
    last range, the ranges' counters summed)"""
    spp = kw.get("spp", 64)
    assert sum(plan) == spp
    total = dict.fromkeys(SUMMED + ("tri_tests_executed",), 0)
    b = 0
    for k, n in enumerate(plan):
        last = b + n == spp
        extra = dict(kw, **(per_range[k] if per_range else {}))
        out = r.render(variant, w, h, SEEDS, samples=(b, b + n), read_image=last, want_accum=last, want_rng=last, **extra)
        for c in total:
            total[c] += out.counters[c]
        b += n
    return out, total


def assert_same(got, ref, what):
    assert np.array_equal(got.image, ref.image), what
    assert np.array_equal(got.accum.view(np.uint32), ref.accum.view(np.uint32)), what
    assert np.array_equal(got.rng_state, ref.rng_state), what


def assert_same_rows(got, ref, rows, what):
    r0, r1 = rows
    w = got.image.shape[1]
    assert np.array_equal(got.image[r0:r1], ref["image"][r0:r1]), what
    assert np.array_equal(got.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)), what
    assert np.array_equal(got.rng_state.reshape(-1, w, 4)[r0:r1], ref["rng_state"].reshape(-1, w, 4)[r0:r1]), what


def oracle_frame(o, scene_dirs, name, variant, rows):
    osc = o.load_scene_dir(scene_dirs["bidir" if variant in ("bidir", "vlpgrid") else name], variant)
    if variant == "vlpgrid":
        return o.render("vlpgrid", W, H, SEEDS, osc, vpls=GOLDEN["bidir_vpl"].view(np.float32), grid=_golden_grid("bidir"), rows=rows)
    return o.render(variant, W, H, SEEDS, osc, rows=rows)          # bidir: the oracle runs the light tracer with SEEDS


# ---------------------------------------------------------------------------------------------------- 1. ranges = one launch
@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("name", list(SCENES))
def test_ranges_equal_one_launch(renderer, scene_dirs, oracle_fma, oracle_sep, name, arith):
    variant = setup(renderer, scene_dirs, name, arith)
    for k in SCENES[name][1]:
        kw = dict(rows=ROWS, arith=arith, kernel=k)
        ref = one_launch(renderer, variant, **kw)
        exact_work = renderer.last_kernel() == "mega"       # SPEC also counts the tests of discarded speculation
        for plan in PLANS:
            got, total = progress(renderer, variant, plan, **kw)
            what = (name, arith, k, plan)
            assert_same(got, ref, what)
            for c in SUMMED + (("tri_tests_executed",) if exact_work else ()):
                assert total[c] == ref.counters[c], what + (c,)
            if k == "auto" and plan == [5, 27, 32] and name != "gridsoup":
                assert_same_rows(got, oracle_frame(oracle_fma if arith == "fma" else oracle_sep, scene_dirs, name, variant, ROWS), ROWS, what)


# ------------------------------------------------------------------------------------------ 2. the scale is the frame's
def test_scale_is_fixed_by_the_total(renderer, scene_dirs):
    setup(renderer, scene_dirs, "base")
    ref = one_launch(renderer, "base", rows=ROWS, spp=256)
    got, _ = progress(renderer, "base", [100, 156], rows=ROWS, spp=256)
    assert_same(got, ref, "256 spp in [100, 156]")


# ---------------------------------------------------------------------------------- 3. brute force, per-cluster culling
@pytest.mark.parametrize("name", ["base", "lmem"])
def test_cluster_cull_instantiation(renderer, scene_dirs, name):
    variant = setup(renderer, scene_dirs, name)
    for k in ("mega", "spec"):
        kw = dict(rows=ROWS, kernel=k, cluster_cull="on")
        ref = one_launch(renderer, variant, **kw)
        for plan in ([1, 63], [16] * 4):
            got, _ = progress(renderer, variant, plan, **kw)
            assert_same(got, ref, (name, k, plan))


# ------------------------------------------------------------------------------- 4. big-grid tile order across ranges
def test_tile_order_records_then_sorts(renderer, scene_dirs):
    """1280x720: 7200 tiles (> 148 x 16), ranges of >= 16 samples: the first range records the CTA times, the second runs
    in the sorted order"""
    setup(renderer, scene_dirs, "gridsoup")
    ref = one_launch(renderer, "grid", w=1280, h=720)
    with pt.Renderer(device=0) as fresh:
        setup(fresh, scene_dirs, "gridsoup")
        got, total = progress(fresh, "grid", [16, 16, 32], w=1280, h=720)
    assert_same(got, ref, "tile order")
    for c in SUMMED:
        assert total[c] == ref.counters[c], c


# ------------------------------------------------------------------------------------------------- 5. rows and stripes
@pytest.mark.parametrize("name", ["base", "grid"])
def test_rows_and_stripes(renderer, scene_dirs, name):
    variant = setup(renderer, scene_dirs, name)
    for kw in (dict(rows=(112, 144)), dict(interleave=8, rank=1, nranks=3)):
        ref = one_launch(renderer, variant, **kw)
        got, _ = progress(renderer, variant, [16, 5, 43], **kw)
        assert_same(got, ref, (name, kw))


# -------------------------------------------------------------------------------------- 6. flavours switch between ranges
def test_switching_flavours_between_ranges(renderer, scene_dirs):
    setup(renderer, scene_dirs, "base")
    ref = one_launch(renderer, "base", rows=ROWS)
    got, _ = progress(renderer, "base", [16, 32, 16], rows=ROWS,
                      per_range=[dict(kernel="spec"), dict(kernel="mega"), dict(kernel="mega", dead_rays="elide")])
    assert_same(got, ref, "spec, mega, mega with dead rays elided")


# --------------------------------------------------------------------------------------------------------- 7. checkpoint
@pytest.mark.parametrize("name", ["base", "grid", "bidir"])
def test_checkpoint_and_resume_in_another_context(renderer, scene_dirs, name):
    variant = setup(renderer, scene_dirs, name)
    ref = one_launch(renderer, variant, rows=ROWS)
    with pt.Renderer(device=0) as r1:
        setup(r1, scene_dirs, name)
        cp = r1.render(variant, W, H, SEEDS, samples=(0, 24), rows=ROWS, want_accum=True, want_rng=True)
    with pt.Renderer(device=0) as r2:
        setup(r2, scene_dirs, name)
        r2.set_render_state(variant, W, H, SEEDS, 24, cp.accum, cp.rng_state, rows=ROWS)
        got = r2.render(variant, W, H, SEEDS, samples=(24, 64), rows=ROWS, want_accum=True, want_rng=True)
    assert_same(got, ref, name)


# ------------------------------------------------------------------------------------------------------------ 8. preview
def preview(accum, spp, end):
    f = np.float32(spp) / np.float32(end)
    v = ((accum[..., :3] - np.float32(13.0)) * f) + np.float32(13.0)          # float32, every operation rounded
    rgb = np.clip(np.trunc(v), 0, 255).astype(np.uint8)
    return np.concatenate([rgb, np.full(rgb.shape[:-1] + (1,), 255, np.uint8)], axis=-1)


def test_preview_image(renderer, scene_dirs):
    setup(renderer, scene_dirs, "base")
    r0, r1 = ROWS
    for b, e in ((0, 16), (16, 21)):                          # f = 4, and 64 / 21 (inexact)
        out = renderer.render("base", W, H, SEEDS, samples=(b, e), rows=ROWS, want_accum=True)
        assert np.array_equal(out.image[r0:r1], preview(out.accum[r0:r1], 64, e)), (b, e)


# ----------------------------------------------------------------------------------------------------------- 9. refusals
def test_refusals_leave_the_progression_intact(renderer, scene_dirs):
    w = h = 64
    with pt.Renderer(device=0) as r:
        setup(r, scene_dirs, "base")

        def rng(b, e, variant="base", width=w, seeds=SEEDS, **kw):
            return r.render(variant, width, h, seeds, samples=(b, e), **kw)

        with pytest.raises(pt.PtError, match="continues no progression"):
            rng(16, 32)                                              # fresh context
        rng(0, 16)
        for b, e in ((8, 32), (20, 32), (16, 65), (16, 16), (16, 10), (-1, 8)):
            with pytest.raises(pt.PtError):
                rng(b, e)
        for kw in (dict(seeds=SEED_SETS[0]), dict(spp=128), dict(width=65), dict(arith="separate"), dict(rows=(0, 32))):
            with pytest.raises(pt.PtError, match="differ"):
                rng(16, 32, **kw)
        saved = r.cam
        r.cam = pt.camera()
        r.cam.eye_offset[0] += 0.5
        with pytest.raises(pt.PtError, match="differ"):
            rng(16, 32)
        r.cam = saved
        with pytest.raises(pt.PtError, match="NoDoF"):
            rng(0, 16, variant="nodof")
        with pytest.raises(pt.PtError, match="sample_blocks"):
            rng(0, 16, sample_block=0, sample_blocks=2)
        for k in ("persistent", "wavefront"):
            with pytest.raises(pt.PtError, match="MEGA, SPEC and AUTO"):
                rng(16, 32, kernel=k)
        rng(16, 32)                                                  # still continues after every refusal
        r.render("base", w, h, SEEDS)                                # a plain render ends the progression
        with pytest.raises(pt.PtError, match="continues no progression"):
            rng(32, 48)
        rng(0, 32)
        setup(r, scene_dirs, "base")                                 # pt_set_scene between ranges
        with pytest.raises(pt.PtError, match="differ"):
            rng(32, 48)

        setup(r, scene_dirs, "grid")
        rng(0, 16, variant="grid")
        for k in ("persistent", "wavefront", "grid_tma", "grid_stream", "grid_pool", "grid_queue", "grid_async"):
            with pytest.raises(pt.PtError, match="MEGA, SPEC and AUTO"):
                rng(16, 32, variant="grid", kernel=k)
        rng(16, 32, variant="grid")
        r.build_grid(pt.grid_dims(pt.load_scene_dir(scene_dirs["grid"], "grid")))   # pt_build_grid between ranges
        with pytest.raises(pt.PtError, match="differ"):
            rng(32, 48, variant="grid")

        setup(r, scene_dirs, "bidir")
        rng(0, 16, variant="bidir")
        r.set_vpls(r.read_vpls())                                    # pt_set_vpls between ranges (same contents)
        with pytest.raises(pt.PtError, match="differ"):
            rng(16, 32, variant="bidir")
        rng(0, 16, variant="bidir")
        got = rng(16, 64, variant="bidir", want_accum=True, want_rng=True)
        assert_same(got, r.render("bidir", w, h, SEEDS, want_accum=True, want_rng=True), "bidir after the refusals")
        with pytest.raises(pt.PtError):
            r.set_render_state("bidir", w, h, SEEDS, 64, got.accum, got.rng_state)     # samples_done must be < spp
