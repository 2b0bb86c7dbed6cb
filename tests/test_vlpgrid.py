"""VLP bounding box and VLP grid of CLSuperMetropolisPathTracer_vlpgrid — the parts of that program that are pure functions
of a VLP buffer: kernels reduceMinAndMax_lmem / reduceMinAndMax_lmem_nwg (metropolispathtracer.ocl:538-619), the host's grid
formula (CLSuperMetropolisPathTracer.c:628-636) and kernel initVLPsGrid (:621-647).
tests/golden/golden_vlpgrid.npz holds what the reference's OWN kernels (compiled through oracle/refrt, launched as its host
launches them) produce for four VLP buffers; make_golden.py is the generating script.  Bar: bit-exact box, identical cell
contents (as sorted sets: the reference appends with atomic_inc; its counter keeps counting past the 62 stored entries).

Also kernel pathTracer of that program (metropolispathtracer.ocl:649-684; its Sample :296-386 is the bidirectional one with the
gather restricted to the VLP-grid cell of the hit point): the golden file holds frames the reference's OWN kernel rendered from
two injected VPL buffers and their grids (lists in ascending light order).  Bar: the oracle reproduces those frames byte for
byte; CUDA (PT_VARIANT_VLPGRID through the C ABI) equals the oracle bit for bit — image, accumulation buffer, RNG states,
counters — under both arithmetic policies, and the reference's bytes under the `separate` policy."""
import hashlib
import os

import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import ROOT

GOLDEN = np.load(os.path.join(ROOT, "tests", "golden", "golden_vlpgrid.npz"))
NAMES = ("bidir", "synthetic", "few", "all_dummy")


def _golden_csr(name):
    nels, ids = GOLDEN[name + "_nels"], GOLDEN[name + "_ids"]
    n = np.minimum(nels, 62).astype(np.int64)
    start = np.concatenate([[0], np.cumsum(n)]).astype(np.uint32)
    refs = np.concatenate([ids[c, :n[c]] for c in range(len(n))] + [np.zeros(0, np.uint16)]).astype(np.uint32)
    return start, refs


@pytest.mark.parametrize("name", NAMES)
def test_oracle_vlp_bounds_and_grid_equal_the_reference_kernels(oracle_sep, name):
    vpl = GOLDEN[name + "_vpl"].view(np.float32)
    lo, hi = oracle_sep.vlp_bounds(vpl)
    assert np.array_equal(lo.view(np.uint32), GOLDEN[name + "_vmin"]) and np.array_equal(hi.view(np.uint32), GOLDEN[name + "_vmax"])
    if name == "all_dummy":
        assert lo[0] == np.finfo(np.float32).max and hi[0] == np.finfo(np.float32).tiny       # the reference's empty box
        return
    res, cell = oracle_sep.grid_dims(lo, hi, vpl.shape[0], 3.0)
    assert np.array_equal(res, GOLDEN[name + "_res"]) and np.array_equal(cell.view(np.uint32), GOLDEN[name + "_cell"])
    start, refs = oracle_sep.build_vlp_grid(vpl, lo, res, cell)
    gstart, grefs = _golden_csr(name)
    assert np.array_equal(start, gstart) and np.array_equal(refs, grefs)


def test_host_vlp_grid_dims_equal_the_oracle(oracle_sep):
    for name in NAMES[:3]:
        lo, hi = GOLDEN[name + "_vmin"].view(np.float32), GOLDEN[name + "_vmax"].view(np.float32)
        n = GOLDEN[name + "_vpl"].shape[0]
        for mod in (3.0, 0.5, 40.0):
            g = pt.vlp_grid_dims(lo, hi, n, mod)
            res, cell = oracle_sep.grid_dims(lo, hi, n, mod)
            assert list(g.res[:3]) == list(res[:3])
            assert np.array_equal(np.array(g.cell_size[:3], np.float32).view(np.uint32), cell[:3].view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_cuda_vlp_bounds_and_grid_equal_reference_and_oracle(renderer, oracle_sep, name):
    vpl = GOLDEN[name + "_vpl"].view(np.float32)
    renderer.set_vpls(vpl)
    lo, hi = renderer.vlp_bounds()
    assert np.array_equal(lo.view(np.uint32), GOLDEN[name + "_vmin"]) and np.array_equal(hi.view(np.uint32), GOLDEN[name + "_vmax"])
    if name == "all_dummy":
        return
    for mod in (3.0, 12.0):
        g = pt.vlp_grid_dims(lo, hi, vpl.shape[0], mod)
        renderer.build_vlp_grid(g)
        start, refs = renderer.read_vlp_grid_csr()
        ostart, orefs = oracle_sep.build_vlp_grid(vpl, lo, np.array(g.res[:]), np.array(g.cell_size[:], np.float32))
        assert np.array_equal(start, ostart) and np.array_equal(refs, orefs), (name, mod)
        if mod == 3.0:
            gstart, grefs = _golden_csr(name)
            assert np.array_equal(start, gstart) and np.array_equal(refs, grefs)
            cells = renderer.read_vlp_grid_cells()                       # the reference's 128-byte Cell layout
            nels = cells[:, :4].copy().view(np.uint32).reshape(-1)
            ids = cells[:, 4:].copy().view(np.uint16).reshape(-1, 62)
            assert np.array_equal(nels, np.minimum(GOLDEN[name + "_nels"], 62))
            for c in np.flatnonzero(nels)[:200]:
                assert np.array_equal(ids[c, :nels[c]], GOLDEN[name + "_ids"][c, :nels[c]])


@pytest.mark.gpu
def test_cuda_vlp_grid_on_the_light_tracers_own_buffer_and_at_scale(renderer, scene_dirs, oracle_sep):
    """pt_launch_lighttracer -> pt_vlp_bounds -> pt_build_vlp_grid without leaving the device, and a 60 000-light buffer
    (every cell overfull: the 62-entry cap and the ascending order)."""
    scene = pt.load_scene_dir(scene_dirs["bidir"], "bidir")
    renderer.set_scene(scene)
    renderer.light_tracer((1, 2, 3, 4), 512, arith="separate")
    vpl = renderer.read_vpls()
    lo, hi = renderer.vlp_bounds()
    olo, ohi = oracle_sep.vlp_bounds(vpl)
    assert np.array_equal(lo.view(np.uint32), olo.view(np.uint32)) and np.array_equal(hi.view(np.uint32), ohi.view(np.uint32))
    rng = np.random.default_rng(5)
    big = np.zeros((60000, 4), np.float32)
    big[:, :3] = rng.uniform(0, 40, (60000, 3))
    big[:, 3] = rng.uniform(0.0005, 0.01, 60000)
    big[::7, 3] = 0
    renderer.set_vpls(big)
    lo, hi = renderer.vlp_bounds()
    g = pt.vlp_grid_dims(lo, hi, big.shape[0], 0.05)
    renderer.build_vlp_grid(g)
    start, refs = renderer.read_vlp_grid_csr()
    ostart, orefs = oracle_sep.build_vlp_grid(big, lo, np.array(g.res[:]), np.array(g.cell_size[:], np.float32))
    assert np.array_equal(start, ostart) and np.array_equal(refs, orefs)
    assert np.diff(start.astype(np.int64)).max() == 62


# ---- kernel pathTracer of the vlpgrid program ---------------------------------------------------------------------------------
FRAME_W, FRAME_H = 256, 192
FRAME_ROWS = [40, 60, 80, 100, 130, 160, 191]
FRAME_SEEDS = [(1, 2, 3, 4), (123456789, 42, 7, 99999)]


def _golden_grid(name):
    return {"box_min": GOLDEN[name + "_vmin"].view(np.float32), "res": GOLDEN[name + "_res"], "cell_size": GOLDEN[name + "_cell"].view(np.float32),
            "csr": _golden_csr(name)}


@pytest.mark.parametrize("name", ["bidir", "synthetic"])
def test_oracle_vlpgrid_frames_equal_the_reference_kernel(oracle_sep, scene_dirs, name):
    sc = oracle_sep.load_scene_dir(scene_dirs["bidir"], "bidir")
    vpl = GOLDEN[name + "_vpl"].view(np.float32)
    for si, seeds in enumerate(FRAME_SEEDS):
        out = oracle_sep.render("vlpgrid", FRAME_W, FRAME_H, seeds, sc, vpls=vpl, grid=_golden_grid(name), want_accum=False, want_rng=False)
        assert np.array_equal(out["image"][FRAME_ROWS], GOLDEN["%s_frame_s%d_rows" % (name, si)]), (name, si)
        assert hashlib.sha256(out["image"].tobytes()).digest() == bytes(GOLDEN["%s_frame_s%d_sha256" % (name, si)]), (name, si)


def test_oracle_vlpgrid_builds_the_grid_the_reference_host_would(oracle_sep, scene_dirs):
    """grid=None: bounds of the buffer, the host's grid formula, initVLPsGrid — the same grid as the golden one, same frame rows"""
    sc = oracle_sep.load_scene_dir(scene_dirs["bidir"], "bidir")
    vpl = GOLDEN["synthetic_vpl"].view(np.float32)
    out = oracle_sep.render("vlpgrid", FRAME_W, FRAME_H, FRAME_SEEDS[0], sc, vpls=vpl, rows=(60, 61), want_accum=False, want_rng=False)
    assert np.array_equal(out["image"][60], GOLDEN["synthetic_frame_s0_rows"][1])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bidir", "synthetic"])
def test_cuda_vlpgrid_frames_equal_reference_and_oracle(renderer, oracle_sep, oracle_fma, scene_dirs, name):
    scene = pt.load_scene_dir(scene_dirs["bidir"], "bidir")
    renderer.set_scene(scene)
    vpl = GOLDEN[name + "_vpl"].view(np.float32)
    renderer.set_vpls(vpl)
    lo, hi = renderer.vlp_bounds()
    renderer.build_vlp_grid(pt.vlp_grid_dims(lo, hi, vpl.shape[0], 3.0))
    # the reference's own bytes (separate policy)
    for si, seeds in enumerate(FRAME_SEEDS):
        res = renderer.render("vlpgrid", FRAME_W, FRAME_H, seeds, arith="separate")
        assert np.array_equal(res.image[FRAME_ROWS], GOLDEN["%s_frame_s%d_rows" % (name, si)]), (name, si)
        assert hashlib.sha256(res.image.tobytes()).digest() == bytes(GOLDEN["%s_frame_s%d_sha256" % (name, si)]), (name, si)
    # the oracle, everything, both policies, at 512x512 on row windows (mesh + spheres, floor + shadows)
    W = H = 512
    for arith, o in (("fma", oracle_fma), ("separate", oracle_sep)):
        osc = o.load_scene_dir(scene_dirs["bidir"], "bidir")
        for rows in ((112, 144), (340, 372)):
            ref = o.render("vlpgrid", W, H, FRAME_SEEDS[0], osc, vpls=vpl, grid=_golden_grid(name), rows=rows)
            res = renderer.render("vlpgrid", W, H, FRAME_SEEDS[0], rows=rows, arith=arith, want_accum=True, want_rng=True)
            r0, r1 = rows
            assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), (name, arith, rows)
            assert np.array_equal(res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)), (name, arith, rows)
            assert np.array_equal(res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]), (name, arith, rows)
            for k in ("samples", "rays", "shadow_rays", "tri_tests", "prim_tests"):
                assert res.counters[k] == ref["counters"][k], (name, arith, rows, k)


@pytest.mark.gpu
def test_cuda_vlpgrid_needs_its_inputs_and_a_fresh_grid(scene_dirs):
    with pt.Renderer(device=0) as r:
        r.set_scene(pt.load_scene_dir(scene_dirs["bidir"], "bidir"))
        with pytest.raises(pt.PtError):
            r.render("vlpgrid", 64, 64, (1, 2, 3, 4))                     # no VPL buffer
        vpl = GOLDEN["few_vpl"].view(np.float32)
        r.set_vpls(vpl)
        with pytest.raises(pt.PtError):
            r.render("vlpgrid", 64, 64, (1, 2, 3, 4))                     # no VLP grid
        lo, hi = r.vlp_bounds()
        r.build_vlp_grid(pt.vlp_grid_dims(lo, hi, vpl.shape[0], 3.0))
        r.render("vlpgrid", 64, 64, (1, 2, 3, 4))
        r.set_vpls(vpl)                                                   # a new buffer invalidates the grid
        with pytest.raises(pt.PtError):
            r.render("vlpgrid", 64, 64, (1, 2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("nlights", [1, 5])
def test_cuda_vlpgrid_other_light_counts(renderer, scene_dirs, oracle_fma, nlights):
    """lightTracer -> VLP bounds -> VLP grid -> pathTracer, all on the device, with 1 and 5 lights (n_vlp VPLs per light)"""
    from test_bidir_gpu import same_floats
    from test_spec_kernel_gpu import FIVE_LIGHTS
    scene = pt.load_scene_dir(scene_dirs["bidir"], "bidir")
    scene.lights = FIVE_LIGHTS[:nlights]
    renderer.set_scene(scene)
    osc = oracle_fma.load_scene_dir(scene_dirs["bidir"], "bidir")
    osc["lights"] = scene.lights
    seeds, n = FRAME_SEEDS[1], 300
    renderer.light_tracer(seeds, n)
    vpl = renderer.read_vpls()
    ovpl = oracle_fma.light_tracer(seeds, osc, n)
    assert vpl.shape == (n * nlights, 4) and same_floats(vpl, ovpl)
    lo, hi = renderer.vlp_bounds()
    olo, ohi = oracle_fma.vlp_bounds(ovpl)
    assert np.array_equal(lo.view(np.uint32), olo.view(np.uint32)) and np.array_equal(hi.view(np.uint32), ohi.view(np.uint32))
    g = pt.vlp_grid_dims(lo, hi, vpl.shape[0], 3.0)
    renderer.build_vlp_grid(g)
    start, refs = renderer.read_vlp_grid_csr()
    ostart, orefs = oracle_fma.build_vlp_grid(ovpl, olo, np.array(g.res[:]), np.array(g.cell_size[:], np.float32))
    assert np.array_equal(start, ostart) and np.array_equal(refs, orefs)
    W = H = 512
    for rows in ((112, 144), (340, 372)):
        ref = oracle_fma.render("vlpgrid", W, H, seeds, osc, vpls=ovpl, rows=rows)        # grid=None: the reference host's grid
        res = renderer.render("vlpgrid", W, H, seeds, rows=rows, want_accum=True, want_rng=True)
        r0, r1 = rows
        assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), (nlights, rows)
        assert same_floats(res.accum[r0:r1], ref["accum"][r0:r1]), (nlights, rows)
        assert np.array_equal(res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]), (nlights, rows)
        for k in ("samples", "rays", "shadow_rays", "tri_tests", "prim_tests"):
            assert res.counters[k] == ref["counters"][k], (nlights, rows, k)
        assert ref["counters"]["shadow_rays"] > 0
