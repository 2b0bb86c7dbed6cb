"""Sample-range sharding ("throughput mode", SURVEY.md 8e): pt_render_params.sample_block / sample_blocks.
Each block is bit-exact against the oracle's statement of the same definition; the SUM of the blocks is the frame and
agrees with the unsharded reference render statistically (different RNG streams), block 0 IS the reference stream."""
import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import SEED_SETS
from test_spec_kernel_gpu import FIVE_LIGHTS

pytestmark = pytest.mark.gpu
W = H = 512
ROWS = (340, 356)


def _setup(renderer, scene_dirs, o, variant):
    d = scene_dirs[variant]
    scene = pt.load_scene_dir(d, variant)
    renderer.set_scene(scene)
    if variant == "grid":
        renderer.build_grid(pt.grid_dims(scene))
    extra = {}
    if variant == "bidir":
        renderer.light_tracer(SEED_SETS[0], 512)
        extra["vpls"] = renderer.read_vpls()
    return o.load_scene_dir(d, variant), extra


@pytest.mark.parametrize("variant,kernels", [("base", ("mega", "persistent", "wavefront", "spec")), ("lmem", ("mega", "persistent", "spec")),
                                             ("grid", ("mega", "persistent", "wavefront", "grid_tma", "grid_stream", "grid_pool", "grid_queue",
                                                       "grid_async")),
                                             ("bidir", ("mega",))])
def test_blocks_bit_exact_and_sum_to_the_frame(renderer, scene_dirs, oracle_fma, variant, kernels):
    osc, extra = _setup(renderer, scene_dirs, oracle_fma, variant)
    R = 4
    r0, r1 = ROWS
    total = np.zeros((r1 - r0, W, 4), np.float32)
    for b in range(R):
        ref = oracle_fma.render(variant, W, H, SEED_SETS[0], osc, rows=ROWS, sample_block=b, sample_blocks=R, **extra)
        for k in kernels:
            res = renderer.render(variant, W, H, SEED_SETS[0], rows=ROWS, kernel=k, sample_block=b, sample_blocks=R, want_accum=True, want_rng=True)
            assert np.array_equal(res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)), (variant, k, b)
            assert np.array_equal(res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]), (variant, k, b)
            assert res.counters["samples"] == ref["counters"]["samples"] == (r1 - r0) * W * 64 // R
        total += ref["accum"][r0:r1]
        assert (ref["accum"][r0:r1, :, 3] == (255.0 if b == 0 else 0.0)).all()
    # the blocks' sum is a frame: alpha 255, and statistically the same picture as the unsharded render
    full = oracle_fma.render(variant, W, H, SEED_SETS[0], osc, rows=ROWS, **extra)["accum"][r0:r1]
    assert (total[..., 3] == 255.0).all()
    a, f = np.clip(np.trunc(total[..., :3]), 0, 255), np.clip(np.trunc(full[..., :3]), 0, 255)
    diff = a - f
    assert abs(diff.mean()) < 0.35, diff.mean()                    # no bias: only Monte-Carlo noise of other streams
    assert np.sqrt((diff ** 2).mean()) < 14.0, np.sqrt((diff ** 2).mean())
    # block 0 is the reference's own stream: after its 16 samples the RNG is where a 16-spp reference render ends
    b0 = renderer.render(variant, W, H, SEED_SETS[0], rows=ROWS, sample_block=0, sample_blocks=R, want_rng=True)
    short = oracle_fma.render(variant, W, H, SEED_SETS[0], osc, rows=ROWS, spp=16, **extra)
    assert np.array_equal(b0.rng_state.reshape(H, W, 4)[r0:r1], short["rng_state"].reshape(H, W, 4)[r0:r1])


@pytest.mark.parametrize("nlights", [1, 5])
def test_blocks_at_other_light_counts(renderer, scene_dirs, oracle_fma, nlights):
    """Blocks b > 0 (own seeds, no bias 13) with an odd light count: a hit sample draws 2 + nlights pairs"""
    lights = FIVE_LIGHTS[:nlights]
    R = 4
    r0, r1 = ROWS
    for variant, kernels in (("base", ("mega", "spec")), ("lmem", ("spec", "wavefront")), ("grid", ("mega", "grid_queue", "grid_async"))):
        d = scene_dirs[variant]
        scene = pt.load_scene_dir(d, variant)
        scene.lights = lights
        renderer.set_scene(scene)
        if variant == "grid":
            renderer.build_grid(pt.grid_dims(scene))
        osc = oracle_fma.load_scene_dir(d, variant)
        osc["lights"] = lights
        for b in range(R):
            ref = oracle_fma.render(variant, W, H, SEED_SETS[0], osc, rows=ROWS, sample_block=b, sample_blocks=R)
            assert ref["counters"]["shadow_rays"] > 0
            for k in kernels:
                res = renderer.render(variant, W, H, SEED_SETS[0], rows=ROWS, kernel=k, sample_block=b, sample_blocks=R, want_accum=True, want_rng=True)
                what = (variant, nlights, k, b)
                assert np.array_equal(res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)), what
                assert np.array_equal(res.rng_state.reshape(H, W, 4)[r0:r1], ref["rng_state"].reshape(H, W, 4)[r0:r1]), what
                assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), what
                for c in ("samples", "rays", "shadow_rays"):
                    assert res.counters[c] == ref["counters"][c], what + (c,)


def test_sample_sharding_errors(renderer, scene_dirs):
    renderer.set_scene(pt.load_scene_dir(scene_dirs["nodof"], "nodof"))
    with pytest.raises(pt.PtError, match="NoDoF"):
        renderer.render("nodof", 64, 64, SEED_SETS[0], sample_block=0, sample_blocks=2)
    renderer.set_scene(pt.load_scene_dir(scene_dirs["lmem"], "lmem"))
    with pytest.raises(pt.PtError, match="multiple"):
        renderer.render("lmem", 64, 64, SEED_SETS[0], sample_block=0, sample_blocks=3)
    with pytest.raises(pt.PtError, match="outside"):
        renderer.render("lmem", 64, 64, SEED_SETS[0], sample_block=2, sample_blocks=2)
    one = renderer.render("lmem", 64, 64, SEED_SETS[0], want_accum=True)
    same = renderer.render("lmem", 64, 64, SEED_SETS[0], sample_block=0, sample_blocks=1, want_accum=True)
    assert np.array_equal(one.accum.view(np.uint32), same.accum.view(np.uint32))
