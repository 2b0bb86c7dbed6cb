"""The path oracle of the opt-in diffuse bounces (oracle_paths/, DESIGN.md 5b), on the CPU.

- With 0 bounces oracle_render_bounces is oracle_render: image, float buffer, RNG states and work counters, for base, lmem
  and grid under both arithmetic policies.
- The bounce direction is cosine-distributed: over the floor alone, a path straight down with one bounce sees the sky, whose
  colour (0.7, 0.6, 1) (1 - cos)^4 has the mean 1/15 under cosine weighting, times the floor's albedo.
- Russian roulette is unbiased: between the floor and the underside of a square, eight bounces with and without it have the
  same mean.
"""
import numpy as np
import pytest

from conftest import SEED_SETS

W = H = 512
ROWS = (112, 128)           # mesh, sky, spheres
ROWS2 = (352, 360)          # floor, spheres, shadows


@pytest.fixture(scope="module", params=[0, 1], ids=["separate", "fma"])
def paths(request):
    from oracle.pyoracle import cpu_has_fma
    from oracle_paths.pypaths import PathOracle
    if request.param and not cpu_has_fma():
        pytest.skip("host CPU lacks FMA")
    return PathOracle(contract=request.param)


def empty_scene(lights=()):
    return {"spheres": np.zeros(9, np.int32), "squares": np.zeros(9, np.int32), "triangles": np.zeros((0, 12), np.float32),
            "lights": np.asarray(lights, np.float32).reshape(-1, 4)}


def rng_states(n, seed):
    r = np.random.default_rng(seed)
    return r.integers(0, 2 ** 32, size=(n, 4), dtype=np.uint64).astype(np.uint32)


@pytest.mark.parametrize("variant", ["base", "lmem", "grid"])
@pytest.mark.parametrize("rows", [ROWS, ROWS2], ids=["mesh", "floor"])
def test_zero_bounces_is_oracle_render(paths, scene_dirs, variant, rows):
    scene = paths.load_scene_dir(scene_dirs[variant], variant)
    grid = None
    if variant == "grid":
        res, cell = paths.grid_dims(scene["box_min"], scene["box_max"], scene["triangles"].shape[0])
        grid = {"box_min": scene["box_min"], "box_max": scene["box_max"], "res": res, "cell_size": cell}
    ref = paths.render(variant, W, H, SEED_SETS[0], scene, spp=4, rows=rows, grid=grid)
    out = paths.render_bounces(variant, W, H, SEED_SETS[0], scene, 0, spp=4, rows=rows, grid=grid)
    assert np.array_equal(out["image"], ref["image"])
    assert np.array_equal(out["accum"].view(np.uint32), ref["accum"].view(np.uint32))
    assert np.array_equal(out["rng_state"], ref["rng_state"])
    assert out["counters"] == ref["counters"]
    assert out["path_counters"] == {"bounce_rays": 0, "rr_terminations": 0, "tmin_rejections": 0, "disk_exhausted": 0}


@pytest.mark.parametrize("variant", ["base", "lmem", "grid"])
def test_bounces_add_light_and_rays(paths, scene_dirs, variant):
    """B = 2 on the floor rows: the same camera samples, more rays, brighter or equal pixels (the indirect term is >= 0), and
    the bounce-ray count is rays - samples - shadow rays."""
    scene = paths.load_scene_dir(scene_dirs[variant], variant)
    grid = None
    if variant == "grid":
        res, cell = paths.grid_dims(scene["box_min"], scene["box_max"], scene["triangles"].shape[0])
        grid = {"box_min": scene["box_min"], "box_max": scene["box_max"], "res": res, "cell_size": cell}
    b0 = paths.render_bounces(variant, W, H, SEED_SETS[0], scene, 0, spp=4, rows=ROWS2, grid=grid)
    b2 = paths.render_bounces(variant, W, H, SEED_SETS[0], scene, 2, spp=4, rows=ROWS2, grid=grid)
    c0, c2 = b0["counters"], b2["counters"]
    assert c2["samples"] == c0["samples"]
    pc = b2["path_counters"]
    assert pc["bounce_rays"] > 0 and c2["rays"] - c2["samples"] - c2["shadow_rays"] == pc["bounce_rays"]
    assert pc["rr_terminations"] > 0
    assert pc["disk_exhausted"] == 0
    assert not np.array_equal(b2["image"], b0["image"])
    # floor albedo and the clamp keep c >= 0; the RNG streams differ after the first bounce, so compare the frame mean
    assert b2["accum"][ROWS2[0]:ROWS2[1], :, :3].mean() > b0["accum"][ROWS2[0]:ROWS2[1], :, :3].mean()


def test_cosine_sampling_closed_form(paths):
    """Floor only, no lights: the camera vertex is black, the bounce sees the sky.  E[(1 - cos)^4] = 2 int (1-u)^4 u du = 1/15."""
    n = 1_000_000
    st = rng_states(n, 11)
    L, pc = paths.path_samples(empty_scene(), (2.5, 2.5, 3.0), (0.0, 0.0, -1.0), st, bounces=1)
    assert pc["bounce_rays"] == n and pc["disk_exhausted"] == 0
    rho_even = 0.75                                  # X = (2.5, 2.5, 0): ceil(0.5) + ceil(0.5) = 2, an even cell
    want = rho_even * np.array([0.7, 0.6, 1.0]) / 15.0
    mean = L.astype(np.float64).mean(axis=0)
    se = L.astype(np.float64).std(axis=0, ddof=1) / np.sqrt(n)
    assert np.all(np.abs(mean - want) < 5 * se), (mean, want, se)
    assert np.all(se < 0.01 * want)                  # the check has teeth: 5 se is under 5 % of the value


def test_russian_roulette_is_unbiased(paths):
    """Between the floor and a square at z = 4 (x in [1, 3], |y| < 1) lit from the side: paths start under the square,
    looking up at it, with 8 bounces, roulette on and off.  The two means agree within 5 standard errors of their
    difference; roulette did end paths.  (Looking down, the camera ray would hit the square BEHIND its origin: the
    reference's square test has no lower bound.)"""
    scene = empty_scene([[6.0, 0.0, 3.0, 40.0]])
    scene["squares"][0] = 1 << 2
    n = 400_000
    o, d = (2.0, 0.0, 2.0), (0.0, 0.0, 1.0)
    on, pc_on = paths.path_samples(scene, o, d, rng_states(n, 21), bounces=8, rr=True)
    off, pc_off = paths.path_samples(scene, o, d, rng_states(n, 22), bounces=8, rr=False)
    assert pc_on["rr_terminations"] > 0 and pc_off["rr_terminations"] == 0
    assert pc_on["tmin_rejections"] > 0                 # bounces off the square re-meet it at r ~ 0
    assert pc_on["bounce_rays"] < pc_off["bounce_rays"]
    a, b = on.astype(np.float64), off.astype(np.float64)
    diff = a.mean(axis=0) - b.mean(axis=0)
    se = np.sqrt(a.var(axis=0, ddof=1) / n + b.var(axis=0, ddof=1) / n)
    assert np.all(np.abs(diff) < 5 * se), (diff, se)
    assert np.all(b.mean(axis=0) > 0.0)
    assert np.all(se < 0.02 * b.mean(axis=0))           # tight enough to see a bias of a few per cent


def test_single_path_entry_point_matches_batch(paths):
    """oracle_path_sample (one path) and oracle_path_samples (a batch) are the same function."""
    import ctypes as C
    from oracle.pyoracle import oracle_counters
    from oracle_paths.pypaths import oracle_path_counters
    scene = empty_scene([[6.0, 0.0, 3.0, 40.0]])
    scene["squares"][0] = 1 << 2
    st = rng_states(64, 5)
    batch, _ = paths.path_samples(scene, (2.0, 0.0, 2.0), (0.0, 0.0, -1.0), st.copy(), bounces=5)
    J, keep = paths._path_job("base", scene)
    o = np.array([2.0, 0.0, 2.0], np.float32)
    d = np.array([0.0, 0.0, -1.0], np.float32)
    for k in range(st.shape[0]):
        s = st[k].copy()
        rgb = np.zeros(3, np.float32)
        cnt, pc = oracle_counters(), oracle_path_counters()
        assert paths.plib.oracle_path_sample(C.byref(J), o.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                                             s.ctypes.data_as(C.c_void_p), 5, 1, rgb.ctypes.data_as(C.c_void_p), C.byref(cnt),
                                             C.byref(pc)) == 0
        assert np.array_equal(rgb.view(np.uint32), batch[k].view(np.uint32))
        assert cnt.samples == 1 and cnt.rays == 1 + cnt.shadow_rays + pc.bounce_rays
    del keep


def test_refusals(paths, scene_dirs):
    scene = paths.load_scene_dir(scene_dirs["base"], "base")
    for variant in ("nodof",):
        with pytest.raises((ValueError, KeyError)):
            paths.render_bounces(variant, W, H, SEED_SETS[0], scene, 1, spp=64, rows=ROWS)
    for b in (-1, 16):
        with pytest.raises(ValueError):
            paths.render_bounces("base", W, H, SEED_SETS[0], scene, b, spp=4, rows=ROWS)
