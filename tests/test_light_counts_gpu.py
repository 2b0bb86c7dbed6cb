"""Every kernel flavour at 0, 1, 3, 4 and 5 lights, against the CPU oracle (bit-exact).

The light count decides how many RNG pairs a sample draws once its camera ray hits (2 + nlights, drawn before any skip,
base:168) and how long its shadow-ray part is, and every flavour restates that per-light logic in its own code: SPEC's
heavy pass places its lanes on the stream with it (odd counts: candidates one pair apart, pt_spec.cuh), the persistent /
grid_stream / grid_pool state machines, the wavefront's one queue generation per light, the light loops of grid_tma,
grid_queue and grid_async, the megakernels (brute force, cluster-culled, big grid) and the dead-ray elision, which skips
nlights pairs.  The light sets are prefixes of the five lights the oracle is pinned to the reference with
(test_oracle_vs_ref.py): a zero-intensity light (base skips it after drawing its pair, lmem and grid trace it), a light
at z = 3 below the squares (the lam < 0 no-ray branch), plus a set with a light just above the mesh, inside its bounding
sphere and over the grid box, so floor pixels' shadow rays scan the triangles.

Bar: image bytes, float accumulation buffer, final RNG state of every work-item and the work counters equal the
oracle's for every flavour; with dead_rays="elide" the same bits and samples with fewer shadow rays."""
import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import SEED_SETS
from test_spec_kernel_gpu import COUNTERS, FIVE_LIGHTS as LIGHTS5

pytestmark = pytest.mark.gpu

W = H = 512
SEEDS = SEED_SETS[0]
# (7.5, 4.5, 11.8): 0.25 above the default mesh's box (z <= 11.548), 1.3 from its centre (7.5, 4.45, 10.5)
NEAR_MESH = np.array([[7.5, 4.5, 11.8, 150], [10, 4, 10, 200], [15, 2, 7, 0]], np.float32)
LIGHT_SETS = {"0": LIGHTS5[:0], "1": LIGHTS5[:1], "3": LIGHTS5[:3], "4": LIGHTS5[:4], "5": LIGHTS5, "near-mesh": NEAR_MESH}

GRID_COUNTERS = ("samples", "rays", "shadow_rays", "cells_visited", "tri_tests")
GRID_KERNELS = ("mega", "persistent", "wavefront", "grid_tma", "grid_stream", "grid_pool", "grid_queue", "grid_async")
BRUTE = (("mega", {"scene_mem": "smem"}), ("mega", {"scene_mem": "const"}), ("spec", {}), ("persistent", {}), ("wavefront", {}))
ELIDING = ("mega", "spec", "grid_queue", "grid_async")            # the flavours that honour dead_rays="elide"

# case: (variant, scene, flavours as (kernel, extra render keywords))
CASES = {
    "base": ("base", "default", BRUTE),
    "lmem": ("lmem", "default", BRUTE),
    "base-silhouette": ("base", "silhouette", (("spec", {}), ("mega", {}))),
    "lmem-silhouette": ("lmem", "silhouette", (("spec", {}), ("mega", {}))),
    "base-cluster-cull": ("base", "default", (("mega", {"cluster_cull": "on"}), ("spec", {"cluster_cull": "on"}))),
    "nodof": ("nodof", "default", (("mega", {}), ("persistent", {}), ("wavefront", {}))),
    "grid": ("grid", "default", tuple((k, {}) for k in GRID_KERNELS)),
    "grid-soup": ("grid", "soup", (("mega", {}), ("grid_queue", {}))),
}
# row windows: mesh, sky, spheres and squares / floor, spheres and shadows
WINDOWS = {"default": ((112, 144), (340, 372)), "silhouette": ((140, 172), (340, 372)), "soup": ((250, 266), (420, 436))}


def silhouette_triangles():
    """400 sparse triangles in front of the camera and above its height: sky behind them, so along their edges hit and
    sky samples alternate inside one pixel (SPEC mispredicts and switches to window mode); rows 0-196 of the frame."""
    import gen_mesh
    tris = gen_mesh.soup(400, seed=3, box_lo=8.0, box_size=6.0, edge=(0.5, 0.9))
    tris[:, [0, 4, 8]] += 1.8
    tris[:, [1, 5, 9]] -= 6.2
    tris[:, [2, 6, 10]] += 1.0
    return tris


def soup_triangles():
    """20 000 triangles: above the 16 384 at which the grid megakernel switches to its big-grid instantiation"""
    import gen_mesh
    return gen_mesh.soup(20000, seed=11, box_size=24.0)


def build_scene(scene_dirs, variant, scene, lights):
    """-> (pt.Scene, oracle scene dict) of `scene` with `lights` in place of the scene files' two"""
    if scene == "default":
        s = pt.load_scene_dir(scene_dirs[variant], variant)
    else:
        import gen_mesh
        tris = silhouette_triangles() if scene == "silhouette" else soup_triangles()
        lo, hi = gen_mesh.bbox_like_reference(tris)
        z = np.zeros(9, np.int32)
        sph = z if scene == "silhouette" else np.array([1024, 0, 0, 0, 145, 0, 0, 2048, 0], np.int32)
        sq = z if scene == "silhouette" else np.array([4096, 0, 0, 0, 0, 0, 129, 0, 8192], np.int32)
        s = pt.Scene(sph, sq, tris, lights, lo, hi)
    s.lights = np.ascontiguousarray(lights, np.float32).reshape(-1, 4)
    osc = {"spheres": s.spheres, "squares": s.squares, "triangles": s.triangles, "lights": s.lights, "box_min": s.box_min,
           "box_max": s.box_max}
    return s, osc


def set_scene(renderer, variant, s):
    renderer.set_scene(s)
    if variant == "grid":
        renderer.build_grid(pt.grid_dims(s))


@pytest.fixture(scope="module")
def oracle_frames():
    """oracle renders, one per (variant, scene, light set, policy, window): shared by the cases and legs that need them"""
    return {}


def oracle_window(cache, o, variant, scene, lset, osc, rows):
    key = (variant, scene, lset, o.contract, rows)
    if key not in cache:
        cache[key] = o.render(variant, W, H, SEEDS, osc, rows=rows)
    return cache[key]


def rng_rows(st, variant, rows):
    r0, r1 = rows
    if variant == "nodof":                                       # 8 x 8 work-items per pixel
        return st.reshape(8 * H, 8 * W, 4)[8 * r0:8 * r1]
    return st.reshape(H, W, 4)[r0:r1]


def same_bits(res, ref, variant, rows, what):
    r0, r1 = rows
    a, b = rng_rows(res.rng_state, variant, rows), rng_rows(ref["rng_state"], variant, rows)
    assert np.array_equal(a, b), "%s: RNG state differs in %d work-items" % (what, int((a != b).any(axis=-1).sum()))
    a, b = res.accum[r0:r1].view(np.uint32), ref["accum"][r0:r1].view(np.uint32)
    assert np.array_equal(a, b), "%s: accumulation differs in %d pixels" % (what, int((a != b).any(axis=2).sum()))
    assert np.array_equal(res.image[r0:r1], ref["image"][r0:r1]), "%s: image bytes" % what


@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("lset", list(LIGHT_SETS))
@pytest.mark.parametrize("case", list(CASES))
def test_light_counts_bit_exact(renderer, scene_dirs, oracle_fma, oracle_sep, oracle_frames, case, lset, arith):
    variant, scene, flavours = CASES[case]
    o = oracle_fma if arith == "fma" else oracle_sep
    lights = LIGHT_SETS[lset]
    s, osc = build_scene(scene_dirs, variant, scene, lights)
    set_scene(renderer, variant, s)
    counters = GRID_COUNTERS if variant == "grid" else COUNTERS
    saved = {}
    for rows in WINDOWS[scene]:
        ref = oracle_window(oracle_frames, o, variant, scene, lset, osc, rows)
        if len(lights):
            assert ref["counters"]["shadow_rays"] > 0, rows
        executed = {}
        for kernel, kw in flavours:
            what = "%s/%s lights/%s/%s%s rows %s" % (case, lset, arith, kernel, "".join("/%s=%s" % i for i in kw.items()), rows)
            res = renderer.render(variant, W, H, SEEDS, rows=rows, arith=arith, kernel=kernel, want_accum=True, want_rng=True,
                                  dead_rays="trace", **kw)
            same_bits(res, ref, variant, rows, what)
            for k in counters:
                assert res.counters[k] == ref["counters"][k], (what, k, res.counters[k], ref["counters"][k])
            executed.setdefault(kernel, res.counters["tri_tests_executed"])
            if kernel not in ELIDING:
                continue
            el = renderer.render(variant, W, H, SEEDS, rows=rows, arith=arith, kernel=kernel, want_accum=True, want_rng=True,
                                 dead_rays="elide", **kw)
            same_bits(el, ref, variant, rows, what + " elide")
            assert el.counters["samples"] == ref["counters"]["samples"], what + " elide"
            assert el.counters["shadow_rays"] <= ref["counters"]["shadow_rays"], what + " elide"
            assert el.counters["rays"] - el.counters["shadow_rays"] == ref["counters"]["rays"] - ref["counters"]["shadow_rays"], what
            saved[kernel] = saved.get(kernel, 0) + ref["counters"]["shadow_rays"] - el.counters["shadow_rays"]
        if "spec" in executed and "mega" in executed and case != "base-cluster-cull":
            # SPEC counts the triangle tests of the speculation it throws away, the megakernel has none to throw away.
            # (Not with cluster culling: the megakernel's cooperative scan skips the cluster cull in partial warps.)
            if scene == "silhouette" and rows == WINDOWS[scene][0]:
                assert executed["spec"] > executed["mega"], (case, lset, arith, rows, executed)
            elif rows == WINDOWS[scene][1]:
                # floor rows: every sample hits, SPEC's predictions all hold and it runs exactly the megakernel's tests
                assert executed["spec"] == executed["mega"], (case, lset, arith, rows, executed)
                if lset == "near-mesh":
                    assert executed["spec"] > 0              # shadow rays queued floor pixels for SPEC's heavy pass
    if len(lights) and variant != "nodof":                   # the NoDoF scene shows no triangle (its mesh is a placeholder)
        for kernel, n in saved.items():
            assert n > 0, (case, lset, arith, kernel)


def test_zero_intensity_light_is_traced_only_by_lmem(scene_dirs, oracle_fma):
    """Reach of the light sets: the zero-intensity light costs base no shadow rays and lmem one per hit sample"""
    for lset in ("3", "4", "5", "near-mesh"):
        _, osc = build_scene(scene_dirs, "lmem", "default", LIGHT_SETS[lset])
        rows = WINDOWS["default"][1]
        base = oracle_fma.render("base", W, H, SEEDS, osc, rows=rows, spp=8)
        lmem = oracle_fma.render("lmem", W, H, SEEDS, osc, rows=rows, spp=8)
        assert 0 < base["counters"]["shadow_rays"] < lmem["counters"]["shadow_rays"], lset


def test_near_mesh_light_sits_on_the_mesh(scene_dirs):
    s, _ = build_scene(scene_dirs, "grid", "default", NEAR_MESH)
    lo, hi = s.box_min[:3], s.box_max[:3]
    p = NEAR_MESH[0, :3]
    assert (lo[:2] < p[:2]).all() and (p[:2] < hi[:2]).all() and hi[2] < p[2] < hi[2] + 0.5      # just above the grid box
    assert np.linalg.norm(p - (lo + hi) / 2) < np.linalg.norm(hi - lo) / 2                     # inside the box's sphere


def test_switching_light_sets_on_one_renderer(renderer, scene_dirs):
    """5 -> 1 -> 0 -> 5 lights on the same context: the second 5-light frame equals the first bit for bit (wavefront
    graph, SPEC scratch and AUTO's estimate are refreshed with the scene)"""
    rows = (112, 144)
    first = {}
    for lset in ("5", "1", "0", "5"):
        s, _ = build_scene(scene_dirs, "base", "default", LIGHT_SETS[lset])
        renderer.set_scene(s)
        for kernel in ("wavefront", "spec", "auto"):
            res = renderer.render("base", W, H, SEEDS, rows=rows, kernel=kernel, want_accum=True, want_rng=True, dead_rays="trace")
            if lset != "5":
                continue
            if kernel not in first:
                first[kernel] = res
                continue
            a = first[kernel]
            assert np.array_equal(res.image, a.image), kernel
            assert np.array_equal(res.accum.view(np.uint32), a.accum.view(np.uint32)), kernel
            assert np.array_equal(res.rng_state, a.rng_state), kernel
            for k in COUNTERS:
                assert res.counters[k] == a.counters[k], (kernel, k)
