"""Edge geometry through EVERY kernel flavour (the single-ray probe reaches only the reference traversal): whole frames
against oracle.render with the same camera, bit for bit — image bytes, accumulation buffer, final RNG state and the
work counters (test_parity_gpu._compare).

Cameras built from camera_ray (pt_device.cuh):
  axis_ray  up = right = 0, eye = (-1, 0, 0): every camera ray is exactly (17, 16, 8) + t (-1, 0, 0), with signed zeros in y, z;
  fan_z8    right = (0, s, 0), up = 0, eye.z = 0: o.z == 8 and d.z == +0 exactly, the rays fan out in the plane z = 8.
Meshes: one whose box ends exactly at z = 8 (a box face in that plane), one whose z range is pinned to [0, 16] with
res.z a power of two (z = 8 an interior cell plane); under the default camera a flat mesh (zero-thickness box, 1x1x1
grid with cell_size.z = 0) and a mesh in negative x / y.  Ties: every triangle duplicated at a higher index with the
opposite winding (the winner's normal shows in the facing ratio) plus one large triangle spanning many cells."""
import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt
from conftest import SEED_SETS
from test_parity_gpu import _compare
from test_trace_probe_gpu import grid_dict, grid_for, mesh_scene, oracle_scene

pytestmark = pytest.mark.gpu

F32 = np.float32
GRID_KERNELS = ["mega", "persistent", "wavefront", "grid_tma", "grid_stream", "grid_pool", "grid_queue", "grid_async"]


def _q(x):
    return np.round(np.asarray(x, np.float64) * 1024) / 1024          # exactly representable coordinates


def _soup_in(lo, hi, n, seed, size=0.8):
    rng = np.random.default_rng(seed)
    c = rng.uniform(lo, hi, (n, 3))
    v = c[:, None, :] + rng.uniform(-size, size, (n, 3, 3))
    return _q(np.clip(v, lo, hi))


def z8_face_mesh():
    """soup in [4, 12] x [10, 22] x [0.5, 8]: the box's max z is exactly 8, some triangles have an edge or a vertex there"""
    v = _soup_in((4, 10, 0.5), (12, 22, 8), 300, 21)
    v[:40, :2, 2] = 8.0                                               # edges at z = 8
    v[40:60, 0, 2] = 8.0                                              # vertices at z = 8
    return mesh_scene(v)


def z8_cell_plane_mesh():
    """soup in [4, 12] x [10, 22] x [0, 16]: z pinned to [0, 16], so with res.z = 16 z = 8 is an interior cell plane"""
    v = _soup_in((4, 10, 0), (12, 22, 16), 400, 22)
    v[0, 0, 2], v[1, 0, 2] = 0.0, 16.0
    v[2:40, :2, 2] = 8.0
    return mesh_scene(v)


def _cam_arrays(up, right, eye):
    return {"cam_up": np.array(up + (0,), F32), "cam_right": np.array(right + (0,), F32), "eye_offset": np.array(eye + (0,), F32)}


CAMERAS = {"axis_ray": _cam_arrays((0.0, 0.0, 0.0), (0.0, 0.0, 0.0), (-1.0, 0.0, 0.0)),
           "fan_z8": _cam_arrays((0.0, 0.0, 0.0), (0.0, 1.0 / 256, 0.0), (-1.0, -0.5, 0.0))}


class _camera:
    """sets renderer.cam for the block and restores it afterwards"""

    def __init__(self, renderer, cam):
        self.r, self.cam = renderer, cam

    def __enter__(self):
        self.saved = self.r.cam
        c = pt.camera()
        c.cam_up[:] = [float(x) for x in self.cam["cam_up"]]
        c.cam_right[:] = [float(x) for x in self.cam["cam_right"]]
        c.eye_offset[:] = [float(x) for x in self.cam["eye_offset"]]
        self.r.cam = c

    def __exit__(self, *a):
        self.r.cam = self.saved


def _frame(renderer, o_lib, variant, scene, W, H, kernel, arith, cam=None, rows=None, spp=64, grid=None, what=""):
    renderer.set_scene(scene)
    gd = None
    if variant == "grid":
        renderer.build_grid(grid)
        gd = grid_dict(grid)
    r0, r1 = rows or (0, H)
    ctx = _camera(renderer, cam) if cam is not None else None
    if ctx:
        ctx.__enter__()
    try:
        res = renderer.render(variant, W, H, SEED_SETS[0], rows=(r0, r1), spp=spp, arith=arith, kernel=kernel, want_accum=True, want_rng=True)
    finally:
        if ctx:
            ctx.__exit__()
    ref = o_lib.render(variant, W, H, SEED_SETS[0], oracle_scene(scene), rows=(r0, r1), spp=spp, cam=cam, grid=gd)
    res.rng_state = res.rng_state.reshape(H, W, 4)[r0:r1].reshape(-1, 4)
    ref["rng_state"] = ref["rng_state"].reshape(H, W, 4)[r0:r1].reshape(-1, 4)
    res.accum, ref["accum"] = res.accum[r0:r1], ref["accum"][r0:r1]
    res.image, ref["image"] = res.image[r0:r1], ref["image"][r0:r1]
    _compare(res, ref, what)
    return res, ref


Z8_CASES = {"box_face_z8": (z8_face_mesh, None), "cell_plane_z8": (z8_cell_plane_mesh, (8, 12, 16))}


@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("kernel", GRID_KERNELS)
@pytest.mark.parametrize("mesh", list(Z8_CASES))
@pytest.mark.parametrize("camera", list(CAMERAS))
def test_z8_plane_cameras(renderer, oracle_fma, oracle_sep, camera, mesh, kernel, arith):
    make, res = Z8_CASES[mesh]
    s = make()
    g = grid_for(s, res)
    if mesh == "cell_plane_z8":
        assert g.box_min[2] == 0.0 and g.box_max[2] == 16.0 and g.cell_size[2] == 1.0
    else:
        assert g.box_max[2] == 8.0
    W, H = (8, 8) if camera == "axis_ray" else (8, 512)
    o_lib = oracle_fma if arith == "fma" else oracle_sep
    _, ref = _frame(renderer, o_lib, "grid", s, W, H, kernel, arith, cam=CAMERAS[camera], grid=g,
                    what="%s/%s/%s/%s" % (camera, mesh, kernel, arith))
    if mesh == "cell_plane_z8":
        assert ref["counters"]["cells_visited"] > 0 and ref["counters"]["tri_tests"] > 0
    else:               # the plane z = 8 holds the box face: d.z = +-0 gives a NaN slab, and the reference misses the box
        assert ref["counters"]["cells_visited"] == 0


def _camera_points(rows, cols, depth, seed, n):
    """points the default camera sees: pixel (col, row) at distance `depth` along its (pinhole) ray"""
    cam = pt.camera()
    up, right, eo = (np.array(x[:3], np.float64) for x in (cam.cam_up, cam.cam_right, cam.eye_offset))
    rng = np.random.default_rng(seed)
    i, j = rng.uniform(*cols, n), rng.uniform(*rows, n)
    d = up * i[:, None] + right * j[:, None] + eo
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.array([17.0, 16.0, 8.0]) + depth(d, rng)[:, None] * d


def flat_mesh_in_view():
    """triangles all in the plane z = 2 where the default camera looks down on it (rows 300..420)"""
    c = _camera_points((300, 420), (150, 360), lambda d, rng: (2.0 - 8.0) / d[:, 2], 1, 60)
    rng = np.random.default_rng(2)
    v = np.repeat(c[:, None, :], 3, 1)
    for k in range(3):
        a = 2 * np.pi * k / 3 + rng.uniform(0, 0.5, c.shape[0])
        v[:, k, 0] += 0.7 * np.cos(a)
        v[:, k, 1] += 0.7 * np.sin(a)
    v = _q(v)
    v[:, :, 2] = 2.0
    return mesh_scene(v)


def negative_mesh_in_view():
    """a soup entirely in x < 0, y < 0 (the reference's running max stays FLT_MIN there) seen in rows 200..260"""
    c = _camera_points((200, 260), (120, 400), lambda d, rng: rng.uniform(45, 60, d.shape[0]), 3, 800)
    c = c[(c[:, 0] < -1) & (c[:, 1] < -1) & (c[:, 2] > 1)]
    rng = np.random.default_rng(4)
    v = _q(c[:, None, :] + rng.uniform(-0.9, 0.9, (c.shape[0], 3, 3)))
    v[:, :, 0] = np.minimum(v[:, :, 0], -0.25)
    v[:, :, 1] = np.minimum(v[:, :, 1], -0.25)
    return mesh_scene(v)


OTHER_MESHES = {"flat": (flat_mesh_in_view, (300, 420)), "negative_xy": (negative_mesh_in_view, (200, 260))}


@pytest.mark.parametrize("kernel", GRID_KERNELS)
@pytest.mark.parametrize("mesh", list(OTHER_MESHES))
def test_flat_and_negative_meshes_default_camera(renderer, oracle_fma, mesh, kernel):
    make, rows = OTHER_MESHES[mesh]
    s = make()
    g = grid_for(s)
    if mesh == "flat":
        assert tuple(g.res[:3]) == (1, 1, 1) and g.cell_size[2] == 0.0
    else:
        assert s.box_max[0] == s.box_max[1] == np.finfo(F32).tiny
    _, ref = _frame(renderer, oracle_fma, "grid", s, 512, 512, kernel, "fma", rows=rows, spp=16, grid=g,
                    what="%s/%s" % (mesh, kernel))
    assert ref["counters"]["cells_visited"] > 0


def tie_scene(scene_dirs):
    """the default mesh, every triangle again at a higher index with the opposite winding, and one large triangle"""
    s = pt.load_scene_dir(scene_dirs["lmem"], "lmem")
    t = s.triangles
    rev = t.copy()
    rev[:, 4:8], rev[:, 8:12] = t[:, 8:12], t[:, 4:8]
    big = np.array([[6.0, 3.5, 9.4, 0, 9.0, 3.6, 9.6, 0, 7.4, 5.4, 11.6, 0]], F32)
    tris = np.concatenate([t, rev, big]).astype(F32)
    import gen_mesh
    lo, hi = gen_mesh.bbox_like_reference(tris)
    return pt.Scene(s.spheres, s.squares, tris, s.lights, lo, hi)


@pytest.mark.parametrize("variant,kernel", [("lmem", k) for k in ("mega", "spec", "persistent", "wavefront")]
                         + [("base", "mega"), ("base", "spec")] + [("grid", k) for k in GRID_KERNELS])
def test_duplicate_opposite_winding_ties(renderer, scene_dirs, oracle_fma, variant, kernel):
    s = tie_scene(scene_dirs)
    g = grid_for(s) if variant == "grid" else None
    W = H = 512
    for rows in ((112, 144), (144, 160)):
        _, ref = _frame(renderer, oracle_fma, variant, s, W, H, kernel, "fma", rows=rows, spp=64, grid=g,
                        what="ties/%s/%s/%s" % (variant, kernel, rows))
