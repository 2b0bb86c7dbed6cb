"""Brute-force triangle culls on meshes FAR from the origin (|x|, |y| from 1e5 to 1e7), against the oracle.

The brute-force variants skip the triangle scan for a ray whose line misses the mesh's bounding sphere, and (cluster
cull) the clusters of 8 records whose sphere it misses.  Both are only exact while the spheres contain the mesh around
the centre the device stores.  Rounding a double centre to float moves it by up to half an ulp per axis, which passes
the radius's 0.01 of slack once coordinates pass about 2^18; the device's own margins grow with the distance from the
ray origin to the mesh, so shadow rays that start a few units from a far mesh get almost none.  The meshes here put
the box centre on a half-ulp point, and the rays graze triangles near their vertices, where a sphere measured from the
unrounded centre loses them.

  a. ray by ray through the single-ray probe (mesh sphere), base and lmem, both arithmetic policies;
  b. whole frames whose shadow rays start on the floor next to the far mesh (mesh and cluster spheres), every
     brute-force flavour that reads them, against oracle.render on row windows;
  c. the same scenes through the grid variant's eight kernels (sphere prefilter and DDA far from the origin).

Each leg checks that its rays reach the boundary: line_misses restates the device's float32 line/sphere predicate, and
with the spheres built the old way (old_sphere: radius measured from the double centre, then the centre rounded) some
triangle hits of the oracle must fall outside them."""
import numpy as np
import pytest

from conftest import SEED_SETS
from test_grid_edge_frames_gpu import GRID_KERNELS, _camera
from test_bidir_gpu import same_floats
from test_parity_gpu import _compare
from test_trace_probe_gpu import T_CARRIED, compare, grid_for, grid_dict, mesh_scene, oracle_scene, rand_unit, ulps

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
X0S = (1e5, 3e5, 6e5, 1e6, 3e6, 1e7)
SIGNS = ((1, 1), (-1, 1), (1, -1), (-1, -1))


# ------------------------------------------------------------------------------- the device's cull, restated
def _fmaf(a, b, c):
    return (np.asarray(a, F64) * np.asarray(b, F64) + np.asarray(c, F64)).astype(F32)


def line_misses(c, r, k, o, d):
    """the device's float32 cull (trace_ray / line_near_sphere, pt_device.cuh): True where the ray's line is taken to
    miss the sphere (centre c, radius r, distance margin k).  Products feeding a subtraction are fused, as nvcc emits
    them."""
    c, o, d = np.asarray(c, F32), np.asarray(o, F32), np.asarray(d, F32)
    oc = (c[None, :] - o).astype(F32)
    ox, oy, oz = oc[:, 0], oc[:, 1], oc[:, 2]
    b = _fmaf(oz, d[:, 2], _fmaf(oy, d[:, 1], (ox * d[:, 0]).astype(F32)))
    oc2 = _fmaf(oz, oz, _fmaf(oy, oy, (ox * ox).astype(F32)))
    dist2 = _fmaf(-b, b, oc2)
    rm = _fmaf(F32(k), (np.abs(ox) + np.abs(oy) + np.abs(oz)).astype(F32), F32(r))
    return dist2 > _fmaf(rm, rm, (F32(1e-6) * oc2).astype(F32))


def old_sphere(tris):
    """a sphere as pt_set_scene built it before: radius measured from the DOUBLE box centre, then the centre cast"""
    v = np.asarray(tris, F32).reshape(-1, 3, 4)[:, :, :3].reshape(-1, 3).astype(F64)
    c = 0.5 * (v.min(0) + v.max(0))
    r = np.sqrt(((v - c) ** 2).sum(1).max()) * 1.01 + 0.01
    return c.astype(F32), F32(r)


def mesh_k(tris):
    v = np.asarray(tris, F32).reshape(-1, 3, 4)[:, :, :3].astype(F64)
    k = (np.linalg.norm(v[:, 1] - v[:, 0], axis=1) * np.linalg.norm(v[:, 2] - v[:, 0], axis=1)).max()
    return F32(2e-4 * k + 1e-6)


def culled_hits(tris, o, d, ref):
    """rays the oracle reports as triangle hits whose line the old mesh sphere culls"""
    return (ref["m"] == 4) & line_misses(*old_sphere(tris), mesh_k(tris), o, d)


# ------------------------------------------------------------------------------------------------------ meshes
def far_mesh(kind, x0, sx, sy, seed=0):
    """triangles in a box at (sx x0, sy x0, 1/16) of about 1 (triangle) or 2 (soup) units in x and y and 15/16 in z, x and y on
    the float32 lattice there, the x and y extents an odd number of ulps: the box centre is a half-ulp point, which float32
    cannot hold.  The first triangle spans three corners of the box, among them the corner opposite to where rounding
    moves the centre: the vertex a sphere measured from the unrounded centre loses first.  (n, 3, 3) float32"""
    u = float(np.spacing(F32(x0)))
    n = int(round((1.0 if kind == "triangle" else 2.0) / u)) | 1
    lo = np.array([sx * float(F32(x0)), sy * float(F32(x0)), 0.0625])
    hi = lo + np.array([n * u, n * u, 0.9375])
    mid = 0.5 * (lo + hi)
    shift = mid.astype(F32).astype(F64) - mid
    far, near = np.where(shift > 0, lo, hi), np.where(shift > 0, hi, lo)       # corners opposite to / towards the rounding
    tris = [[[far[0], far[1], lo[2]], [near[0], far[1], hi[2]], [far[0], near[1], hi[2]]]]
    if kind != "triangle":
        rng = np.random.default_rng(seed)
        v = rng.uniform(lo + 0.4, hi - 0.4, (5, 1, 3)) + rng.uniform(-0.4, 0.4, (5, 3, 3)) * np.array([1, 1, 0.5])
        v[:, :, :2] = lo[:2] + np.round((v[:, :, :2] - lo[:2]) / u) * u
        tris += list(v)
    v = np.array(tris, F64)
    assert np.array_equal(v[:, :, :2].astype(F32).astype(F64), v[:, :, :2]), "x, y off the float32 lattice"
    return v.astype(F32)


# ------------------------------------------------------------------------------------------------------- rays
def boundary_targets(rng, v, per=300):
    """points in double just inside and just outside each triangle near its vertices (barycentric offsets from 1e-4 to
    0.05 of an edge) and along its edges; half of them at the first vertex of the mesh (far_mesh).  The rays are aimed
    through these points, not through their float32 roundings, which far from the origin are an ulp apart."""
    v = np.asarray(v, F64)
    pts = []
    for k in (0, 0, 0, 1, 2):
        V, A, B = v[:, k], v[:, (k + 1) % 3], v[:, (k + 2) % 3]
        m = per if k == 0 else per // 2
        s = 10.0 ** rng.uniform(-4, -1.3, (m, v.shape[0], 1))
        t = 10.0 ** rng.uniform(-4, -1.3, (m, v.shape[0], 1))
        pts.append(V + s * (A - V) + t * (B - V))                                      # inside, at the vertex
        pts.append(V - s * (A - V) + t * (B - V))                                      # just outside, across an edge
        w = rng.uniform(0, 1, (m // 4, v.shape[0], 1))
        e = 10.0 ** rng.uniform(-5, -2, (m // 4, v.shape[0], 1)) * rng.choice([-1, 1], (m // 4, v.shape[0], 1))
        pts.append(V + w * (A - V) + e * (B - V))                                      # along the edge V-A, both sides
    return np.concatenate([p.reshape(-1, 3) for p in pts])


def far_mesh_rays(rng, v):
    """through boundary_targets: 3/4 from origins 1 to 50 units away, looking down, 1/4 from near the camera (17, 16, 8)"""
    p = boundary_targets(rng, v)
    p = p[rng.permutation(p.shape[0])]
    m = 3 * p.shape[0] // 4
    d0 = rand_unit(rng, m).astype(F64)
    d0[:, 2] = -np.abs(d0[:, 2])
    o1 = (p[:m] - (10.0 ** rng.uniform(0, np.log10(50), m))[:, None] * d0).astype(F32)
    o2 = (np.array([17.0, 16.0, 8.0]) + rng.uniform(-1, 1, (p.shape[0] - m, 3))).astype(F32)
    o = np.concatenate([o1, o2])
    d = p - o.astype(F64)
    return o, (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(F32)


MESH_KINDS = ["triangle", "soup"]


@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("kind", MESH_KINDS)
def test_far_mesh_rays(renderer, oracle_fma, oracle_sep, kind, arith):
    """material, t and normal bits of every ray equal the oracle's, for base (t reset) and lmem (carried t)"""
    o_lib = oracle_fma if arith == "fma" else oracle_sep
    rng = np.random.default_rng(20261022 + MESH_KINDS.index(kind))
    total, boundary = 0, {}
    for x0 in X0S:
        for sx, sy in SIGNS:
            s = mesh_scene(far_mesh(kind, x0, sx, sy))
            renderer.set_scene(s)
            osc = oracle_scene(s)
            o, d = far_mesh_rays(rng, s.triangles.reshape(-1, 3, 4)[:, :, :3])
            what = "%s x0=%g signs=%+d%+d/%s" % (kind, x0, sx, sy, arith)
            for variant in ("base", "lmem"):
                tin = np.full(o.shape[0], 1e9, F32)
                ref = o_lib.trace_rays(variant, o, d, tin, osc)
                compare(renderer.probe_trace(variant, o, d, tin, arith=arith), ref, "%s/%s" % (what, variant))
                total += o.shape[0]
            boundary[(x0, sx, sy)] = int(culled_hits(s.triangles, o, d, ref).sum())
            # carried bounds: each ray again with every t_in (the hit distance itself, and one ulp either side, included)
            k = min(o.shape[0], 3000)
            th = np.where(ref["m"][:k] == 4, ref["t"][:k], F32(5.0)).astype(F32)
            tc = np.concatenate([np.tile(T_CARRIED, k), th, ulps(th, 1), ulps(th, -1)])
            oo = np.concatenate([np.repeat(o[:k], len(T_CARRIED), 0), o[:k], o[:k], o[:k]])
            dd = np.concatenate([np.repeat(d[:k], len(T_CARRIED), 0), d[:k], d[:k], d[:k]])
            compare(renderer.probe_trace("lmem", oo, dd, tc, arith=arith), o_lib.trace_rays("lmem", oo, dd, tc, osc),
                    "%s/lmem carried t" % what)
            total += oo.shape[0]
    # the sets reach the boundary: beyond 2^19 the spheres of the old construction lose rays the oracle hits
    for key, n in boundary.items():
        if key[0] >= 6e5:
            assert n > 0, "no ray of %s %r grazes the mesh outside the old sphere" % (kind, key)
    assert sum(boundary.values()) >= 200 and total >= 500000, (boundary, total)


# ------------------------------------------------------------------------------------------------------ frames
# The camera looks down at floor points next to the far mesh, and the light sits on the far side of it: every sample's
# shadow ray starts a few units from the mesh.  A floor hit is a float32 point, so there its x and y lie on the lattice
# of x0 (1/16 at 6e5 and 1e6), and the light's jitter too.  The shadow origin X_s is the lattice point one step from
# the mesh's first vertex V0 (far_mesh) into the triangle; the light is placed so that the lines from X_s to the
# jittered light cross the triangle next to V0 nearly tangent to the old sphere: they miss it but hit the triangle.
FW, FH, FROWS = 32, 32, (8, 24)


def shadow_geometry(v):
    """(shadow origin X_s, light position) for the first triangle of far_mesh `v` (see above)"""
    v = np.asarray(v, F64)
    u = float(np.spacing(F32(abs(v[0, 0, 0]))))
    V0 = v[0, 0]
    ix, iy = np.sign(v[0, 1, 0] - V0[0]), np.sign(v[0, 2, 1] - V0[1])        # from V0 into the triangle
    xs = np.array([V0[0] + ix * u, V0[1], 0.0])
    light = np.array([V0[0] - 6.0 * ix - 0.5, V0[1] + 0.46 * iy - 0.5, 7.25])     # - 0.5: the jitter's mean
    return xs, light


def floor_camera(xs):
    """camera whose 32 x 32 focal points (all on the floor) are the floor's float32 lattice points within two steps of xs"""
    u = float(np.spacing(F32(abs(xs[0]))))
    ux, ry = 4 * u / (16 * FW), 4 * u / (16 * FH)
    eye = ((xs[0] - 17.0) / 16 - ux * FW / 2, (xs[1] - 16.0) / 16 - ry * FH / 2, -0.5)
    return {"cam_up": np.array([ux, 0, 0, 0], F32), "cam_right": np.array([0, ry, 0, 0], F32),
            "eye_offset": np.array(eye + (0,), F32)}


def shadow_lines(xs, light, step):
    """the shadow rays of the floor lattice points within two steps of xs to the 16 x 16 float32 positions of the jittered
    light (base:167-171)"""
    g = np.arange(-2, 3) * step
    X = np.stack(np.meshgrid(xs[0] + g, xs[1] + g), -1).reshape(-1, 2)
    X = np.concatenate([X, np.zeros((X.shape[0], 1))], 1).astype(F32)
    j = np.arange(16) / 16.0
    L = np.stack(np.meshgrid((F32(light[0]) + j).astype(F32), (F32(light[1]) + j).astype(F32)), -1).reshape(-1, 2)
    L = np.concatenate([L, np.full((L.shape[0], 1), F32(light[2]))], 1).astype(F32)
    o = np.repeat(X, L.shape[0], 0)
    d = np.tile(L, (X.shape[0], 1)).astype(F64) - o
    return o, (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(F32)


def cluster_mesh(x0, sx, sy, target=17, n=400, seed=8):
    """n small triangles at (sx x0, sy x0) in clusters of 8 that each fill about a unit, the clusters spread over +-20 units;
    cluster `target` is far_mesh("triangle") plus 7 small triangles inside its box, so its FIRST triangle (record
    8 * target) is the one the shadow geometry grazes.  The mesh sphere is large: only the cluster sphere is at stake."""
    rng = np.random.default_rng(seed)
    u = float(np.spacing(F32(x0)))
    corner = far_mesh("triangle", x0, sx, sy).astype(F64)
    lo, hi = corner.min(axis=(0, 1)), corner.max(axis=(0, 1))
    cl = []
    for c in range(n // 8):
        if c == target:
            inner = rng.uniform(lo + 0.2, hi - 0.2, (7, 1, 3)) + rng.uniform(-0.15, 0.15, (7, 3, 3))
            inner[:, :, :2] = np.round(inner[:, :, :2] / u) * u
            cl.append(np.concatenate([corner, inner]))
            continue
        while True:                 # keep the other clusters off the grazing lines (they run within 10 units of V0)
            ctr = corner[0, 0] + np.array([rng.uniform(-20, 20), rng.uniform(-20, 20), 0])
            if np.abs(ctr[:2] - corner[0, 0, :2]).max() > 12:
                break
        t = ctr + np.array([0, 0, 1.0]) + rng.uniform(-0.5, 0.5, (8, 1, 3)) + rng.uniform(-0.3, 0.3, (8, 3, 3))
        t[:, :, :2] = np.round(t[:, :, :2] / u) * u
        cl.append(t)
    return np.concatenate(cl).astype(F32)


def cluster_culled_hits(tris, o, d, c, o_lib):
    """rays whose only triangle hit is in cluster c, which the old cluster sphere of c culls: with it skipped the device
    would have reported no triangle at all"""
    t = np.asarray(tris, F32).reshape(-1, 12)
    part, rest = t[8 * c:8 * c + 8], np.concatenate([t[:8 * c], t[8 * c + 8:]])
    sc = {"spheres": np.zeros(9, np.int32), "squares": np.zeros(9, np.int32), "lights": np.zeros((1, 4), F32)}
    tin = np.full(o.shape[0], 1e9, F32)
    hit = o_lib.trace_rays("base", o, d, tin, dict(sc, triangles=part))["m"] == 4
    other = o_lib.trace_rays("base", o, d, tin, dict(sc, triangles=rest))["m"] == 4
    return hit & ~other & line_misses(*old_sphere(part), mesh_k(t), o, d)


def far_frame_scene(mesh, x0, sx, sy):
    """(scene, camera, shadow lines, number of those the old spheres lose) for mesh "single" (far_mesh triangle) or
    "clusters" (cluster_mesh)"""
    from oracle.pyoracle import OracleLib
    v = far_mesh("triangle", x0, sx, sy) if mesh == "single" else cluster_mesh(x0, sx, sy)
    xs, light = shadow_geometry(v[8 * 17:] if mesh == "clusters" else v)
    s = mesh_scene(v, lights=[tuple(light) + (400.0,)])
    s.spheres[:], s.squares[:] = 0, 0                      # nothing near the origin stands between camera and mesh
    o, d = shadow_lines(xs, light, float(np.spacing(F32(x0))))
    o_lib = OracleLib(contract=0)
    if mesh == "single":
        lost = culled_hits(s.triangles, o, d, o_lib.trace_rays("base", o, d, np.full(o.shape[0], 1e9, F32), oracle_scene(s)))
    else:
        lost = cluster_culled_hits(s.triangles, o, d, 17, o_lib)
    return s, floor_camera(xs), (o, d), int(lost.sum())


def far_soup(x0, sx, sy, n=17000, seed=9):
    """far_mesh("triangle") and n small soup triangles in 30 x 30 x 10 units around it, above z = 0.5: more than the
    16384 triangles of the small-grid kernels, and the shadow rays of the floor camera walk it"""
    import gen_mesh
    first = far_mesh("triangle", x0, sx, sy)
    t = gen_mesh.soup(n, seed=seed, box_lo=0.0, box_size=30.0).reshape(-1, 3, 4)[:, :, :3].astype(F64)
    t[:, :, 2] = 0.5 + t[:, :, 2] / 3
    t[:, :, :2] += first[0, 0, :2].astype(F64) - 15.0
    return np.concatenate([first, t.astype(F32)])


def _far_frame(renderer, o_lib, variant, scene, cam, kernel, arith="fma", spp=32, grid=None, what="", **kw):
    """one row window rendered on the device and by the oracle; every bit of the window compared (_compare: image,
    accumulation buffer, RNG states, counters), or with dead_rays="elide" every bit but the ray counters"""
    W, H, (r0, r1) = FW, FH, FROWS
    renderer.set_scene(scene)
    gd = None
    if variant == "grid":
        renderer.build_grid(grid)
        gd = grid_dict(grid)
    vpls = None
    if variant == "bidir":
        renderer.light_tracer(SEED_SETS[0], 512, arith=arith)
        vpls = o_lib.light_tracer(SEED_SETS[0], oracle_scene(scene), 512)
        assert same_floats(renderer.read_vpls(), vpls), "%s: VPL buffer differs from oracle.light_tracer" % what
    if variant == "nodof":
        spp = 64
    with _camera(renderer, cam):
        res = renderer.render(variant, W, H, SEED_SETS[0], rows=(r0, r1), spp=spp, arith=arith, kernel=kernel, want_accum=True,
                              want_rng=True, **kw)
    ref = o_lib.render(variant, W, H, SEED_SETS[0], oracle_scene(scene), rows=(r0, r1), spp=spp, cam=cam, grid=gd, vpls=vpls)
    k = 8 if variant == "nodof" else 1                    # NoDoF: 8 x 8 work-items (RNG streams) per pixel
    res.rng_state = res.rng_state.reshape(k * H, k * W, 4)[k * r0:k * r1].reshape(-1, 4)
    ref["rng_state"] = ref["rng_state"].reshape(k * H, k * W, 4)[k * r0:k * r1].reshape(-1, 4)
    res.accum, ref["accum"] = res.accum[r0:r1], ref["accum"][r0:r1]
    res.image, ref["image"] = res.image[r0:r1], ref["image"][r0:r1]
    if kw.get("dead_rays") == "elide":
        ref["counters"] = dict(ref["counters"], rays=res.counters["rays"], shadow_rays=res.counters["shadow_rays"],
                               tri_tests=res.counters["tri_tests"], prim_tests=res.counters["prim_tests"])
    _compare(res, ref, what)
    return ref


FRAME_MESHES = ["single", "clusters"]
PLACES = [(6e5, 1, 1), (1e6, -1, 1), (6e5, 1, -1), (1e6, -1, -1)]


@pytest.fixture(scope="module")
def far_scenes():
    """{(mesh, place): (scene, camera)}, each checked once: the old spheres lose shadow rays of its frame, and the
    mesh changes the oracle's image of the window"""
    from oracle.pyoracle import OracleLib
    o_lib = OracleLib(contract=0)
    out = {}
    for mesh in FRAME_MESHES:
        for place in PLACES:
            s, cam, _, lost = far_frame_scene(mesh, *place)
            assert lost >= 200, "%s %r: only %d shadow lines of the frame graze the mesh outside the old spheres" % (mesh, place, lost)
            bare = oracle_scene(s)
            bare["triangles"] = np.zeros((0, 12), F32)
            a = o_lib.render("base", FW, FH, SEED_SETS[0], oracle_scene(s), rows=FROWS, spp=32, cam=cam)["image"]
            b = o_lib.render("base", FW, FH, SEED_SETS[0], bare, rows=FROWS, spp=32, cam=cam)["image"]
            changed = int((a[FROWS[0]:FROWS[1]] != b[FROWS[0]:FROWS[1]]).any(axis=2).sum())
            assert changed >= 16, "%s %r: the mesh changes only %d pixels of the window" % (mesh, place, changed)
            out[(mesh, place)] = (s, cam)
    return out


BRUTE_FRAMES = ([(v, k, cc) for v in ("base", "lmem") for k in ("mega", "spec", "persistent", "wavefront") for cc in ("on", "off")]
                + [("nodof", "mega", "on"), ("nodof", "persistent", "on"), ("bidir", "mega", "on"), ("bidir", "mega", "off")])


@pytest.mark.parametrize("variant,kernel,cluster_cull", BRUTE_FRAMES)
@pytest.mark.parametrize("mesh", FRAME_MESHES)
def test_far_mesh_frames(renderer, oracle_fma, far_scenes, mesh, variant, kernel, cluster_cull):
    """shadow rays from the floor next to far meshes, through every brute-force flavour that reads the mesh sphere
    ("single") or the cluster spheres ("clusters", whose mesh sphere is large)"""
    for place in PLACES:
        s, cam = far_scenes[(mesh, place)]
        _far_frame(renderer, oracle_fma, variant, s, cam, kernel, cluster_cull=cluster_cull,
                   what="%s %r/%s/%s/cluster cull %s" % (mesh, place, variant, kernel, cluster_cull))


@pytest.mark.parametrize("variant", ["base", "lmem"])
@pytest.mark.parametrize("arith,dead_rays", [("separate", "trace"), ("fma", "elide"), ("separate", "elide")])
def test_far_mesh_frames_policies(renderer, oracle_fma, oracle_sep, far_scenes, variant, arith, dead_rays):
    """the megakernel under the separate arithmetic policy, and with the dead shadow rays elided"""
    o_lib = oracle_fma if arith == "fma" else oracle_sep
    for (mesh, place), (s, cam) in far_scenes.items():
        _far_frame(renderer, o_lib, variant, s, cam, "mega", arith=arith, cluster_cull="on", dead_rays=dead_rays,
                   what="%s %r/%s/%s/dead rays %s" % (mesh, place, variant, arith, dead_rays))


@pytest.mark.parametrize("kernel", GRID_KERNELS)
def test_far_mesh_frames_grid(renderer, oracle_fma, far_scenes, kernel):
    """the same frames through the grid variant (sphere prefilter and DDA far from the origin), and a 17 000-triangle
    soup there (the big-grid kernels)"""
    cases = [(k, s, cam) for k, (s, cam) in far_scenes.items() if k[1] in PLACES[:2]]
    for place in PLACES[:2]:
        s = mesh_scene(far_soup(*place), lights=far_scenes[("single", place)][0].lights)
        s.spheres[:], s.squares[:] = 0, 0
        cases.append((("soup17k", place), s, far_scenes[("single", place)][1]))
    for (mesh, place), s, cam in cases:
        ref = _far_frame(renderer, oracle_fma, "grid", s, cam, kernel, grid=grid_for(s),
                         what="%s %r/grid/%s" % (mesh, place, kernel))
        assert ref["counters"]["cells_visited"] > 0
