"""TraceRay ray by ray: the device intersection code (pt_probe_trace_counts) against the oracle's TraceRay
(oracle_trace_rays) on rays built to sit where the kernels' shortcuts are argued to be safe but could be wrong:
edges and vertices of triangles, near-parallel rays at the |det| = 0.01 cull, square edges, sphere tangents,
zero / signed-zero / subnormal direction components, origins on surfaces, far origins at the cull margins,
carried hit bounds, and for the grid: origins on faces, edges, corners and cell planes, rays through cell edges,
box-touching rays, long diagonal walks and walks cut short by the carried bound.

Bar: BIT-EXACT material and t, the normal's bits on every hit, and on grid rays the cells visited and the
triangle tests (the walk's visit set decides the result: there is no lower bound on t).  The brute-force test
counts are not compared: the device's conservative culls skip tests the reference runs.  Directions are unit
vectors, also with components replaced by 0 / -0 / subnormals and the rest renormalised: the culls assume |d| = 1,
which holds for every ray a render makes (camera and shadow rays are normalised).

Every set is generated from a fixed seed here.  golden_trace.npz pins the device against the reference itself."""
import os

import numpy as np
import pytest

import opencl_montecarlo_path_tracing_b200 as pt

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
F32 = np.float32
SUBN = np.array([1e-45, 1e-40, 1e-39, np.finfo(F32).tiny * 0.5], F32)      # subnormal magnitudes (and FLT_MIN / 2)


# --------------------------------------------------------------------------------------------------------- helpers
def ulps(x, k):
    """x moved by k ulps (k may be negative), elementwise, in float32."""
    x = np.asarray(x, F32).copy()
    k = np.broadcast_to(np.asarray(k), x.shape)
    for step in range(1, int(np.abs(k).max(initial=0)) + 1):
        m = np.abs(k) >= step
        x[m] = np.nextafter(x[m], np.where(k[m] > 0, F32(np.inf), F32(-np.inf)))
    return x


def unit(v):
    v = np.asarray(v, np.float64)
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(F32)


def rand_unit(rng, n):
    return unit(rng.normal(size=(n, 3)))


def aim(rng, target, dist):
    """origins at `dist` from float32 `target` points, directions towards them (unit, float32)."""
    d = rand_unit(rng, target.shape[0])
    o = (target.astype(np.float64) - np.asarray(dist, np.float64).reshape(-1, 1) * d).astype(F32)
    return o, unit(target.astype(np.float64) - o.astype(np.float64))


def tri_vertices(tris):
    t = np.asarray(tris, F32).reshape(-1, 12)
    return t[:, 0:3].astype(np.float64), t[:, 4:7].astype(np.float64), t[:, 8:11].astype(np.float64)


def nudged(p, rng):
    """every point moved by +-1..4 ulp in each coordinate independently (and once unmoved)"""
    p = np.asarray(p, F32)
    k = rng.integers(1, 5, size=p.shape) * rng.choice([-1, 1], size=p.shape)
    return np.concatenate([p, ulps(p, k)])


# --------------------------------------------------------------------------------------------------------- scenes
def oracle_scene(s):
    return {"spheres": s.spheres, "squares": s.squares, "triangles": s.triangles, "lights": s.lights,
            "box_min": s.box_min, "box_max": s.box_max}


def many_prims_scene(scene_dirs):
    """12 spheres and 10 squares: more than fit the kernel-parameter fast path (test_many_analytic_primitives)"""
    s = pt.load_scene_dir(scene_dirs["lmem"], "lmem")
    s.spheres = np.array([1024 + 64 + 4, 2, 0, 16384, 145, 0, 8 + 512, 2048, 65536], np.int32)
    s.squares = np.array([4096, 1, 32, 0, 2 + 1024, 0, 129, 16, 8192 + 8], np.int32)
    return s


def analytic_prims(s):
    """(squares [(x, z)], spheres [(x, z)]) of the bitmaps"""
    sq = [(k, 4 + j) for j in range(9) for k in range(19) if int(s.squares[j]) >> k & 1]
    sp = [(k, 4 + j) for j in range(9) for k in range(19) if int(s.spheres[j]) >> k & 1]
    return np.array(sq, np.float64).reshape(-1, 2), np.array(sp, np.float64).reshape(-1, 2)


def soup_scene(n, seed, box, lo=0.5):
    import gen_mesh
    tris = gen_mesh.soup(n, seed=seed, box_lo=lo, box_size=box)
    blo, bhi = gen_mesh.bbox_like_reference(tris)
    return pt.Scene(np.array([1024, 0, 0, 0, 145, 0, 0, 2048, 0], np.int32), np.array([4096, 0, 0, 0, 0, 0, 129, 0, 8192], np.int32),
                    tris, np.array([[10, 4, 10, 400], [15, 2, 7, 300]], F32), blo, bhi)


def mesh_scene(verts, lights=((10, 4, 10, 400), (15, 2, 7, 300))):
    """scene with the default spheres / squares and the given triangles ((n, 3, 3) vertices); box as the reference host keeps
    it (running max from FLT_MIN)"""
    import gen_mesh
    v = np.asarray(verts, F32).reshape(-1, 3, 3)
    tris = np.zeros((v.shape[0], 12), F32)
    for k in range(3):
        tris[:, 4 * k:4 * k + 3] = v[:, k]
    blo, bhi = gen_mesh.bbox_like_reference(tris)
    return pt.Scene(np.array([1024, 0, 0, 0, 145, 0, 0, 2048, 0], np.int32), np.array([4096, 0, 0, 0, 0, 0, 129, 0, 8192], np.int32),
                    tris, np.array(lights, F32), blo, bhi)


def flat_mesh(z=2.0, n=12, seed=5):
    """triangles all in the plane z = const: the box has zero thickness, pth_grid_dims gives a 1x1x1 grid with cell_size.z 0"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(3, 14, (n, 2))
    v = np.zeros((n, 3, 3))
    for k in range(3):
        a = 2 * np.pi * k / 3 + rng.uniform(0, 1, n)
        v[:, k, 0] = np.round((c[:, 0] + 1.5 * np.cos(a)) * 1024) / 1024
        v[:, k, 1] = np.round((c[:, 1] + 1.5 * np.sin(a)) * 1024) / 1024
        v[:, k, 2] = z
    return mesh_scene(v)


def negative_mesh(n=400, seed=6):
    """a soup entirely in negative x and y: the reference's running max stays FLT_MIN on those axes"""
    import gen_mesh
    t = gen_mesh.soup(n, seed=seed, box_lo=0.5, box_size=12.0)
    v = t.reshape(-1, 3, 4)[:, :, :3].copy()
    v[:, :, 0] = -v[:, :, 0]
    v[:, :, 1] = -v[:, :, 1] - 1.0
    return mesh_scene(v)


def corner_mesh():
    """four small triangles near corners of [0.5, 40.5]^3, off the main diagonals: a 128^3 grid of empty cells to walk"""
    v = [[(0.5, 0.5, 3.0), (2.0, 0.5, 3.0), (0.5, 2.0, 4.0)],
         [(40.5, 40.5, 37.0), (39.0, 40.5, 38.0), (40.5, 39.0, 37.5)],
         [(40.5, 0.5, 40.5), (39.0, 2.0, 40.5), (40.5, 2.5, 39.0)],
         [(0.5, 40.5, 0.5), (2.0, 39.0, 0.5), (0.5, 40.5, 2.5)]]
    return mesh_scene(v)


def grid_for(scene, res=None, modifier=3.0):
    g = pt.grid_dims(scene, modifier)
    if res is not None:
        for a in range(3):
            g.res[a] = int(res[a])
            g.cell_size[a] = float(F32(F32(g.box_max[a]) - F32(g.box_min[a])) / F32(res[a]))
    return g


def grid_dict(g):
    return {"box_min": np.array(g.box_min[:], F32), "box_max": np.array(g.box_max[:], F32),
            "res": np.array(g.res[:], np.int32), "cell_size": np.array(g.cell_size[:], F32)}


# ---------------------------------------------------------------------------------------------- brute-force rays
def rays_triangle_edges(rng, tris, n=30000):
    """points on every triangle's edges (u = 0, v = 0, u + v = 1) and vertices, +-1..4 ulp, from 1..30 away"""
    v0, v1, v2 = tri_vertices(tris)
    per = max(1, n // (6 * v0.shape[0]))
    s = rng.uniform(0, 1, (per, v0.shape[0], 1))
    pts = [v0, v1, v2]
    for a, b in ((v0, v1), (v0, v2), (v1, v2)):
        pts += list(a + s * (b - a))
    p = np.concatenate(pts).astype(F32)
    p = nudged(p, rng)
    return aim(rng, p, rng.uniform(1, 30, p.shape[0]))


def rays_near_parallel(rng, tris, n=30000):
    """|det| = |d . (e0 x e2)| within a few ulp of the 0.01 cull, through a point of the triangle"""
    v0, v1, v2 = tri_vertices(tris)
    e0 = (v1.astype(F32) - v0.astype(F32)).astype(np.float64)
    e2 = (v2.astype(F32) - v0.astype(F32)).astype(np.float64)
    N = np.cross(e0, e2)
    nl = np.linalg.norm(N, axis=1)
    keep = nl > 0.0101
    v0, e0, e2, N, nl = v0[keep], e0[keep], e2[keep], N[keep], nl[keep]
    per = max(1, n // max(1, nl.shape[0]))
    out_o, out_d = [], []
    for _ in range(per):
        a = (0.01 / nl) * (1.0 + rng.integers(-6, 7, nl.shape[0]) * 2.0 ** -23) * rng.choice([-1, 1], nl.shape[0])
        T = np.cross(N, rng.normal(size=N.shape))
        T /= np.linalg.norm(T, axis=1, keepdims=True)
        d = a[:, None] * (N / nl[:, None]) + np.sqrt(1 - a * a)[:, None] * T
        w = rng.dirichlet((1, 1, 1), nl.shape[0])
        P = v0 + w[:, 1:2] * e0 + w[:, 2:3] * e2
        o = P - rng.uniform(0.5, 10, (nl.shape[0], 1)) * d
        out_o.append(o)
        out_d.append(d)
    return np.concatenate(out_o).astype(F32), np.concatenate(out_d).astype(F32)


def rays_square_edges(rng, sq, n=30000):
    """hit points with |k - P.x| or |P.y| = 1 +- 1..4 ulp on every square (and its corners)"""
    pts = []
    per = max(1, n // (3 * len(sq)))
    for (k, z) in sq:
        e = ulps(np.full(per, 1.0, F32), rng.integers(-4, 5, per)).astype(np.float64)
        y = rng.uniform(-1, 1, per)
        sgn = rng.choice([-1, 1], per)
        pts += [np.stack([k + sgn * e, y, np.full(per, z)], 1), np.stack([k + y, sgn * e, np.full(per, z)], 1),
                np.stack([k + sgn * e, rng.choice([-1, 1], per) * e[::-1], np.full(per, z)], 1)]
    p = np.concatenate(pts).astype(F32)
    return aim(rng, p, rng.uniform(0.5, 40, p.shape[0]))


def rays_sphere_tangents(rng, sp, n=30000):
    """lines passing the centre at 1 +- a few ulp (qq ~ 0), and hits at r ~ 0.01"""
    os_, ds = [], []
    per = max(1, n // (2 * len(sp)))
    for (k, z) in sp:
        c = np.array([k, 0.0, z])
        u = rand_unit(rng, per).astype(np.float64)
        w = np.cross(u, rng.normal(size=(per, 3)))
        w /= np.linalg.norm(w, axis=1, keepdims=True)
        off = 1.0 + rng.integers(-8, 9, per) * 2.0 ** -23
        os_.append(c + off[:, None] * w - rng.uniform(1.5, 20, (per, 1)) * u)
        ds.append(u)
        n = rand_unit(rng, per).astype(np.float64)                    # r ~ 0.01: just outside the surface, looking in
        rr = 0.01 * (1.0 + rng.integers(-30, 31, per) * 2.0 ** -20)
        dn = -n + 0.05 * rng.normal(size=(per, 3))
        dn /= np.linalg.norm(dn, axis=1, keepdims=True)
        os_.append(c + (1.0 + rr)[:, None] * n)
        ds.append(dn)
    return np.concatenate(os_).astype(F32), unit(np.concatenate(ds))


def zero_like_dz(rng, n):
    return rng.choice(np.concatenate([[F32(0.0), F32(-0.0)], SUBN, -SUBN]), n).astype(F32)


def with_zero_like(d, mask, vals):
    """unit directions whose components under `mask` become the zero-like `vals`, the rest renormalised: still unit
    vectors, as every ray a render makes is (the device's conservative culls rely on that)"""
    d = np.where(mask, 0.0, np.asarray(d, np.float64))
    d = unit(d)
    d[mask] = vals
    return d


def rays_floor(rng, n=20000):
    """o.z = 0 (and +-0, subnormal) with d.z in {0, -0, +-subnormal} and ordinary d.z"""
    o = rng.uniform(-30, 40, (n, 3)).astype(F32)
    o[:, 2] = rng.choice(np.concatenate([[F32(0.0), F32(-0.0)], SUBN, -SUBN]), n)
    m = rng.uniform(size=n) < 0.75
    mask = np.zeros((n, 3), bool)
    mask[m, 2] = True
    return o, with_zero_like(rand_unit(rng, n), mask, zero_like_dz(rng, int(m.sum())))


def rays_square_planes(rng, sq, n=20000):
    """origins exactly on a square's plane (o.z = 4 + j), over or near the square, with d.z 0 / -0 / subnormal"""
    os_, ds = [], []
    per = max(9, n // len(sq))
    for (k, z) in sq:
        o = np.stack([k + rng.uniform(-1.3, 1.3, per), rng.uniform(-1.3, 1.3, per), np.full(per, z)], 1).astype(F32)
        mask = np.zeros((per, 3), bool)
        mask[:, 2] = True
        d = with_zero_like(rand_unit(rng, per), mask, zero_like_dz(rng, per))
        if per > 8:
            d[:4] = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0]], F32)
        os_.append(o)
        ds.append(d)
    return np.concatenate(os_), np.concatenate(ds)


def rays_far(rng, targets, n=60000):
    """|o| from 1e3 to 1e6, aimed at grazing points (edges, silhouettes): the distance-proportional cull margins"""
    p = targets[rng.integers(0, targets.shape[0], n)]
    return aim(rng, p, 10.0 ** rng.uniform(3, 6, n))


def brute_force_set(rng, s):
    sq, sp = analytic_prims(s)
    sets = {"triangle_edges": rays_triangle_edges(rng, s.triangles), "near_parallel": rays_near_parallel(rng, s.triangles),
            "square_edges": rays_square_edges(rng, sq), "sphere_tangents": rays_sphere_tangents(rng, sp),
            "floor_zero_dz": rays_floor(rng), "square_planes_zero_dz": rays_square_planes(rng, sq)}
    sets["far_origins"] = rays_far(rng, _graze_targets(rng, s, sq, sp))
    return sets


def _graze_targets(rng, s, sq, sp):
    v0, v1, v2 = tri_vertices(s.triangles)
    t = rng.uniform(0, 1, (v0.shape[0], 1))
    pts = [v0 + t * (v1 - v0), v1 + t * (v2 - v1), v2 + t * (v0 - v2)]
    for (k, z) in sq:
        y = rng.uniform(-1, 1, 64)
        pts.append(np.stack([k + np.ones(64), y, np.full(64, z)], 1))
        pts.append(np.stack([k + y, -np.ones(64), np.full(64, z)], 1))
    for (k, z) in sp:
        pts.append(np.array([k, 0, z]) + rand_unit(rng, 64))
    return np.concatenate(pts).astype(F32)


T_CARRIED = np.array([1e9, 0.02, 1e-3, 0.0, -1.0, np.inf], F32)


def compare(got, ref, what, counts=False):
    m, t, n = got[:3]
    bad = (m != ref["m"]) | (t.view(np.uint32) != ref["t"].view(np.uint32))
    hit = ref["m"] != 0
    bad |= hit & (n.view(np.uint32) != ref["n"].view(np.uint32)).any(axis=1)
    if counts:
        bad |= (got[3] != ref["cells"]) | (got[4] != ref["tests"])
    nb = int(bad.sum())
    if nb:
        i = int(np.nonzero(bad)[0][0])
        detail = "first: ray %d  device m=%d t=%r  oracle m=%d t=%r" % (i, m[i], float(t[i]), ref["m"][i], float(ref["t"][i]))
        if counts:
            detail += "  cells %d/%d tests %d/%d" % (got[3][i], ref["cells"][i], got[4][i], ref["tests"][i])
        raise AssertionError("%s: %d of %d rays differ from the oracle (%s)" % (what, nb, m.shape[0], detail))


# ------------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("variant", ["base", "lmem"])
def test_golden_trace_rays_match_reference(renderer, scene_dirs, variant):
    """the 4000 TraceRay probes of the reference itself (golden_trace.npz), separate policy: every bit"""
    g = np.load(os.path.join(G, "golden_trace.npz"))
    renderer.set_scene(pt.load_scene_dir(scene_dirs["lmem"], "lmem"))
    m, t, n = renderer.probe_trace(variant, g["origins"], g["dirs"], g["t_in"], arith="separate")
    bad = (m != g["m_" + variant]) | (t.view(np.uint32) != g["t_" + variant])
    bad |= (m != 0) & (n.view(np.uint32) != g["n_" + variant]).any(axis=1)
    assert not bad.any(), "%s: %d of %d rays differ from the reference's TraceRay" % (variant, int(bad.sum()), m.shape[0])
    assert len(set(m.tolist())) == 4


BRUTE_SCENES = ["default", "torus", "many_prims"]


def _brute_scene(scene_dirs, name):
    if name == "default":
        return pt.load_scene_dir(scene_dirs["lmem"], "lmem")
    if name == "torus":
        return pt.load_scene_dir(scene_dirs["torus"], "base")
    return many_prims_scene(scene_dirs)


@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("scene_name", BRUTE_SCENES)
def test_brute_force_edge_rays(renderer, scene_dirs, oracle_fma, oracle_sep, scene_name, arith):
    o_lib = oracle_fma if arith == "fma" else oracle_sep
    s = _brute_scene(scene_dirs, scene_name)
    renderer.set_scene(s)
    osc = oracle_scene(s)
    rng = np.random.default_rng(20261020 + BRUTE_SCENES.index(scene_name))
    total = 0
    for case, (o, d) in brute_force_set(rng, s).items():
        for variant in ("base", "lmem"):
            tin = np.full(o.shape[0], 1e9, F32)
            got = renderer.probe_trace(variant, o, d, tin, arith=arith)
            ref = o_lib.trace_rays(variant, o, d, tin, osc)
            compare(got, ref, "%s/%s/%s/%s" % (scene_name, case, variant, arith))
            total += o.shape[0]
        if case != "far_origins":          # carried bounds (lmem): each ray again with every t_in
            k = min(o.shape[0], 4000)
            oo, dd = np.repeat(o[:k], len(T_CARRIED), 0), np.repeat(d[:k], len(T_CARRIED), 0)
            tin = np.tile(T_CARRIED, k)
            compare(renderer.probe_trace("lmem", oo, dd, tin, arith=arith), o_lib.trace_rays("lmem", oo, dd, tin, osc),
                    "%s/%s/lmem carried t/%s" % (scene_name, case, arith))
            total += oo.shape[0]
    assert total >= 200000


def test_square_plane_origin_with_subnormal_dz(renderer, scene_dirs, oracle_fma, oracle_sep):
    """origin exactly on a square's plane, d.z subnormal: the reference divides 0 by d.z, gets r = 0 and hits at t = 0"""
    s = pt.load_scene_dir(scene_dirs["lmem"], "lmem")
    renderer.set_scene(s)
    sq, _ = analytic_prims(s)
    k, z = sq[0]
    o = np.array([[k + 0.25, 0.5, z]] * 4, F32)
    d = unit([[0.6, 0.8, 0.0]] * 4)
    d[:, 2] = [1e-40, -1e-40, 1e-45, 0.0]
    for arith, lib in (("fma", oracle_fma), ("separate", oracle_sep)):
        ref = lib.trace_rays("lmem", o, d, np.full(4, 1e9, F32), oracle_scene(s))
        assert list(ref["m"][:3]) == [3, 3, 3] and ref["m"][3] != 3
        compare(renderer.probe_trace("lmem", o, d, np.full(4, 1e9, F32), arith=arith), ref, "square plane origin/" + arith)


# ------------------------------------------------------------------------------------------------------ grid rays
def grid_points(rng, g, n):
    """points on box faces, edges, corners and interior cell planes, exactly / 1 ulp inside / 1 ulp outside"""
    lo, hi = np.array(g.box_min[:3], F32), np.array(g.box_max[:3], F32)
    res, cell = np.array(g.res[:3]), np.array(g.cell_size[:3], F32)
    p = rng.uniform(lo, hi, (n, 3)).astype(F32)
    kind = rng.integers(0, 4, n)                   # 0 face, 1 edge, 2 corner, 3 interior cell plane(s)
    for i in range(n):
        axes = rng.permutation(3)[: {0: 1, 1: 2, 2: 3, 3: rng.integers(1, 4)}[kind[i]]]
        for a in axes:
            if kind[i] == 3 and res[a] > 1:
                p[i, a] = F32(lo[a] + F32(rng.integers(1, res[a])) * cell[a])
            else:
                p[i, a] = lo[a] if rng.uniform() < 0.5 else hi[a]
    shift = rng.integers(-1, 2, (n, 3))
    return ulps(p, shift)


def special_dirs(rng, n):
    """unit directions with components replaced by 0 / -0 / subnormals, axis-parallel ones included"""
    mask = rng.uniform(size=(n, 3)) < 0.35
    mask[mask.all(axis=1), rng.integers(0, 3)] = False
    vals = np.concatenate([[F32(0.0), F32(-0.0)], SUBN, -SUBN])
    d = with_zero_like(rand_unit(rng, n), mask, rng.choice(vals, int(mask.sum())))
    ax = rng.uniform(size=n) < 0.15
    a = rng.integers(0, 3, int(ax.sum()))
    dd = np.zeros((int(ax.sum()), 3), F32)
    dd[np.arange(a.shape[0]), a] = rng.choice([-1, 1], a.shape[0])
    dd[rng.uniform(size=dd.shape) < 0.3] = F32(-0.0)
    dd[np.arange(a.shape[0]), a] = rng.choice([-1, 1], a.shape[0])
    d[ax] = dd
    return d


def grid_rays(rng, g, n=60000):
    lo, hi = np.array(g.box_min[:3], np.float64), np.array(g.box_max[:3], np.float64)
    res, cell = np.array(g.res[:3]), np.array(g.cell_size[:3], np.float64)
    size = hi - lo
    sets = {}
    # origins on faces / edges / corners / cell planes (+-1 ulp), random and special directions
    p = grid_points(rng, g, n // 4)
    sets["origins_on_box_and_cell_planes"] = (p, np.where(rng.uniform(size=(p.shape[0], 1)) < 0.5, rand_unit(rng, p.shape[0]),
                                                          special_dirs(rng, p.shape[0])))
    # special directions from anywhere in and around the box
    o = rng.uniform(lo - 0.2 * size - 1, hi + 0.2 * size + 1, (n // 4, 3)).astype(F32)
    sets["zero_and_subnormal_dirs"] = (o, special_dirs(rng, o.shape[0]))
    # through cell edges and corners of the lattice
    i = np.stack([rng.integers(0, r + 1, n // 4) for r in res], 1)
    q = (lo + i * cell).astype(F32)
    keep = rng.uniform(size=q.shape) < 0.33                          # some coordinates free: through cell edges only
    q[keep] = rng.uniform(lo, hi, q.shape)[keep].astype(F32)
    oo, dd = aim(rng, q, rng.uniform(0.5, 2, q.shape[0]) * np.linalg.norm(size))
    sets["through_cell_edges_and_corners"] = (oo, dd)
    # rays touching the box along an edge (t0 == t1) or missing it by 1 ulp
    m = n // 8
    a = rng.integers(0, 3, m)
    b = (a + rng.integers(1, 3, m)) % 3
    c = 3 - a - b
    o = np.zeros((m, 3), np.float64)
    d = np.zeros((m, 3), np.float64)
    off = rng.uniform(0.1, 5, m)
    sa, sb = rng.choice([0, 1], m), rng.choice([0, 1], m)
    ea = np.where(sa, hi[a], lo[a])
    eb = np.where(sb, hi[b], lo[b])
    ra = np.arange(m)
    # approach edge (ea, eb) from outside along axis a, leave outside along axis b: slab entry of a == slab exit of b
    o[ra, a] = ea + np.where(sa, 1, -1) * off
    o[ra, b] = eb - np.where(sb, 1, -1) * off
    o[ra, c] = rng.uniform(lo[c], hi[c])
    d[ra, a] = np.where(sa, -1, 1)
    d[ra, b] = np.where(sb, 1, -1)
    o32 = o.astype(F32)
    d32 = unit(d)
    sh = rng.integers(-1, 2, (m, 1)) * np.eye(3, dtype=int)[b]
    sets["touching_the_box"] = (ulps(o32, sh), d32)
    # 1-cell walks: inside a corner or face cell, heading straight out
    m = n // 8
    corner = rng.choice([0, 1], (m, 3))
    o = lo + np.where(corner, size - 0.5 * cell, 0.5 * cell) * rng.uniform(0.2, 1.8, (m, 3))
    d = np.where(corner, 1, -1) * rng.uniform(0.1, 1, (m, 3))
    sets["one_cell_walks"] = (o.astype(F32), unit(d))
    return sets


def diagonal_walks(rng, g, n=2000):
    """corner to corner of the box, slightly off the diagonal: >= 3 * res - 2 cells"""
    lo, hi = np.array(g.box_min[:3], np.float64), np.array(g.box_max[:3], np.float64)
    c = rng.choice([0, 1], (n, 3))
    a = np.where(c, hi, lo) + np.where(c, 1, -1) * rng.uniform(0.01, 0.5, (n, 3))
    b = np.where(c, lo, hi) + rng.normal(scale=0.05, size=(n, 3))
    return a.astype(F32), unit(b - a)


GRID_CASES = ["default", "default_res_1x1x1", "default_res_128x1x1", "default_res_1x1x128", "soup30k", "soup70k", "flat", "negative_xy",
              "corners_128cubed"]


def _grid_case(scene_dirs, name):
    if name.startswith("default"):
        s = pt.load_scene_dir(scene_dirs["grid"], "grid")
        res = {"default": None, "default_res_1x1x1": (1, 1, 1), "default_res_128x1x1": (128, 1, 1),
               "default_res_1x1x128": (1, 1, 128)}[name]
        return s, grid_for(s, res)
    if name == "soup30k":
        s = soup_scene(30000, 11, 24.0)
    elif name == "soup70k":
        s = soup_scene(70000, 11, 30.0)
    elif name == "flat":
        s = flat_mesh()
    elif name == "negative_xy":
        s = negative_mesh()
    else:
        s = corner_mesh()
        return s, grid_for(s, (128, 128, 128))
    return s, grid_for(s)


@pytest.mark.parametrize("arith", ["fma", "separate"])
@pytest.mark.parametrize("case", GRID_CASES)
def test_grid_edge_rays(renderer, scene_dirs, oracle_fma, oracle_sep, case, arith):
    o_lib = oracle_fma if arith == "fma" else oracle_sep
    s, g = _grid_case(scene_dirs, case)
    renderer.set_scene(s)
    renderer.build_grid(g)
    gd = grid_dict(g)
    start, refs = renderer.read_grid_csr()
    gd["csr"] = o_lib.build_grid(s.triangles, gd["box_min"], gd["res"], gd["cell_size"])
    assert np.array_equal(start, gd["csr"][0]) and np.array_equal(refs, gd["csr"][1]), "%s: device grid != oracle binning" % case
    osc = oracle_scene(s)
    rng = np.random.default_rng(77 + GRID_CASES.index(case))
    sets = grid_rays(rng, g)
    if case == "corners_128cubed":
        sets["box_diagonal_walks"] = diagonal_walks(rng, g)
    total = 0
    for name, (o, d) in sets.items():
        tin = np.full(o.shape[0], 1e9, F32)
        ref = o_lib.trace_rays("grid", o, d, tin, osc, grid=gd)
        compare(renderer.probe_trace("grid", o, d, tin, arith=arith, counts=True), ref, "%s/%s/%s" % (case, name, arith), counts=True)
        total += o.shape[0]
        if name == "box_diagonal_walks":
            assert int(ref["cells"].max()) >= 380, ref["cells"].max()
        # a carried bound that ends the walk mid-grid: half the distance to the hit (or into the box on a miss)
        walked = ref["cells"] > 1
        if walked.any():
            oo, dd = o[walked], d[walked]
            tt = np.where(ref["m"][walked] != 0, ref["t"][walked] * F32(0.5),
                          F32(0.5) * F32(np.linalg.norm(gd["box_max"][:3] - gd["box_min"][:3]))).astype(F32)
            tt = np.concatenate([tt, ulps(tt, 1), ulps(tt, -1)])
            oo, dd = np.concatenate([oo] * 3), np.concatenate([dd] * 3)
            ref2 = o_lib.trace_rays("grid", oo, dd, tt, osc, grid=gd)
            compare(renderer.probe_trace("grid", oo, dd, tt, arith=arith, counts=True), ref2, "%s/%s carried t/%s" % (case, name, arith),
                    counts=True)
            total += oo.shape[0]
    assert total >= 60000
