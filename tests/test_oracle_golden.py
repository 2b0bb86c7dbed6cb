"""The oracle against the golden vectors produced by the REFERENCE ITSELF (tests/golden/make_golden.py:
unmodified reference .c/.ocl compiled through oracle/refrt).  CPU only."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import SEED_SETS

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_rng_known_answers(oracle_sep):
    g = json.load(open(os.path.join(G, "golden_rng.json")))
    for k, v in g["randomize_id"].items():
        assert oracle_sep.lib.oracle_randomize_id(int(k)) == v
    for s in g["streams"]:
        f, u, st = oracle_sep.rng_kat(s["seeds"], s["gid"], 64)
        assert [int(x) for x in f.view(np.uint32)] == s["float_bits"]
        assert [int(x) for x in st] == s["state"]
        # first output is pixel independent: (s.x ^ s.z, s.y ^ s.w)   (SURVEY.md appendix B)
        assert int(u[0]) == s["seeds"][0] ^ s["seeds"][2] and int(u[1]) == s["seeds"][1] ^ s["seeds"][3]


def test_rng_is_not_textbook_mwc64x(oracle_sep):
    """The reference adds 0xFFFFFFFF on carry; a textbook +1 MWC64X would give these out3 values instead."""
    wrong = {((1, 2, 3, 4), 0): (0x1985e7ad, 0xe1858108), ((1, 2, 3, 4), 12345): (0xdd135ba1, 0x07877929),
             ((123456789, 42, 7, 99999), 262143): (0x4b823e8a, 0x8e372978)}
    right = {((1, 2, 3, 4), 0): (0x199a77e7, 0xe18030c6), ((1, 2, 3, 4), 12345): (0xdd135ba3, 0x07877929),
             ((123456789, 42, 7, 99999), 262143): (0x4b9faed0, 0x89ca9932)}
    for (seeds, gid), w in wrong.items():
        _, u, _ = oracle_sep.rng_kat(seeds, gid, 4)
        assert (int(u[6]), int(u[7])) == right[(seeds, gid)]
        assert (int(u[6]), int(u[7])) != w


def test_trace_ray_golden(oracle_sep, scene_dirs):
    g = np.load(os.path.join(G, "golden_trace.npz"))
    sc = oracle_sep.load_scene_dir(scene_dirs["lmem"], "lmem")
    n = g["origins"].shape[0]
    for variant, carry in (("base", 0), ("lmem", 1)):
        bad = 0
        for k in range(n):
            m, t, nn = oracle_sep.trace_ray(carry, g["origins"][k], g["dirs"][k], float(g["t_in"][k]), sc["spheres"], sc["squares"], sc["triangles"])
            ok = m == int(g["m_" + variant][k]) and np.float32(t).view(np.uint32) == g["t_" + variant][k]
            if m:
                ok = ok and np.array_equal(nn.view(np.uint32), g["n_" + variant][k])
            bad += not ok
        assert bad == 0, "%s: %d of %d rays differ from the reference TraceRay" % (variant, bad, n)
    assert len(set(g["m_lmem"].tolist())) == 4    # the vectors cover sky, floor, diffuse and triangle hits


def test_batched_trace_rays_equal_single_ray_probe(oracle_sep, scene_dirs):
    """oracle_trace_rays (the batch entry the device probe is compared with) gives the golden rays the bits of
    oracle_trace_ray (the entry the reference's own answers pin above)"""
    g = np.load(os.path.join(G, "golden_trace.npz"))
    sc = oracle_sep.load_scene_dir(scene_dirs["lmem"], "lmem")
    for variant, carry in (("base", 0), ("lmem", 1)):
        out = oracle_sep.trace_rays(variant, g["origins"], g["dirs"], g["t_in"], sc)
        for k in range(0, g["origins"].shape[0], 7):
            m, t, nn = oracle_sep.trace_ray(carry, g["origins"][k], g["dirs"][k], float(g["t_in"][k]), sc["spheres"], sc["squares"], sc["triangles"])
            assert out["m"][k] == m and out["t"][k].view(np.uint32) == np.float32(t).view(np.uint32), (variant, k)
            assert np.array_equal(out["n"][k].view(np.uint32), nn.view(np.uint32)), (variant, k)
        assert np.array_equal(out["m"], g["m_" + variant]) and np.array_equal(out["t"].view(np.uint32), g["t_" + variant])
        assert (out["cells"] == 0).all() and (out["tests"] == sc["triangles"].shape[0]).all()


@pytest.mark.parametrize("oracle_name", ["oracle_sep", "oracle_fma"])
def test_one_cell_grid_walk_equals_brute_force(request, scene_dirs, oracle_name):
    """A 1x1x1 grid over a mesh of at most 62 triangles lists every triangle, in index order, in its one cell, and the
    slab test has no lower bound on t: every ray whose line crosses the box tests all of them, as the brute-force scan
    does.  So the grid walk and the scan must give the same material, t and normal bits, from inside and outside the box."""
    o_lib = request.getfixturevalue(oracle_name)
    sc = o_lib.load_scene_dir(scene_dirs["torus"], "grid")
    assert sc["triangles"].shape[0] <= 62
    lo, hi = sc["box_min"][:3].astype(np.float64), sc["box_max"][:3].astype(np.float64)
    grid = {"box_min": sc["box_min"], "box_max": sc["box_max"], "res": np.array([1, 1, 1, 0], np.int32),
            "cell_size": np.append((hi - lo), 0).astype(np.float32)}
    rng = np.random.default_rng(3)
    n = 40000
    target = rng.uniform(lo, hi, (n, 3))
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = (target - rng.uniform(-3, 20, (n, 1)) * d).astype(np.float32)
    d = rng.choice([-1.0, 1.0], (n, 1)) * (target - o)
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    tin = np.full(n, 1e9, np.float32)
    g = o_lib.trace_rays("grid", o, d, tin, sc, grid=grid)
    b = o_lib.trace_rays("lmem", o, d, tin, sc)
    assert np.array_equal(g["m"], b["m"]) and np.array_equal(g["t"].view(np.uint32), b["t"].view(np.uint32))
    assert np.array_equal(g["n"].view(np.uint32), b["n"].view(np.uint32))
    assert (g["m"] == 4).sum() > n // 10 and (g["t"] < 0).sum() > 0 and (g["cells"] == 1).mean() > 0.99


@pytest.mark.parametrize("variant", ["base", "lmem", "nodof", "grid"])
def test_image_rows_golden(oracle_sep, scene_dirs, variant):
    g = np.load(os.path.join(G, "golden_images.npz"))
    sc = oracle_sep.load_scene_dir(scene_dirs[variant], variant)
    for si, seeds in enumerate(SEED_SETS):
        for ri, row in enumerate(g["rows"]):
            out = oracle_sep.render(variant, 512, 512, seeds, sc, rows=(int(row), int(row) + 1), want_rng=False)
            assert np.array_equal(out["image"][row], g["%s_s%d_rows" % (variant, si)][ri]), (variant, si, int(row))


def test_full_frame_hash_golden(oracle_sep, scene_dirs):
    g = np.load(os.path.join(G, "golden_images.npz"))
    sc = oracle_sep.load_scene_dir(scene_dirs["nodof"], "nodof")
    out = oracle_sep.render("nodof", 512, 512, SEED_SETS[0], sc, want_rng=False, want_accum=False)
    assert hashlib.sha256(out["image"].tobytes()).digest() == g["nodof_s0_sha256"].tobytes()
    sc = oracle_sep.load_scene_dir(scene_dirs["torus"], "base")
    out = oracle_sep.render("base", 640, 360, SEED_SETS[0], sc, want_rng=False, want_accum=False)
    assert hashlib.sha256(out["image"].tobytes()).digest() == g["torus_640x360_sha256"].tobytes()


def test_grid_with_other_mesh_and_modifier_golden(oracle_sep, tmp_path):
    import write_scenes
    g = np.load(os.path.join(G, "golden_images.npz"))
    d = str(tmp_path / "gt")
    write_scenes.write_variant("grid", d, mesh="torus")
    sc = oracle_sep.load_scene_dir(d, "grid")
    for ri, row in enumerate(g["rows"]):
        out = oracle_sep.render("grid", 512, 512, SEED_SETS[0], sc, rows=(int(row), int(row) + 1), want_rng=False, modifier=6.5)
        assert np.array_equal(out["image"][row], g["gridtorus_m6.5_rows"][ri])


def test_grid_build_golden(oracle_sep, tmp_path):
    import write_scenes
    g = np.load(os.path.join(G, "golden_grid.npz"))
    for name, mesh in (("default", None), ("torus", "torus"), ("torus_fine", "torus")):
        d = str(tmp_path / name)
        write_scenes.write_variant("grid", d, mesh=mesh)
        sc = oracle_sep.load_scene_dir(d, "grid")
        res, cell = oracle_sep.grid_dims(sc["box_min"], sc["box_max"], sc["triangles"].shape[0], float(g[name + "_modifier"]))
        assert np.array_equal(res, g[name + "_res"]) and np.array_equal(cell.view(np.uint32), g[name + "_cell"])
        start, refs = oracle_sep.build_grid(sc["triangles"], sc["box_min"], res, cell)
        nels = g[name + "_nels"]
        for c in range(len(nels)):
            mine = refs[start[c]:start[c + 1]]
            if nels[c] <= 62:      # below the cap the reference's (unordered) cell holds exactly this set
                assert np.array_equal(np.sort(mine), g[name + "_ids"][c][: nels[c]].astype(np.uint32)), (name, c)
            else:                  # reference overflows (bug); ours keeps the first 62 by triangle id
                assert len(mine) == 62
            assert np.all(np.diff(mine.astype(np.int64)) > 0)   # triangle-id order


def test_host_golden(oracle_sep, scene_dirs):
    g = json.load(open(os.path.join(G, "golden_host.json")))
    cam = oracle_sep.camera()
    line = "Cam_forward %f %f %f\nCam_up %f %f %f\nCam_right %f %f %f\n eye_offset %f %f %f" % (
        *cam["cam_forward"][:3], *cam["cam_up"][:3], *cam["cam_right"][:3], *cam["eye_offset"][:3])
    assert line == g["base"]["camera_print"]
    # hex constants of SURVEY.md appendix B
    assert [float(x).hex() for x in cam["cam_up"][:2]] == ["-0x1.eae7fc0000000p-10", "0x1.702dfe0000000p-11"]
    assert [float(x).hex() for x in cam["eye_offset"][:3]] == ["0x1.06b6280000000p-3", "-0x1.1db9040000000p+0", "0x1.0624de0000000p-1"]
    for v in ("base", "lmem", "nodof", "grid"):
        sc = oracle_sep.load_scene_dir(scene_dirs[v], v)
        assert sc["triangles"].shape[0] == g[v]["ntriangles"] and sc["lights"].shape[0] == g[v]["nlights"]
    sc = oracle_sep.load_scene_dir(scene_dirs["grid"], "grid")
    assert "vmax: %f %f %f, vmin: %f %f %f" % (*sc["box_max"][:3], *sc["box_min"][:3]) == g["grid"]["bbox_print"]
    res, _ = oracle_sep.grid_dims(sc["box_min"], sc["box_max"], 96, 3.0)
    assert list(res[:3]) == g["grid"]["grid_size"] == [8, 5, 6]
    sc = oracle_sep.load_scene_dir(scene_dirs["torus"], "base")
    assert sc["triangles"].shape[0] == g["torus"]["ntriangles"] == 32


def test_contract_modes_agree_within_tolerance(oracle_sep, oracle_fma, scene_dirs):
    """The two legal arithmetic policies: identical RNG streams on almost every pixel, images within 1 LSB."""
    sc = oracle_sep.load_scene_dir(scene_dirs["lmem"], "lmem")
    rows = (330, 362)
    a = oracle_sep.render("lmem", 512, 512, SEED_SETS[0], sc, rows=rows)
    b = oracle_fma.render("lmem", 512, 512, SEED_SETS[0], sc, rows=rows)
    same_rng = (a["rng_state"] == b["rng_state"]).all(axis=1).reshape(512, 512)[rows[0]:rows[1]]
    assert same_rng.mean() >= 0.999
    diff = np.abs(a["image"][rows[0]:rows[1]].astype(int) - b["image"][rows[0]:rows[1]].astype(int))
    assert (diff <= 1).mean() >= 0.995 and np.sqrt((diff.astype(float) ** 2).mean()) <= 0.5
    rel = np.abs(a["accum"] - b["accum"])[rows[0]:rows[1]][same_rng] / np.maximum(np.abs(a["accum"][rows[0]:rows[1]][same_rng]), 1e-6)
    assert np.median(rel) <= 1e-6


# ---- CLSuperBidirectionalPathTracer (SURVEY.md 8f, rank 2) --------------------------------------------------
def test_bidir_light_tracer_golden(oracle_sep, scene_dirs):
    """The VPL buffer of the reference's lightTracer kernel, bit for bit — including N_VLP*nlights < 512,
    where the reference divides by (total_vlp/512) == 0 and deposits inf / NaN intensities."""
    g = np.load(os.path.join(G, "golden_bidir.npz"))
    sc = oracle_sep.load_scene_dir(scene_dirs["bidir"], "bidir")
    for si, seeds in enumerate(SEED_SETS):
        for n in (512, 700, 96):
            got = oracle_sep.light_tracer(seeds, sc, n)
            ref = g["vpl_s%d_n%d" % (si, n)]
            assert np.array_equal(got.view(np.uint32), ref), (si, n)
    f = g["vpl_s0_n96"].view(np.float32)[:, 3]
    assert np.isnan(f).any() and np.isinf(f).any()
    # only surfaces hit from BEHIND keep a non-zero intensity (the reference dots the incoming direction with the
    # outward normal): every non-zero VPL of the default scene lies on a square (z = 4, 10 or 12)
    v = g["vpl_s0_n512"].view(np.float32)
    z = v[v[:, 3] != 0][:, 2]
    assert np.abs(z[:, None] - np.array([4.0, 10.0, 12.0])[None]).min(axis=1).max() < 1e-5


def test_bidir_image_golden(oracle_sep, scene_dirs):
    g = np.load(os.path.join(G, "golden_bidir.npz"))
    sc = oracle_sep.load_scene_dir(scene_dirs["bidir"], "bidir")
    out = oracle_sep.render("bidir", 512, 512, SEED_SETS[0], sc, want_rng=False, want_accum=False)
    assert hashlib.sha256(out["image"].tobytes()).digest() == g["img_s0_sha256"].tobytes()
    for ri, row in enumerate(g["rows"]):
        o2 = oracle_sep.render("bidir", 512, 512, SEED_SETS[1], sc, rows=(int(row), int(row) + 1), want_rng=False)
        assert np.array_equal(o2["image"][row], g["img_s1_rows"][ri]), int(row)
    # N_VLP given on the command line (argv[3]): 700 and the degenerate 96
    w, h = (int(x) for x in g["img_n700_size"])
    out = oracle_sep.render("bidir", w, h, SEED_SETS[0], sc, n_vlp=700, want_rng=False, want_accum=False)
    assert hashlib.sha256(out["image"].tobytes()).digest() == g["img_n700_sha256"].tobytes()
    w, h = (int(x) for x in g["img_n96_size"])
    out = oracle_sep.render("bidir", w, h, SEED_SETS[0], sc, n_vlp=96, want_rng=False, want_accum=False)
    assert np.array_equal(out["image"], g["img_n96"])
    host = json.loads(bytes(g["host_json"]).decode())["bidir"]
    assert sc["triangles"].shape[0] == host["ntriangles"] and sc["lights"].shape[0] == host["nlights"]
    assert int(host["vpl_print"]) == 512 * host["nlights"]


def test_sample_blocks_definition(oracle_sep, scene_dirs):
    """Sample-range sharding as the oracle states it (oracle.h): R = 1 is the plain render; block 0 walks the reference's
    own stream; the blocks' float buffers sum to a frame with alpha 255 that matches the unsharded one statistically."""
    sc = oracle_sep.load_scene_dir(scene_dirs["lmem"], "lmem")
    rows = (344, 352)
    full = oracle_sep.render("lmem", 512, 512, SEED_SETS[0], sc, rows=rows)
    one = oracle_sep.render("lmem", 512, 512, SEED_SETS[0], sc, rows=rows, sample_block=0, sample_blocks=1)
    assert np.array_equal(full["accum"].view(np.uint32), one["accum"].view(np.uint32))
    parts = [oracle_sep.render("lmem", 512, 512, SEED_SETS[0], sc, rows=rows, sample_block=b, sample_blocks=4) for b in range(4)]
    short = oracle_sep.render("lmem", 512, 512, SEED_SETS[0], sc, rows=rows, spp=16)
    assert np.array_equal(parts[0]["rng_state"], short["rng_state"])
    assert not np.array_equal(parts[1]["rng_state"], parts[2]["rng_state"])
    total = sum(p["accum"][rows[0]:rows[1]] for p in parts)
    assert (total[..., 3] == 255.0).all()
    diff = np.clip(np.trunc(total[..., :3]), 0, 255) - np.clip(np.trunc(full["accum"][rows[0]:rows[1], :, :3]), 0, 255)
    assert abs(diff.mean()) < 0.5 and np.sqrt((diff ** 2).mean()) < 14.0
    with pytest.raises(ValueError):
        oracle_sep.render("lmem", 64, 64, SEED_SETS[0], sc, sample_block=0, sample_blocks=3)
