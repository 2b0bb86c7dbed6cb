"""ctypes access to the CPU oracle (oracle/oracle.c) — TEST INFRASTRUCTURE ONLY.

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference legs.
The product package never imports this module.

    lib = OracleLib(contract=1)          # 1: FMA policy (bit-exact target of the CUDA path), 0: separate
    out = lib.render("base", 64, 64, (1, 2, 3, 4), scene_dict)
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")
VARIANTS = {"base": 0, "lmem": 1, "nodof": 2, "grid": 3, "bidir": 4, "vlpgrid": 5}


def build(force=False):
    """Compile the oracle shared libraries with gcc (seconds)."""
    need = force or not all(os.path.exists(os.path.join(BUILD, n)) for n in ("liboracle.so", "liboracle_fma.so", "oracle_cli"))
    if need:
        subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])


def cpu_has_fma():
    try:
        return " fma " in open("/proc/cpuinfo").read()
    except OSError:
        return False


class oracle_counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("samples", "rays", "shadow_rays", "tri_tests", "cells_visited", "prim_tests")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class oracle_job(C.Structure):
    _fields_ = [
        ("variant", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32),
        ("row_begin", C.c_int32), ("row_end", C.c_int32),
        ("seeds", C.c_uint32 * 4), ("spheres", C.c_int32 * 9), ("squares", C.c_int32 * 9),
        ("triangles", C.POINTER(C.c_float)), ("ntriangles", C.c_int32),
        ("lights", (C.c_float * 4) * 5), ("nlights", C.c_int32),
        ("cam_up", C.c_float * 4), ("cam_right", C.c_float * 4), ("eye_offset", C.c_float * 4),
        ("box_min", C.c_float * 4), ("box_max", C.c_float * 4), ("grid_res", C.c_int32 * 4), ("cell_size", C.c_float * 4),
        ("cell_start", C.POINTER(C.c_uint32)), ("cell_refs", C.POINTER(C.c_uint32)),
        ("nthreads", C.c_int32),
        ("vpls", C.POINTER(C.c_float)), ("nvpl", C.c_int32),
        ("sample_block", C.c_int32), ("sample_blocks", C.c_int32),
    ]


class OracleLib:
    def __init__(self, contract=1):
        build()
        if contract and not cpu_has_fma():
            raise RuntimeError("this CPU has no FMA instruction; liboracle_fma.so cannot run here")
        self.contract = int(bool(contract))
        self.lib = C.CDLL(os.path.join(BUILD, "liboracle_fma.so" if contract else "liboracle.so"))
        L = self.lib
        L.oracle_render.restype = C.c_int
        L.oracle_render.argtypes = [C.POINTER(oracle_job), C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(oracle_counters)]
        L.oracle_light_tracer.restype = C.c_int
        L.oracle_light_tracer.argtypes = [C.POINTER(oracle_job), C.c_int, C.c_void_p, C.c_void_p, C.POINTER(oracle_counters)]
        L.oracle_contract_mode.restype = C.c_int
        L.oracle_threads_used.restype = C.c_int
        L.oracle_randomize_id.restype = C.c_uint32
        L.oracle_randomize_id.argtypes = [C.c_uint32]
        L.oracle_build_grid.restype = C.c_uint64
        L.oracle_trace_ray.restype = C.c_int
        L.oracle_trace_rays.restype = C.c_int
        L.oracle_trace_rays.argtypes = [C.POINTER(oracle_job), C.c_int] + [C.c_void_p] * 7
        L.oracle_save_pam.restype = C.c_int
        L.oracle_save_pam.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p]
        assert L.oracle_contract_mode() == self.contract

    # ---- host-side restatements -------------------------------------------------------------
    def camera(self):
        f, u, r, e = [(C.c_float * 4)() for _ in range(4)]
        self.lib.oracle_camera(f, u, r, e)
        return {k: np.array(v[:], np.float32) for k, v in (("cam_forward", f), ("cam_up", u), ("cam_right", r), ("eye_offset", e))}

    def parse_array(self, path):
        a = (C.c_int32 * 9)()
        n = self.lib.oracle_parse_array(path.encode(), a)
        if n < 0:
            raise FileNotFoundError(path)
        return np.array(a[:], np.int32), n

    def parse_triangles(self, path, max_triangles):
        buf = np.zeros((max_triangles, 12), np.float32)
        mn, mx = (C.c_float * 4)(), (C.c_float * 4)()
        n = self.lib.oracle_parse_triangles(path.encode(), buf.ctypes.data_as(C.c_void_p), max_triangles, mn, mx)
        if n < 0:
            raise FileNotFoundError(path)
        return buf[:n].copy(), np.array(mn[:], np.float32), np.array(mx[:], np.float32)

    def parse_lights(self, path):
        l = ((C.c_float * 4) * 5)()
        n = self.lib.oracle_parse_lights(path.encode(), l)
        if n < 0:
            raise FileNotFoundError(path)
        return np.array([[l[i][k] for k in range(4)] for i in range(n)], np.float32).reshape(n, 4)

    def load_scene_dir(self, path, variant, max_triangles=None):
        if max_triangles is None:
            max_triangles = 65536 if variant == "grid" else 512
        sq = "planes.txt" if variant == "nodof" and os.path.exists(os.path.join(path, "planes.txt")) else "squares.txt"
        tris, mn, mx = self.parse_triangles(os.path.join(path, "triangles.txt"), max_triangles)
        return {"spheres": self.parse_array(os.path.join(path, "spheres.txt"))[0],
                "squares": self.parse_array(os.path.join(path, sq))[0],
                "triangles": tris, "lights": self.parse_lights(os.path.join(path, "lights.txt")),
                "box_min": mn, "box_max": mx}

    def grid_dims(self, box_min, box_max, ntriangles, modifier=3.0):
        res, cell = (C.c_int32 * 4)(), (C.c_float * 4)()
        self.lib.oracle_grid_dims((C.c_float * 4)(*box_min), (C.c_float * 4)(*box_max), int(ntriangles), C.c_float(modifier), res, cell)
        return np.array(res[:], np.int32), np.array(cell[:], np.float32)

    def build_grid(self, tris, box_min, res, cell, cap=62):
        tris = np.ascontiguousarray(tris, np.float32)
        ncells = int(res[0]) * int(res[1]) * int(res[2])
        start = np.zeros(ncells + 1, np.uint32)
        a = (tris.ctypes.data_as(C.c_void_p), C.c_int(tris.shape[0]), (C.c_float * 4)(*box_min), (C.c_int32 * 4)(*[int(x) for x in res]),
             (C.c_float * 4)(*cell), C.c_int(cap))
        total = self.lib.oracle_build_grid(*a, start.ctypes.data_as(C.c_void_p), None)
        refs = np.zeros(max(int(total), 1), np.uint32)
        self.lib.oracle_build_grid(*a, start.ctypes.data_as(C.c_void_p), refs.ctypes.data_as(C.c_void_p))
        return start, refs[: int(total)]

    def vlp_bounds(self, vpl):
        vpl = np.ascontiguousarray(vpl, np.float32).reshape(-1, 4)
        lo, hi = (C.c_float * 4)(), (C.c_float * 4)()
        self.lib.oracle_vlp_bounds(vpl.ctypes.data_as(C.c_void_p), C.c_int(vpl.shape[0]), lo, hi)
        return np.array(lo[:], np.float32), np.array(hi[:], np.float32)

    def build_vlp_grid(self, vpl, box_min, res, cell, cap=62):
        vpl = np.ascontiguousarray(vpl, np.float32).reshape(-1, 4)
        ncells = int(res[0]) * int(res[1]) * int(res[2])
        start = np.zeros(ncells + 1, np.uint32)
        a = (vpl.ctypes.data_as(C.c_void_p), C.c_int(vpl.shape[0]), (C.c_float * 4)(*box_min), (C.c_int32 * 4)(*[int(x) for x in res]),
             (C.c_float * 4)(*cell), C.c_int(cap))
        self.lib.oracle_build_vlp_grid.restype = C.c_uint64
        total = self.lib.oracle_build_vlp_grid(*a, start.ctypes.data_as(C.c_void_p), None)
        refs = np.zeros(max(int(total), 1), np.uint32)
        self.lib.oracle_build_vlp_grid(*a, start.ctypes.data_as(C.c_void_p), refs.ctypes.data_as(C.c_void_p))
        return start, refs[: int(total)]

    def save_pam(self, path, image):
        img = np.ascontiguousarray(image, np.uint8)
        return self.lib.oracle_save_pam(path.encode(), img.shape[1], img.shape[0], img.ctypes.data_as(C.c_void_p))

    # ---- device-side restatement ------------------------------------------------------------
    def rng_kat(self, seeds, gid, nsteps):
        f = np.zeros(2 * nsteps, np.float32)
        u = np.zeros(2 * nsteps, np.uint32)
        st = np.zeros(4, np.uint32)
        self.lib.oracle_rng_kat((C.c_uint32 * 4)(*seeds), C.c_uint32(gid), nsteps, f.ctypes.data_as(C.c_void_p),
                                u.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p))
        return f, u, st

    def trace_ray(self, carry, o, d, t, spheres, squares, tris):
        tris = np.ascontiguousarray(tris, np.float32)
        tt = C.c_float(t)
        n = (C.c_float * 3)()
        m = self.lib.oracle_trace_ray(int(carry), (C.c_float * 3)(*o), (C.c_float * 3)(*d), C.byref(tt), n,
                                      (C.c_int32 * 9)(*[int(x) for x in spheres]), (C.c_int32 * 9)(*[int(x) for x in squares]),
                                      tris.ctypes.data_as(C.c_void_p), int(tris.shape[0]))
        return m, tt.value, np.array(n[:], np.float32)

    @staticmethod
    def _fill_scene(J, seeds, scene):
        """Scene + seeds part of an oracle_job; returns the arrays that must stay alive while J is used."""
        J.seeds[:] = [int(s) & 0xFFFFFFFF for s in seeds]
        J.spheres[:] = [int(v) for v in scene["spheres"]]
        J.squares[:] = [int(v) for v in scene["squares"]]
        tris = np.ascontiguousarray(scene["triangles"], np.float32).reshape(-1, 12)
        J.triangles = tris.ctypes.data_as(C.POINTER(C.c_float))
        J.ntriangles = tris.shape[0]
        lights = np.asarray(scene["lights"], np.float32).reshape(-1, 4)
        J.nlights = lights.shape[0]
        for i in range(J.nlights):
            for k in range(4):
                J.lights[i][k] = float(lights[i, k])
        return tris

    def _fill_grid(self, J, tris, scene, grid, modifier):
        """Triangle grid part of an oracle_job.  `grid`: {"box_min", "box_max", "res", "cell_size"[, "csr"]}; None sizes it as the
        reference host does (scene box, CELL_SIZE_MODIFIER `modifier`).  The binning is stored back into `grid` as "csr", so
        callers that keep `grid` reuse it.  Returns the arrays that must stay alive while J is used."""
        if grid is None:
            res, cell = self.grid_dims(scene["box_min"], scene["box_max"], tris.shape[0], modifier)
            grid = {"box_min": scene["box_min"], "box_max": scene["box_max"], "res": res, "cell_size": cell}
        if "csr" in grid:
            start, refs = grid["csr"]
        else:
            start, refs = self.build_grid(tris, grid["box_min"], grid["res"], grid["cell_size"])
            grid["csr"] = (start, refs)
        if refs.size == 0:
            refs = np.zeros(1, np.uint32)
        J.box_min[:] = [float(x) for x in grid["box_min"]]; J.box_max[:] = [float(x) for x in grid["box_max"]]
        J.grid_res[:] = [int(x) for x in grid["res"]]; J.cell_size[:] = [float(x) for x in grid["cell_size"]]
        J.cell_start = start.ctypes.data_as(C.POINTER(C.c_uint32))
        J.cell_refs = refs.ctypes.data_as(C.POINTER(C.c_uint32))
        return start, refs

    def trace_rays(self, variant, origins, dirs, t_in, scene, grid=None, modifier=3.0):
        """TraceRay on single rays (oracle_trace_rays): variant "base" (t reset per call), "lmem" (carried t) or "grid"
        (lmem semantics, triangles through the uniform grid; `grid` as for render).  -> dict of material, t, normal,
        cells (grid cells visited) and tests (Moller-Trumbore tests started), one entry per ray."""
        J = oracle_job()
        J.variant = VARIANTS[variant]
        tris = self._fill_scene(J, (0, 0, 0, 0), scene)
        keep = self._fill_grid(J, tris, scene, grid, modifier) if variant == "grid" else None
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(t_in, np.float32).reshape(-1).copy()
        n = o.shape[0]
        if d.shape[0] != n or t.shape[0] != n:
            raise ValueError("trace_rays: origins, dirs and t_in must describe the same number of rays")
        m = np.zeros(n, np.int32)
        nrm = np.zeros((n, 3), np.float32)
        cells = np.zeros(n, np.uint32)
        tests = np.zeros(n, np.uint32)
        vp = C.c_void_p
        rc = self.lib.oracle_trace_rays(C.byref(J), int(n), o.ctypes.data_as(vp), d.ctypes.data_as(vp), t.ctypes.data_as(vp),
                                        m.ctypes.data_as(vp), nrm.ctypes.data_as(vp), cells.ctypes.data_as(vp), tests.ctypes.data_as(vp))
        del tris, keep
        if rc:
            raise ValueError("oracle_trace_rays rejected the job")
        return {"m": m, "t": t, "n": nrm, "cells": cells, "tests": tests}

    def light_tracer(self, seeds, scene, n_vlp=512, want_rng=False):
        """Kernel lightTracer (bidirectionalpathtracer.ocl:280-326): -> (n_vlp*nlights, 4) float32 VPL buffer."""
        J = oracle_job()
        tris = self._fill_scene(J, seeds, scene)
        vpl = np.zeros((n_vlp * J.nlights, 4), np.float32)
        rng = np.zeros((n_vlp, 4), np.uint32) if want_rng else None
        cnt = oracle_counters()
        rc = self.lib.oracle_light_tracer(C.byref(J), int(n_vlp), vpl.ctypes.data_as(C.c_void_p),
                                          rng.ctypes.data_as(C.c_void_p) if want_rng else None, C.byref(cnt))
        del tris
        if rc:
            raise ValueError("oracle_light_tracer rejected the job")
        return (vpl, rng) if want_rng else vpl

    def metropolis_light_tracer(self, seeds, scene, n_paths=512, rounds=8):
        """FIX-mode lightTracer + MetropolisLightTracer -> (seed paths (n*nl, 20) uint32, VPLs (4*n*nl, 4) float32)."""
        J = oracle_job()
        self._fill_scene(J, seeds, scene)
        paths = np.zeros((n_paths * J.nlights, 20), np.uint32)
        vpl = np.zeros((4 * n_paths * J.nlights, 4), np.float32)
        self.lib.oracle_metropolis_light_tracer.restype = C.c_int
        rc = self.lib.oracle_metropolis_light_tracer(C.byref(J), int(n_paths), int(rounds), paths.ctypes.data_as(C.c_void_p), vpl.ctypes.data_as(C.c_void_p))
        if rc:
            raise ValueError("oracle_metropolis_light_tracer rejected the job")
        return paths, vpl

    def metropolis_mutate(self, seeds, scene, gid, origin, path, rounds):
        """Mutate x rounds on one path (20 uint32 words, the reference's Path layout) -> mutated path."""
        J = oracle_job()
        self._fill_scene(J, seeds, scene)
        p = np.ascontiguousarray(path, np.uint32).copy()
        o = (C.c_float * 3)(*[float(x) for x in origin])
        self.lib.oracle_metropolis_mutate.restype = C.c_int
        if self.lib.oracle_metropolis_mutate(C.byref(J), C.c_uint32(int(gid)), o, p.ctypes.data_as(C.c_void_p), int(rounds)):
            raise ValueError("oracle_metropolis_mutate rejected the job")
        return p

    def render(self, variant, width, height, seeds, scene, spp=64, rows=None, cam=None, grid=None, want_accum=True,
               want_rng=True, nthreads=0, modifier=3.0, vpls=None, n_vlp=512, sample_block=0, sample_blocks=0):
        """scene: dict with spheres, squares, triangles (n,12), lights (nl,4) [, box_min, box_max].
        bidir: `vpls` (n,4) is the lightTracer buffer; None runs light_tracer(seeds, scene, n_vlp) first, as the
        reference host does (CLSuperBidirectionalPathTracer.c:370-375: same seeds for both kernels)."""
        J = oracle_job()
        J.variant = VARIANTS[variant]
        J.width, J.height, J.spp = width, height, spp
        J.sample_block, J.sample_blocks = int(sample_block), int(sample_blocks)
        if rows is not None:
            J.row_begin, J.row_end = rows
        tris = self._fill_scene(J, seeds, scene)
        if variant in ("bidir", "vlpgrid"):
            if vpls is None:
                vpls = self.light_tracer(seeds, scene, n_vlp)
            vpls = np.ascontiguousarray(vpls, np.float32).reshape(-1, 4)
            J.vpls = vpls.ctypes.data_as(C.POINTER(C.c_float))
            J.nvpl = vpls.shape[0]
        cam = cam or self.camera()
        J.cam_up[:] = list(cam["cam_up"]); J.cam_right[:] = list(cam["cam_right"]); J.eye_offset[:] = list(cam["eye_offset"])
        keep = None
        if variant == "vlpgrid":
            # `grid`: the VLP grid {"box_min", "res", "cell_size", "csr": (start, refs)}; None builds it as the reference host
            # would (bounds of the buffer, its grid formula with `modifier`, initVLPsGrid)
            if grid is None:
                lo, hi = self.vlp_bounds(vpls)
                res, cell = self.grid_dims(lo, hi, vpls.shape[0], modifier)
                grid = {"box_min": lo, "res": res, "cell_size": cell, "csr": self.build_vlp_grid(vpls, lo, res, cell)}
            start, refs = grid["csr"]
            if refs.size == 0:
                refs = np.zeros(1, np.uint32)
            keep = (start, refs)
            J.box_min[:] = [float(x) for x in grid["box_min"]]
            J.grid_res[:] = [int(x) for x in grid["res"]]; J.cell_size[:] = [float(x) for x in grid["cell_size"]]
            J.cell_start = start.ctypes.data_as(C.POINTER(C.c_uint32))
            J.cell_refs = refs.ctypes.data_as(C.POINTER(C.c_uint32))
        if variant == "grid":
            keep = self._fill_grid(J, tris, scene, grid, modifier)
        J.nthreads = nthreads
        img = np.zeros((height, width, 4), np.uint8)
        acc = np.zeros((height, width, 4), np.float32) if want_accum else None
        items = width * height * (64 if variant == "nodof" else 1)
        rng = np.zeros((items, 4), np.uint32) if want_rng else None
        cnt = oracle_counters()
        rc = self.lib.oracle_render(C.byref(J), img.ctypes.data_as(C.c_void_p), acc.ctypes.data_as(C.c_void_p) if want_accum else None,
                                    rng.ctypes.data_as(C.c_void_p) if want_rng else None, C.byref(cnt))
        if rc:
            raise ValueError("oracle_render rejected the job")
        del keep
        out = {"image": img, "accum": acc, "rng_state": rng, "counters": cnt.as_dict(), "threads": int(self.lib.oracle_threads_used())}
        if variant in ("bidir", "vlpgrid"):
            out["vpls"] = vpls
        if variant == "vlpgrid":
            out["vlp_grid"] = grid
        return out
