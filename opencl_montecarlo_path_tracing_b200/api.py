"""Python face of the CLSuperPathTracer drop-in (thin: everything real happens behind the C ABI).

    scene = load_scene_dir("scenes/_gen/base", variant="base")      # the reference's .txt files
    with Renderer(device=0) as r:
        r.set_scene(scene)
        out = r.render(variant="base", width=512, height=512, seeds=(1, 2, 3, 4))
        out.image  # (H, W, 4) uint8 == what the reference writes into result.ppm

Host-side steps (parsing, camera, grid sizing) call libpthost.so, the same C code the drop-in
executables use; rendering calls libptcuda.so.  No CPU fallback exists.
"""
import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import PT_ARITH, PT_KERNEL, PT_SCENE_MEM, PT_VARIANT, pt_camera, pt_counters, pt_grid, pt_render_params, pt_scene


class PtError(RuntimeError):
    pass


def _check(rc, what):
    if rc:
        raise PtError("%s failed: %s" % (what, _lib.cuda_lib().pt_last_error().decode()))


@dataclass
class Scene:
    spheres: np.ndarray                      # int32[9]
    squares: np.ndarray                      # int32[9]
    triangles: np.ndarray                    # float32[n, 12]  (v0 v1 v2 as float4, w = 0)
    lights: np.ndarray                       # float32[nlights, 4]
    box_min: np.ndarray = field(default_factory=lambda: np.zeros(4, np.float32))
    box_max: np.ndarray = field(default_factory=lambda: np.zeros(4, np.float32))

    @property
    def ntriangles(self):
        return int(self.triangles.shape[0])

    def to_c(self):
        s = pt_scene()
        s.spheres[:] = [int(v) for v in self.spheres]
        s.squares[:] = [int(v) for v in self.squares]
        self._tri_keepalive = np.ascontiguousarray(self.triangles, dtype=np.float32).reshape(-1)
        s.triangles = self._tri_keepalive.ctypes.data_as(C.POINTER(C.c_float))
        s.ntriangles = self.ntriangles
        s.nlights = int(self.lights.shape[0])
        for i in range(s.nlights):
            for k in range(4):
                s.lights[i][k] = float(self.lights[i, k])
        return s


def default_max_triangles(variant):
    """MAX_TRIANGLES of the reference hosts (CLSuperPathTracer.c:14; trianglegrid :15)."""
    return 65536 if variant == "grid" else 512


def load_scene_dir(path, variant="base", max_triangles=None, triangles_file="triangles.txt"):
    """Parse spheres.txt / squares.txt (planes.txt for nodof) / triangles.txt / lights.txt of a directory
    with the drop-in's own C parsers (reference semantics incl. the feof() quirks)."""
    h = _lib.host_lib()
    if max_triangles is None:
        max_triangles = default_max_triangles(variant)

    def bitmap(name):
        arr = (C.c_int32 * 9)()
        if h.pth_parse_bitmap(os.path.join(path, name).encode(), arr) < 0:
            raise FileNotFoundError(os.path.join(path, name))
        return np.array(arr[:], dtype=np.int32)

    spheres = bitmap("spheres.txt")
    sq_name = "squares.txt"
    if variant == "nodof" and os.path.exists(os.path.join(path, "planes.txt")):
        sq_name = "planes.txt"
    squares = bitmap(sq_name)
    ptr = C.POINTER(C.c_float)()
    bmin, bmax = (C.c_float * 4)(), (C.c_float * 4)()
    n = h.pth_parse_triangles(os.path.join(path, triangles_file).encode(), max_triangles, C.byref(ptr), bmin, bmax)
    if n < 0:
        raise FileNotFoundError(os.path.join(path, triangles_file))
    tris = np.ctypeslib.as_array(ptr, shape=(max(n, 1) * 12,))[: n * 12].copy().reshape(n, 12)
    C.CDLL(None).free(ptr)
    lights_c = ((C.c_float * 4) * 5)()
    nl = h.pth_parse_lights(os.path.join(path, "lights.txt").encode(), C.byref(lights_c), 0)
    if nl < 0:
        raise FileNotFoundError(os.path.join(path, "lights.txt"))
    lights = np.array([[lights_c[i][k] for k in range(4)] for i in range(nl)], dtype=np.float32).reshape(nl, 4)
    return Scene(spheres, squares, tris, lights, np.array(bmin[:], np.float32), np.array(bmax[:], np.float32))


def camera():
    """The four camera kernel arguments (CLSuperPathTracer.c:236-243)."""
    cam = pt_camera()
    _lib.host_lib().pth_camera(C.byref(cam))
    return cam


def grid_dims(scene, cell_size_modifier=3.0):
    g = pt_grid()
    bmin = (C.c_float * 4)(*[float(v) for v in scene.box_min])
    bmax = (C.c_float * 4)(*[float(v) for v in scene.box_max])
    _lib.host_lib().pth_grid_dims(bmin, bmax, scene.ntriangles, C.c_float(cell_size_modifier), C.byref(g))
    return g


def vlp_grid_dims(vmin, vmax, n_vlp, cell_size_modifier=3.0):
    """Resolution / cell size of the VLP grid from its bounding box (CLSuperMetropolisPathTracer.c:628-636: the triangle
    grid's formula with the VLP count)."""
    g = pt_grid()
    bmin = (C.c_float * 4)(*[float(v) for v in vmin])
    bmax = (C.c_float * 4)(*[float(v) for v in vmax])
    _lib.host_lib().pth_grid_dims(bmin, bmax, int(n_vlp), C.c_float(cell_size_modifier), C.byref(g))
    return g


def save_pam(path, image):
    img = np.ascontiguousarray(image, dtype=np.uint8)
    hgt, wid = img.shape[:2]
    if _lib.host_lib().pth_save_pam(path.encode(), wid, hgt, img.ctypes.data_as(C.c_void_p)):
        raise PtError("error writing %s" % path)


def load_pam(path):
    """pamalign.h load_pam: -> (array (H, W, C') uint8/uint16, maxval); 3-channel files come back padded to 4."""
    img = _lib.pth_image()
    if _lib.host_lib().pth_load_pam(path.encode(), C.byref(img)):
        raise PtError("error reading %s" % path)
    try:
        stride = img.channels + (1 if img.channels == 3 else 0)
        dt = np.uint8 if img.depth == 8 else np.uint16
        n = img.width * img.height * stride
        arr = np.ctypeslib.as_array(C.cast(img.data, C.POINTER(C.c_uint8 if img.depth == 8 else C.c_uint16)), shape=(max(n, 1),))[:n]
        return arr.astype(dt).reshape(img.height, img.width, stride).copy(), int(img.maxval)
    finally:
        _lib.host_lib().pth_free_image(C.byref(img))


def save_ppm(path, image):
    img = np.ascontiguousarray(image, dtype=np.uint8)
    if _lib.host_lib().pth_save_ppm(path.encode(), img.shape[1], img.shape[0], img.ctypes.data_as(C.c_void_p)):
        raise PtError("error writing %s" % path)


def save_png(path, image):
    img = np.ascontiguousarray(image, dtype=np.uint8)
    if _lib.host_lib().pth_save_png(path.encode(), img.shape[1], img.shape[0], img.ctypes.data_as(C.c_void_p)):
        raise PtError("error writing %s" % path)


def import_obj(obj_path, triangles_txt_path, scale=1.0, translate=(0.0, 0.0, 0.0)):
    """Wavefront OBJ -> triangles.txt; returns the number of triangles written."""
    t = (C.c_float * 3)(*[float(x) for x in translate])
    n = _lib.host_lib().pth_import_obj(obj_path.encode(), triangles_txt_path.encode(), C.c_float(scale), t)
    if n < 0:
        raise PtError("error importing %s" % obj_path)
    return int(n)


@dataclass
class RenderResult:
    image: np.ndarray                 # (H, W, 4) uint8
    ms: float                         # device time of the launch (CUDA events)
    counters: dict
    accum: np.ndarray = None          # (H, W, 4) float32 if requested
    rng_state: np.ndarray = None      # (items, 4) uint32 if requested


def make_params(variant, width, height, seeds, spp=64, kernel="auto", scene_mem=None, arith="fma", rows=None,
                want_accum=False, want_rng=False, interleave=0, rank=0, nranks=1, cull=True, n_vlp=0, sample_block=0, sample_blocks=0,
                cluster_cull="auto", dead_rays="auto"):
    """dead_rays: "auto" / "elide" — shadow rays of triangle-material samples (their result is never used) are not traced;
    "trace" — every ray of the reference is traced and the work counters equal the reference's (include/ptcuda.h)."""
    p = pt_render_params()
    p.variant = PT_VARIANT[variant]
    p.width, p.height, p.spp = int(width), int(height), int(spp)
    if rows is not None:
        p.row_begin, p.row_end = int(rows[0]), int(rows[1])
    p.seeds[:] = [int(s) & 0xFFFFFFFF for s in seeds]
    p.kernel = PT_KERNEL[kernel]
    if scene_mem is None:
        scene_mem = "auto"
    p.scene_mem = PT_SCENE_MEM[scene_mem]
    p.arith = PT_ARITH[arith]
    p.want_accum, p.want_rng = int(bool(want_accum)), int(bool(want_rng))
    p.row_interleave, p.rank, p.nranks = int(interleave), int(rank), int(nranks)
    p.no_cull = 0 if cull else 1
    p.n_vlp = int(n_vlp)
    p.sample_block, p.sample_blocks = int(sample_block), int(sample_blocks)
    p.cluster_cull = {"auto": 0, "on": 1, "off": 2}[cluster_cull]
    p.dead_rays = {"auto": 0, "trace": 1, "elide": 2}[dead_rays]
    return p


class Renderer:
    """One pt_ctx: one CUDA device, one stream."""

    def __init__(self, device=0, stream=None):
        self._l = _lib.cuda_lib()
        if self._l.pt_device_count() <= 0:
            raise PtError("no CUDA device visible; libptcuda has no CPU fallback")
        self.ctx = self._l.pt_create_on_stream(device, C.c_void_p(stream)) if stream is not None else self._l.pt_create(device)
        if not self.ctx:
            raise PtError("pt_create failed: %s" % self._l.pt_last_error().decode())
        self.device = device
        self._scene = None
        self.cam = camera()

    def close(self):
        if self.ctx:
            self._l.pt_destroy(self.ctx)
            self.ctx = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def device_props(self):
        sm, khz = C.c_int(), C.c_int()
        self._l.pt_device_props(self.ctx, C.byref(sm), C.byref(khz))
        name = C.create_string_buffer(256)
        self._l.pt_device_name(self.ctx, name, 256)
        return {"name": name.value.decode(), "sm_count": sm.value, "clock_khz": khz.value}

    def set_scene(self, scene):
        self._scene = scene
        cs = scene.to_c()
        _check(self._l.pt_set_scene(self.ctx, C.byref(cs)), "pt_set_scene")

    def build_grid(self, grid):
        evt = self._l.pt_build_grid(self.ctx, C.byref(grid))
        if not evt:
            raise PtError("pt_build_grid failed: %s" % self._l.pt_last_error().decode())
        ms = self._l.pt_runtime_ms(evt)
        self._l.pt_release_event(evt)
        self._grid = grid
        return ms

    def read_grid_csr(self):
        total = C.c_uint64()
        _check(self._l.pt_read_grid_csr(self.ctx, None, None, C.byref(total)), "pt_read_grid_csr")
        g = self._grid
        ncells = g.res[0] * g.res[1] * g.res[2]
        start = np.zeros(ncells + 1, np.uint32)
        refs = np.zeros(max(int(total.value), 1), np.uint32)
        _check(self._l.pt_read_grid_csr(self.ctx, start.ctypes.data_as(C.POINTER(C.c_uint32)),
                                        refs.ctypes.data_as(C.POINTER(C.c_uint32)), None), "pt_read_grid_csr")
        return start, refs[: int(total.value)]

    def read_grid_cells(self):
        g = self._grid
        ncells = g.res[0] * g.res[1] * g.res[2]
        raw = np.zeros(ncells * 128, np.uint8)
        _check(self._l.pt_read_grid_cells(self.ctx, raw.ctypes.data_as(C.c_void_p), ncells), "pt_read_grid_cells")
        return raw.reshape(ncells, 128)

    # ---- bidirectional variant (CLSuperBidirectionalPathTracer): virtual point lights ----
    def light_tracer(self, seeds, n_vlp=512, arith="fma", wait=True):
        """Kernel lightTracer (CLSuperBidirectionalPathTracer.c:143-184): fills the context's VPL buffer, which the next
        variant="bidir" render gathers.  Returns the device time in ms (wait=False: only enqueues, returns None)."""
        s = (C.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in seeds])
        evt = self._l.pt_launch_lighttracer(self.ctx, int(n_vlp), s, PT_ARITH[arith])
        if not evt:
            raise PtError("pt_launch_lighttracer failed: %s" % self._l.pt_last_error().decode())
        if not wait:
            self._l.pt_release_event(evt)
            return None
        _check(self._l.pt_wait(evt), "pt_wait")
        ms = self._l.pt_runtime_ms(evt)
        self._l.pt_release_event(evt)
        return ms

    def metropolis_light_tracer(self, seeds, n_paths=512, rounds=8, arith="fma"):
        """Kernels lightTracer + MetropolisLightTracer of CLSuperMetropolisPathTracer(_vlpgrid) in FIX mode (include/ptcuda.h):
        fills the context's VPL buffer with 4*n_paths*nlights entries.  Returns (seed paths (n*nl, 20) uint32, VPLs (4*n*nl, 4))."""
        s = (C.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in seeds])
        evt = self._l.pt_launch_metropolis_lighttracer(self.ctx, int(n_paths), s, int(rounds), PT_ARITH[arith])
        if not evt:
            raise PtError("pt_launch_metropolis_lighttracer failed: %s" % self._l.pt_last_error().decode())
        _check(self._l.pt_wait(evt), "pt_wait")
        self._l.pt_release_event(evt)
        return self.read_metropolis_paths(mutated=False), self.read_vpls()

    def read_metropolis_paths(self, mutated=False):
        n = self._l.pt_read_metropolis_paths(self.ctx, None, 0, 0)
        if n < 0:
            raise PtError("pt_read_metropolis_paths failed: %s" % self._l.pt_last_error().decode())
        p = np.zeros((max(n, 1), 20), np.uint32)
        if self._l.pt_read_metropolis_paths(self.ctx, p.ctypes.data_as(C.POINTER(C.c_uint32)), max(n, 1), int(bool(mutated))) < 0:
            raise PtError("pt_read_metropolis_paths failed: %s" % self._l.pt_last_error().decode())
        return p[:n]

    def set_vpls(self, vpls):
        v = np.ascontiguousarray(vpls, np.float32).reshape(-1, 4)
        _check(self._l.pt_set_vpls(self.ctx, v.ctypes.data_as(C.POINTER(C.c_float)), v.shape[0]), "pt_set_vpls")

    def read_vpls(self):
        n = self._l.pt_read_vpls(self.ctx, None, 0)
        if n < 0:
            raise PtError("pt_read_vpls failed: %s" % self._l.pt_last_error().decode())
        v = np.zeros((max(n, 1), 4), np.float32)
        if self._l.pt_read_vpls(self.ctx, v.ctypes.data_as(C.POINTER(C.c_float)), max(n, 1)) < 0:
            raise PtError("pt_read_vpls failed: %s" % self._l.pt_last_error().decode())
        return v[:n]

    # ---- VLP bounding box / VLP grid (CLSuperMetropolisPathTracer_vlpgrid) on the context's VLP buffer ----
    def vlp_bounds(self):
        """reduceMinAndMax_lmem(+_nwg): -> (vmin[4], vmax[4]) float32."""
        lo, hi = (C.c_float * 4)(), (C.c_float * 4)()
        _check(self._l.pt_vlp_bounds(self.ctx, lo, hi), "pt_vlp_bounds")
        return np.array(lo[:], np.float32), np.array(hi[:], np.float32)

    def build_vlp_grid(self, grid):
        """initVLPsGrid on the VLP buffer; `grid` from vlp_grid_dims().  Returns the device time in ms."""
        evt = self._l.pt_build_vlp_grid(self.ctx, C.byref(grid))
        if not evt:
            raise PtError("pt_build_vlp_grid failed: %s" % self._l.pt_last_error().decode())
        ms = self._l.pt_runtime_ms(evt)
        self._l.pt_release_event(evt)
        self._vlp_grid = grid
        return ms

    def read_vlp_grid_csr(self):
        total = C.c_uint64()
        _check(self._l.pt_read_vlp_grid_csr(self.ctx, None, None, C.byref(total)), "pt_read_vlp_grid_csr")
        g = self._vlp_grid
        ncells = g.res[0] * g.res[1] * g.res[2]
        start = np.zeros(ncells + 1, np.uint32)
        refs = np.zeros(max(int(total.value), 1), np.uint32)
        _check(self._l.pt_read_vlp_grid_csr(self.ctx, start.ctypes.data_as(C.POINTER(C.c_uint32)),
                                            refs.ctypes.data_as(C.POINTER(C.c_uint32)), None), "pt_read_vlp_grid_csr")
        return start, refs[: int(total.value)]

    def read_vlp_grid_cells(self):
        g = self._vlp_grid
        ncells = g.res[0] * g.res[1] * g.res[2]
        raw = np.zeros(ncells * 128, np.uint8)
        _check(self._l.pt_read_vlp_grid_cells(self.ctx, raw.ctypes.data_as(C.c_void_p), ncells), "pt_read_vlp_grid_cells")
        return raw.reshape(ncells, 128)

    def set_bounces(self, bounces):
        """Diffuse bounces per path (0..15) for the following renders of this context (pt_set_bounces; DESIGN.md 5b)."""
        _check(self._l.pt_set_bounces(self.ctx, int(bounces)), "pt_set_bounces")

    def render(self, variant, width, height, seeds, read_image=True, samples=None, bounces=0, **kw):
        """Renders the frame in one launch, or with samples=(b, e) samples [b, e) of it as one range of a progression
        (include/ptcuda.h, "progressive rendering"): the last range gives the one-launch frame bit for bit, earlier ones a
        preview image.  accum / rng_state are read back when want_accum / want_rng are set.
        bounces: diffuse bounces per path with Russian roulette (include/ptcuda.h, DESIGN.md 5b); 0 is the reference.

            kw = dict(spp=256)
            for b, e in ((0, 16), (16, 64), (64, 256)):
                out = r.render("base", 1920, 1080, seeds, samples=(b, e), **kw)      # out.image: preview, then the frame
            # checkpoint after a range, and resume it later, in this or another Renderer with the same scene:
            cp = r.render("base", 1920, 1080, seeds, samples=(0, 16), want_accum=True, want_rng=True, **kw)
            r2.set_render_state("base", 1920, 1080, seeds, 16, cp.accum, cp.rng_state, **kw)
            out = r2.render("base", 1920, 1080, seeds, samples=(16, 256), **kw)
        """
        p = make_params(variant, width, height, seeds, **kw)
        self.set_bounces(bounces)
        if samples is None:
            evt = self._l.pt_launch_pathtracer(self.ctx, C.byref(self.cam), C.byref(p))
        else:
            evt = self._l.pt_launch_pathtracer_range(self.ctx, C.byref(self.cam), C.byref(p), int(samples[0]), int(samples[1]))
        if not evt:
            raise PtError("%s failed: %s" % ("pt_launch_pathtracer" if samples is None else "pt_launch_pathtracer_range",
                                             self._l.pt_last_error().decode()))
        image = None
        if read_image:
            ptr = self._l.pt_map_render(self.ctx, None)
            if not ptr:
                raise PtError("pt_map_render failed: %s" % self._l.pt_last_error().decode())
            image = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(height, width, 4)).copy()
        ms = self._l.pt_runtime_ms(evt)
        self._l.pt_release_event(evt)
        cnt = pt_counters()
        _check(self._l.pt_get_counters(self.ctx, C.byref(cnt)), "pt_get_counters")
        res = RenderResult(image=image, ms=ms, counters=cnt.as_dict())
        if p.want_accum:
            acc = np.zeros((height, width, 4), np.float32)
            _check(self._l.pt_read_accum(self.ctx, acc.ctypes.data_as(C.POINTER(C.c_float)), acc.size), "pt_read_accum")
            res.accum = acc
        if p.want_rng:
            items = width * height * (64 if variant == "nodof" else 1)
            st = np.zeros((items, 4), np.uint32)
            _check(self._l.pt_read_rng_state(self.ctx, st.ctypes.data_as(C.POINTER(C.c_uint32)), st.size), "pt_read_rng_state")
            res.rng_state = st
        return res

    def set_render_state(self, variant, width, height, seeds, samples_done, accum, rng_state, bounces=0, **kw):
        """Restores a progression saved after samples_done samples (accum (H, W, 4) float32 and rng_state (H*W, 4) uint32, as
        render(..., samples=(b, samples_done), want_accum=True, want_rng=True) returned them); keywords as for render().  The
        next render(..., samples=(samples_done, e)) with the same params continues it."""
        p = make_params(variant, width, height, seeds, **kw)
        acc = np.ascontiguousarray(accum, np.float32)
        st = np.ascontiguousarray(rng_state, np.uint32)
        if acc.size != width * height * 4 or st.size != width * height * 4:
            raise ValueError("set_render_state: accum and rng_state must hold width * height * 4 values each")
        self.set_bounces(bounces)
        _check(self._l.pt_set_render_state(self.ctx, C.byref(self.cam), C.byref(p), int(samples_done),
                                           acc.ctypes.data_as(C.POINTER(C.c_float)), st.ctypes.data_as(C.POINTER(C.c_uint32))),
               "pt_set_render_state")

    def render_device(self, variant, width, height, seeds, d_rgba8, d_accum=None, bounces=0, **kw):
        """Render into caller-owned device memory (raw pointers, e.g. torch tensors' data_ptr())."""
        p = make_params(variant, width, height, seeds, **kw)
        self.set_bounces(bounces)
        _check(self._l.pt_render_device(self.ctx, C.byref(self.cam), C.byref(p), C.c_void_p(d_rgba8),
                                        C.c_void_p(d_accum) if d_accum else None), "pt_render_device")

    def tonemap_device(self, d_accum, d_rgba8, width, height):
        _check(self._l.pt_tonemap_device(self.ctx, C.c_void_p(d_accum), C.c_void_p(d_rgba8), width, height), "pt_tonemap_device")

    def counters(self):
        cnt = pt_counters()
        _check(self._l.pt_get_counters(self.ctx, C.byref(cnt)), "pt_get_counters")
        return cnt.as_dict()

    def last_kernel(self):
        """Name of the kernel flavour the most recent render resolved to (what "auto" picked)."""
        k = self._l.pt_last_kernel(self.ctx)
        return {v: n for n, v in _lib.PT_KERNEL.items()}.get(k, str(k))

    def synchronize(self):
        _check(self._l.pt_synchronize(self.ctx), "pt_synchronize")

    def probe_trace(self, variant, origins, dirs, t_in, arith="fma", counts=False):
        """Device TraceRay on single rays -> (material, t, normal), plus (cells visited, triangle tests) with counts=True
        (include/ptcuda.h pt_probe_trace_counts)."""
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(t_in, np.float32).reshape(-1).copy()
        n = o.shape[0]
        if d.shape[0] != n or t.shape[0] != n:
            raise ValueError("probe_trace: origins, dirs and t_in must describe the same number of rays")
        m = np.zeros(n, np.int32)
        nrm = np.zeros((n, 3), np.float32)
        cells = np.zeros(n, np.uint32)
        tests = np.zeros(n, np.uint32)
        fp, up = C.POINTER(C.c_float), C.POINTER(C.c_uint32)
        _check(self._l.pt_probe_trace_counts(self.ctx, PT_VARIANT[variant], PT_ARITH[arith], n, o.ctypes.data_as(fp),
                                             d.ctypes.data_as(fp), t.ctypes.data_as(fp), m.ctypes.data_as(C.POINTER(C.c_int32)),
                                             nrm.ctypes.data_as(fp), cells.ctypes.data_as(up), tests.ctypes.data_as(up)),
               "pt_probe_trace")
        return (m, t, nrm, cells, tests) if counts else (m, t, nrm)

    def selftest_fastmath(self, npairs, seed=1):
        out = (C.c_uint64 * 3)()
        _check(self._l.pt_selftest_fastmath(self.ctx, int(npairs), int(seed), out), "pt_selftest_fastmath")
        return {"div_mismatches": int(out[0]), "sqrt_mismatches": int(out[1]), "pairs_tested": int(out[2])}

    def measure_peaks(self):
        """Measured FP32 / issue-slot peaks of this device (pt_measure_peaks)."""
        out = (C.c_double * 4)()
        _check(self._l.pt_measure_peaks(self.ctx, out), "pt_measure_peaks")
        return {"fp32_tflops": out[0], "ffma_gwarp_inst_per_s": out[1], "mixed_gwarp_inst_per_s": out[2], "mixed_kernel_ms": out[3]}

    def probe_rng(self, seeds, gid, nsteps):
        s = (C.c_uint32 * 4)(*[int(v) for v in seeds])
        out = np.zeros(2 * nsteps, np.float32)
        st = np.zeros(4, np.uint32)
        _check(self._l.pt_probe_rng(self.ctx, s, gid, nsteps, out.ctypes.data_as(C.POINTER(C.c_float)),
                                    st.ctypes.data_as(C.POINTER(C.c_uint32))), "pt_probe_rng")
        return out, st
