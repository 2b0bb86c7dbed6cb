"""ctypes access to the path oracle (oracle_paths/oracle_paths.c) — TEST INFRASTRUCTURE ONLY.

Importable only from tests/ and tools/; the product package never imports it.

    lib = PathOracle(contract=1)            # 1: FMA policy (bit-exact target of the CUDA path), 0: separate
    out = lib.render_bounces("base", 64, 64, (1, 2, 3, 4), scene_dict, bounces=2)
    rgb, pc = lib.path_samples(scene_dict, o, d, rng_states, bounces=1)

Scene dicts, grids and cameras are those of oracle.pyoracle.OracleLib, whose helpers (scene loading, grid binning) this
class inherits.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle.pyoracle import VARIANTS, OracleLib, cpu_has_fma, oracle_counters, oracle_job

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")


def build(force=False):
    """Compile the path oracle with gcc (seconds)."""
    need = force or not all(os.path.exists(os.path.join(BUILD, n)) for n in ("liboracle_paths.so", "liboracle_paths_fma.so"))
    if need:
        subprocess.check_call(["make", "-s", "-C", HERE])


class oracle_path_counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("bounce_rays", "rr_terminations", "tmin_rejections", "disk_exhausted")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class PathOracle(OracleLib):
    def __init__(self, contract=1):
        super().__init__(contract)
        build()
        self.plib = C.CDLL(os.path.join(BUILD, "liboracle_paths_fma.so" if contract else "liboracle_paths.so"))
        P = self.plib
        vp = C.c_void_p
        P.oracle_render_bounces.restype = C.c_int
        P.oracle_render_bounces.argtypes = [C.POINTER(oracle_job), C.c_int, vp, vp, vp, C.POINTER(oracle_counters),
                                            C.POINTER(oracle_path_counters)]
        P.oracle_path_sample.restype = C.c_int
        P.oracle_path_sample.argtypes = [C.POINTER(oracle_job), vp, vp, vp, C.c_int, C.c_int, vp, C.POINTER(oracle_counters),
                                         C.POINTER(oracle_path_counters)]
        P.oracle_path_samples.restype = C.c_int
        P.oracle_path_samples.argtypes = [C.POINTER(oracle_job), C.c_int, vp, vp, vp, C.c_int, C.c_int, vp,
                                          C.POINTER(oracle_path_counters)]
        P.oracle_contract_mode.restype = C.c_int
        assert P.oracle_contract_mode() == self.contract

    def _path_job(self, variant, scene, seeds=(0, 0, 0, 0), grid=None, modifier=3.0):
        J = oracle_job()
        J.variant = VARIANTS[variant]
        tris = self._fill_scene(J, seeds, scene)
        keep = self._fill_grid(J, tris, scene, grid, modifier) if variant == "grid" else None
        return J, (tris, keep)

    def render_bounces(self, variant, width, height, seeds, scene, bounces, spp=64, rows=None, cam=None, grid=None,
                       nthreads=0, modifier=3.0, sample_block=0, sample_blocks=0):
        """oracle_render_bounces -> dict like OracleLib.render (image, accum, rng_state, counters) plus path_counters."""
        J, keep = self._path_job(variant, scene, seeds, grid, modifier)
        J.width, J.height, J.spp = width, height, spp
        J.sample_block, J.sample_blocks = int(sample_block), int(sample_blocks)
        if rows is not None:
            J.row_begin, J.row_end = rows
        cam = cam or self.camera()
        J.cam_up[:] = list(cam["cam_up"]); J.cam_right[:] = list(cam["cam_right"]); J.eye_offset[:] = list(cam["eye_offset"])
        J.nthreads = nthreads
        img = np.zeros((height, width, 4), np.uint8)
        acc = np.zeros((height, width, 4), np.float32)
        rng = np.zeros((width * height, 4), np.uint32)
        cnt, pc = oracle_counters(), oracle_path_counters()
        rc = self.plib.oracle_render_bounces(C.byref(J), int(bounces), img.ctypes.data_as(C.c_void_p), acc.ctypes.data_as(C.c_void_p),
                                             rng.ctypes.data_as(C.c_void_p), C.byref(cnt), C.byref(pc))
        del keep
        if rc:
            raise ValueError("oracle_render_bounces rejected the job")
        return {"image": img, "accum": acc, "rng_state": rng, "counters": cnt.as_dict(), "path_counters": pc.as_dict()}

    def path_samples(self, scene, o, d, rng_states, bounces, rr=True, variant="base", grid=None, nthreads=0):
        """n paths from o along d, one per RNG state (n x 4 uint32, advanced in place) -> (L (n, 3) float32, path counters)."""
        J, keep = self._path_job(variant, scene, grid=grid)
        J.nthreads = nthreads
        st = np.ascontiguousarray(rng_states, np.uint32).reshape(-1, 4)
        n = st.shape[0]
        out = np.zeros((n, 3), np.float32)
        of = np.ascontiguousarray(o, np.float32).reshape(3)
        df = np.ascontiguousarray(d, np.float32).reshape(3)
        pc = oracle_path_counters()
        rc = self.plib.oracle_path_samples(C.byref(J), int(n), of.ctypes.data_as(C.c_void_p), df.ctypes.data_as(C.c_void_p),
                                           st.ctypes.data_as(C.c_void_p), int(bounces), int(bool(rr)), out.ctypes.data_as(C.c_void_p),
                                           C.byref(pc))
        del keep
        if rc:
            raise ValueError("oracle_path_samples rejected the job")
        if st is not rng_states:
            np.asarray(rng_states)[...] = st.reshape(np.shape(rng_states))
        return out, pc.as_dict()


__all__ = ["PathOracle", "build", "cpu_has_fma", "oracle_path_counters"]
