"""ctypes binding of the C ABI (include/ptcuda.h, include/pthost.h).

The shared libraries are built in-tree by `make -C opencl_montecarlo_path_tracing_b200/csrc`
(see __graft_entry__.build).  There is NO fallback: if libptcuda.so is missing or cannot be
loaded, every entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "lib")
BIN_DIR = os.path.join(_HERE, "bin")

PT_VARIANT = {"base": 0, "lmem": 1, "nodof": 2, "grid": 3, "bidir": 4, "vlpgrid": 5}
PT_KERNEL = {"mega": 0, "persistent": 1, "wavefront": 2, "auto": 3, "grid_tma": 4, "grid_stream": 5, "grid_pool": 6, "spec": 7, "grid_queue": 8, "grid_async": 9}
PT_SCENE_MEM = {"const": 0, "smem": 1, "auto": 2}
PT_ARITH = {"separate": 0, "fma": 1}


class pt_scene(C.Structure):
    _fields_ = [
        ("spheres", C.c_int32 * 9),
        ("squares", C.c_int32 * 9),
        ("triangles", C.POINTER(C.c_float)),
        ("ntriangles", C.c_int32),
        ("lights", (C.c_float * 4) * 5),
        ("nlights", C.c_int32),
    ]


class pt_camera(C.Structure):
    _fields_ = [
        ("cam_forward", C.c_float * 4),
        ("cam_up", C.c_float * 4),
        ("cam_right", C.c_float * 4),
        ("eye_offset", C.c_float * 4),
    ]


class pt_grid(C.Structure):
    _fields_ = [
        ("box_min", C.c_float * 4),
        ("box_max", C.c_float * 4),
        ("res", C.c_int32 * 4),
        ("cell_size", C.c_float * 4),
        ("max_refs_per_cell", C.c_int32),
    ]


class pt_render_params(C.Structure):
    _fields_ = [
        ("variant", C.c_int32),
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("spp", C.c_int32),
        ("row_begin", C.c_int32),
        ("row_end", C.c_int32),
        ("seeds", C.c_uint32 * 4),
        ("kernel", C.c_int32),
        ("scene_mem", C.c_int32),
        ("arith", C.c_int32),
        ("want_accum", C.c_int32),
        ("want_rng", C.c_int32),
        ("row_interleave", C.c_int32),
        ("rank", C.c_int32),
        ("nranks", C.c_int32),
        ("no_cull", C.c_int32),
        ("sample_block", C.c_int32),
        ("sample_blocks", C.c_int32),
        ("n_vlp", C.c_int32),
        ("cluster_cull", C.c_int32),
        ("dead_rays", C.c_int32),
    ]


class pt_counters(C.Structure):
    _fields_ = [
        ("samples", C.c_uint64),
        ("rays", C.c_uint64),
        ("shadow_rays", C.c_uint64),
        ("tri_tests", C.c_uint64),
        ("cells_visited", C.c_uint64),
        ("prim_tests", C.c_uint64),
        ("tri_tests_executed", C.c_uint64),
        ("vpl_evals", C.c_uint64),
    ]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class pth_image(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("channels", C.c_uint32), ("maxval", C.c_uint32),
        ("depth", C.c_uint32), ("data_size", C.c_size_t), ("data", C.c_void_p),
    ]


_VP, _I, _D = C.c_void_p, C.c_int, C.c_double
_FP, _U32P, _I32P = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_int32)

# name -> (restype, argtypes): every symbol include/ptcuda.h declares
PTCUDA_SYMBOLS = {
    "pt_set_error_mode": (None, [_I]),
    "pt_last_error": (C.c_char_p, []),
    "pt_check": (None, None),  # variadic
    "pt_abi_version": (_I, []),
    "pt_device_count": (_I, []),
    "pt_select_device": (_I, []),
    "pt_create": (_VP, [_I]),
    "pt_create_on_stream": (_VP, [_I, _VP]),
    "pt_destroy": (None, [_VP]),
    "pt_device_name": (_I, [_VP, C.c_char_p, C.c_size_t]),
    "pt_device_props": (_I, [_VP, C.POINTER(_I), C.POINTER(_I)]),
    "pt_set_scene": (_I, [_VP, C.POINTER(pt_scene)]),
    "pt_build_grid": (_VP, [_VP, C.POINTER(pt_grid)]),
    "pt_read_grid_cells": (_I, [_VP, _VP, C.c_size_t]),
    "pt_read_grid_csr": (_I, [_VP, _U32P, _U32P, C.POINTER(C.c_uint64)]),
    "pt_launch_pathtracer": (_VP, [_VP, C.POINTER(pt_camera), C.POINTER(pt_render_params)]),
    "pt_launch_pathtracer_range": (_VP, [_VP, C.POINTER(pt_camera), C.POINTER(pt_render_params), _I, _I]),
    "pt_set_render_state": (_I, [_VP, C.POINTER(pt_camera), C.POINTER(pt_render_params), _I, _FP, _U32P]),
    "pt_map_render": (_VP, [_VP, C.POINTER(_VP)]),
    "pt_read_accum": (_I, [_VP, _FP, C.c_size_t]),
    "pt_read_rng_state": (_I, [_VP, _U32P, C.c_size_t]),
    "pt_get_counters": (_I, [_VP, C.POINTER(pt_counters)]),
    "pt_launch_lighttracer": (_VP, [_VP, _I, _U32P, _I]),
    "pt_launch_metropolis_lighttracer": (_VP, [_VP, _I, _U32P, _I, _I]),
    "pt_read_metropolis_paths": (_I, [_VP, _U32P, _I, _I]),
    "pt_set_vpls": (_I, [_VP, _FP, _I]),
    "pt_read_vpls": (_I, [_VP, _FP, _I]),
    "pt_render_device": (_I, [_VP, C.POINTER(pt_camera), C.POINTER(pt_render_params), _VP, _VP]),
    "pt_tonemap_device": (_I, [_VP, _VP, _VP, _I, _I]),
    "pt_render_host": (_I, [_VP, C.POINTER(pt_scene), C.POINTER(pt_grid), C.POINTER(pt_camera),
                            C.POINTER(pt_render_params), C.POINTER(C.c_uint8)]),
    "pt_multi_create": (_VP, [_I]),
    "pt_multi_destroy": (None, [_VP]),
    "pt_multi_set_scene": (_I, [_VP, C.POINTER(pt_scene)]),
    "pt_multi_build_grid": (_VP, [_VP, C.POINTER(pt_grid)]),
    "pt_multi_launch_lighttracer": (_VP, [_VP, _I, _U32P, _I]),
    "pt_multi_launch_pathtracer": (_VP, [_VP, C.POINTER(pt_camera), C.POINTER(pt_render_params)]),
    "pt_multi_map_render": (_VP, [_VP, C.POINTER(_VP)]),
    "pt_multi_get_counters": (_I, [_VP, C.POINTER(pt_counters)]),
    "pt_multi_set_bounces": (_I, [_VP, _I]),
    "pt_set_bounces": (_I, [_VP, _I]),
    "pt_wait": (_I, [_VP]),
    "pt_runtime_ms": (_D, [_VP]),
    "pt_release_event": (None, [_VP]),
    "pt_synchronize": (_I, [_VP]),
    "pt_probe_trace": (_I, [_VP, _I, _I, _I, _FP, _FP, _FP, _I32P, _FP]),
    "pt_probe_trace_counts": (_I, [_VP, _I, _I, _I, _FP, _FP, _FP, _I32P, _FP, _U32P, _U32P]),
    "pt_selftest_fastmath": (_I, [_VP, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64)]),
    "pt_probe_rng": (_I, [_VP, _U32P, C.c_uint32, _I, _FP, _U32P]),
    "pt_measure_peaks": (_I, [_VP, C.POINTER(C.c_double)]),
    "pt_last_kernel": (_I, [_VP]),
    "pt_vlp_bounds": (_I, [_VP, _FP, _FP]),
    "pt_build_vlp_grid": (_VP, [_VP, C.POINTER(pt_grid)]),
    "pt_read_vlp_grid_csr": (_I, [_VP, _U32P, _U32P, C.POINTER(C.c_uint64)]),
    "pt_read_vlp_grid_cells": (_I, [_VP, C.c_void_p, C.c_size_t]),
    "pt_query_device": (_I, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_size_t]),
    "pt_debug_read_scratch": (_I, [_VP, C.c_void_p, C.c_size_t, C.c_size_t]),
}

PTHOST_SYMBOLS = {
    "pth_parse_bitmap": (_I, [C.c_char_p, _I32P]),
    "pth_parse_triangles": (_I, [C.c_char_p, _I, C.POINTER(_FP), _FP, _FP]),
    "pth_parse_lights": (_I, [C.c_char_p, C.POINTER((C.c_float * 4) * 5), _I]),
    "pth_camera": (None, [C.POINTER(pt_camera)]),
    "pth_grid_dims": (None, [_FP, _FP, _I, C.c_float, C.POINTER(pt_grid)]),
    "pth_save_pam": (_I, [C.c_char_p, _I, _I, _VP]),
    "pth_seeds": (None, [_U32P]),
    "pth_load_pam": (_I, [C.c_char_p, C.POINTER(pth_image)]),
    "pth_free_image": (None, [C.POINTER(pth_image)]),
    "pth_save_ppm": (_I, [C.c_char_p, _I, _I, _VP]),
    "pth_save_png": (_I, [C.c_char_p, _I, _I, _VP]),
    "pth_import_obj": (C.c_long, [C.c_char_p, C.c_char_p, C.c_float, _FP]),
    "pth_cli_main": (_I, [_I, _I, C.POINTER(C.c_char_p)]),
    "pth_cli_metropolis_main": (_I, [_I, C.POINTER(C.c_char_p)]),
}

_cuda = None
_host = None


def _load(name, symbols):
    path = os.path.join(LIB_DIR, name)
    if not os.path.exists(path):
        raise RuntimeError(
            "%s not found: build it with `make -C %s` (or __graft_entry__.build()). "
            "There is no CPU fallback." % (path, os.path.join(_HERE, "csrc")))
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for sym, (res, args) in symbols.items():
        fn = getattr(lib, sym)  # AttributeError if the symbol is not exported
        fn.restype = res
        if args is not None:
            fn.argtypes = args
    return lib


def cuda_lib():
    """libptcuda.so (CUDA kernels + C ABI)."""
    global _cuda
    if _cuda is None:
        _cuda = _load("libptcuda.so", PTCUDA_SYMBOLS)
        _cuda.pt_set_error_mode(1)  # Python wants status codes, not exit(1)
    return _cuda


def host_lib():
    """libpthost.so (scene parsers, camera, grid sizing, PAM writer; plain C)."""
    global _host
    if _host is None:
        cuda_lib()
        _host = _load("libpthost.so", PTHOST_SYMBOLS)
    return _host
