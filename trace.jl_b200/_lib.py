"""ctypes binding of libtrace_cuda.so (include/trace_cuda.h).  There is no CPU fallback: if the shared library is
missing the import of any compute entry point raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libtrace_cuda.so")

ABI_VERSION = 3
COMM_ID_BYTES = 128
NODE_LEAF = 0xC0000000
PRIM_TRIANGLE, PRIM_SPHERE = 0, 1
TRI_FLIP, TRI_HAS_NORMALS = 1, 2
MAT_MATTE, MAT_MIRROR, MAT_GLASS, MAT_PLASTIC = 0, 1, 2, 3
LIGHT_POINT, LIGHT_SPOT, LIGHT_DIRECTIONAL = 0, 1, 2

node_dtype = np.dtype([("bmin", "<f4", 3), ("bmax", "<f4", 3), ("offset", "<u4"), ("meta", "<u4")])
prim_dtype = np.dtype([("kind", "<u4"), ("index", "<u4"), ("material", "<u4"), ("original", "<u4")])
sphere_dtype = np.dtype([("m", "<f4", 16), ("inv_m", "<f4", 16), ("radius", "<f4"), ("z_min", "<f4"), ("z_max", "<f4"),
                         ("theta_min", "<f4"), ("theta_max", "<f4"), ("phi_max", "<f4"), ("flip", "<u4"), ("pad", "<u4")])
material_dtype = np.dtype([("kind", "<u4"), ("a", "<f4", 3), ("b", "<f4", 3), ("eta", "<f4"), ("rough_u", "<f4"),
                           ("rough_v", "<f4"), ("remap", "<u4")])
light_dtype = np.dtype([("kind", "<u4"), ("m", "<f4", 16), ("inv_m", "<f4", 16), ("I", "<f4", 3), ("position", "<f4", 3),
                        ("cos_total_width", "<f4"), ("cos_falloff_start", "<f4")])
assert node_dtype.itemsize == 32 and prim_dtype.itemsize == 16 and sphere_dtype.itemsize == 160
assert material_dtype.itemsize == 44 and light_dtype.itemsize == 164


class SceneDesc(C.Structure):
    _fields_ = [("n_nodes", C.c_int64), ("nodes", C.c_void_p),
                ("n_prims", C.c_int64), ("prims", C.c_void_p),
                ("n_tris", C.c_int64), ("tri_vertices", C.c_void_p), ("tri_normals", C.c_void_p), ("tri_flags", C.c_void_p),
                ("n_spheres", C.c_int64), ("spheres", C.c_void_p),
                ("n_materials", C.c_int64), ("materials", C.c_void_p),
                ("n_lights", C.c_int64), ("lights", C.c_void_p)]


class MeshDeviceDesc(C.Structure):
    """trace_mesh_device_desc: per-triangle arrays in device memory (raw pointers), materials and lights in host memory"""
    _fields_ = [("n_tris", C.c_int64), ("tri_vertices", C.c_void_p), ("tri_normals", C.c_void_p),
                ("tri_flags", C.c_void_p), ("tri_materials", C.c_void_p),
                ("max_node_primitives", C.c_int32), ("pad", C.c_int32),
                ("n_materials", C.c_int64), ("materials", C.c_void_p),
                ("n_lights", C.c_int64), ("lights", C.c_void_p)]


class Camera(C.Structure):
    _fields_ = [("raster_to_camera", C.c_float * 16), ("camera_to_world", C.c_float * 16),
                ("lens_radius", C.c_float), ("focal_distance", C.c_float),
                ("shutter_open", C.c_float), ("shutter_close", C.c_float)]


class FilmDesc(C.Structure):
    _fields_ = [("crop_x0", C.c_int32), ("crop_y0", C.c_int32), ("crop_x1", C.c_int32), ("crop_y1", C.c_int32),
                ("filter_radius", C.c_float * 2), ("filter_table", C.c_float * 256), ("scale", C.c_float)]


class Stats(C.Structure):
    _fields_ = [("rays_extend", C.c_uint64), ("rays_shadow", C.c_uint64), ("nodes_visited", C.c_uint64),
                ("prims_tested", C.c_uint64), ("kernel_launches", C.c_uint64), ("ms_extend", C.c_double),
                ("ms_shadow", C.c_double), ("ms_total", C.c_double), ("queue_overflows", C.c_uint64),
                ("sppm_deposits", C.c_uint64), ("extend_launches", C.c_uint64), ("shadow_launches", C.c_uint64),
                ("ms_kind", C.c_double * 9), ("launches_kind", C.c_uint64 * 9), ("sppm_candidates", C.c_uint64),
                ("sppm_requests", C.c_uint64), ("sppm_grid_items", C.c_uint64), ("primary_rays", C.c_uint64),
                ("primary_hits", C.c_uint64)]

    def as_dict(self):
        return {k: (list(getattr(self, k)) if k in ("ms_kind", "launches_kind") else getattr(self, k)) for k, _ in self._fields_}


K_EXTEND, K_SHADOW, K_GENERATE, K_SHADE, K_SPLAT, K_GRID, K_DEPOSIT, K_UPDATE = range(8)
KIND_NAMES = ["extend", "shadow", "generate", "shade", "splat", "grid", "deposit", "update", "comm"]


SPPM_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_float))

# every symbol include/trace_cuda.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "trace_bvh_build": (C.c_int, [_P, C.c_int64, C.c_int, C.POINTER(_P)]),
    "trace_bvh_build_sah": (C.c_int, [_P, C.c_int64, C.c_int, C.POINTER(_P)]),
    "trace_bvh_build_gpu": (C.c_int, [C.c_int, _P, C.c_int64, C.c_int, C.POINTER(_P)]),
    "trace_bvh_num_nodes": (C.c_int64, [_P]),
    "trace_bvh_num_prims": (C.c_int64, [_P]),
    "trace_bvh_copy": (C.c_int, [_P, _P, _P]),
    "trace_bvh_free": (None, [_P]),
    "trace_abi_version": (C.c_int, []),
    "trace_create": (C.c_int, [C.POINTER(_P), C.c_int, _P]),
    "trace_destroy": (None, [_P]),
    "trace_last_error": (C.c_char_p, [_P]),
    "trace_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "trace_get_stats": (C.c_int, [_P, C.POINTER(Stats)]),
    "trace_reset_stats": (C.c_int, [_P]),
    "trace_synchronize": (C.c_int, [_P]),
    "trace_comm_unique_id": (C.c_int, [_P]),
    "trace_comm_init": (C.c_int, [_P, _P, C.c_int, C.c_int]),
    "trace_comm_destroy": (C.c_int, [_P]),
    "trace_comm_info": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "trace_scene_upload": (C.c_int, [_P, C.POINTER(SceneDesc)]),
    "trace_scene_upload_mesh_device": (C.c_int, [_P, C.POINTER(MeshDeviceDesc), C.POINTER(C.c_int64)]),
    "trace_scene_attach_mesh_device": (C.c_int, [_P, C.POINTER(MeshDeviceDesc), C.POINTER(C.c_int64)]),
    "trace_scene_attach_meshes_device": (C.c_int, [_P, C.c_int64, C.POINTER(C.POINTER(MeshDeviceDesc)), C.POINTER(C.c_int64)]),
    "trace_scene_refit": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int64, _P]),
    "trace_scene_refit_device": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int64, _P]),
    "trace_scene_copy_nodes": (C.c_int, [_P, _P]),
    "trace_scene_shadow_tree": (C.c_int, [_P, C.POINTER(C.c_int64), _P]),
    "trace_get_shadow_fallbacks": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "trace_get_hit_fallbacks": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "trace_intersect": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P]),
    "trace_occluded": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P]),
    "trace_intersect_device": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "trace_occluded_device": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "trace_render_whitted": (C.c_int, [_P, C.POINTER(Camera), C.POINTER(FilmDesc), C.c_int, C.c_int, C.c_uint64, _P]),
    "trace_render_whitted_device": (C.c_int, [_P, C.POINTER(Camera), C.POINTER(FilmDesc), C.c_int, C.c_int, C.c_uint64, _P]),
    "trace_render_sppm": (C.c_int, [_P, C.POINTER(Camera), C.POINTER(FilmDesc), C.c_float, C.c_int, C.c_int, C.c_int64,
                                    C.c_int, C.c_uint64, SPPM_CB, _P, _P]),
    "trace_sppm_begin": (C.c_int, [_P, C.POINTER(Camera), C.POINTER(FilmDesc), C.c_float, C.c_int, C.c_int64, C.c_uint64]),
    "trace_sppm_camera_pass": (C.c_int, [_P, C.c_int]),
    "trace_sppm_trace_photons": (C.c_int, [_P, C.c_int, C.c_int64, C.c_int64]),
    "trace_sppm_photon_pass": (C.c_int, [_P, C.c_int, C.c_int64, C.c_int64]),
    "trace_sppm_build_grid": (C.c_int, [_P]),
    "trace_sppm_flux_device": (_P, [_P, C.POINTER(C.c_int64)]),
    "trace_sppm_buffer_device": (_P, [_P, C.c_int, C.POINTER(C.c_int64)]),
    "trace_sppm_update": (C.c_int, [_P]),
    "trace_sppm_image": (C.c_int, [_P, C.c_int, _P]),
    "trace_sppm_end": (C.c_int, [_P]),
    "trace_sppm_iterate": (C.c_int, [_P, C.c_int, C.c_int]),
}

_lib = None


def load():
    """Load libtrace_cuda.so; raises (loudly) when it has not been built."""
    global _lib
    if _lib is None:
        path = os.environ.get("TRACE_CUDA_LIB", LIB_PATH)      # (A/B experiments load an alternative build of the same ABI)
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.trace_abi_version() != ABI_VERSION:
            raise RuntimeError("libtrace_cuda.so ABI version mismatch")
        _lib = lib
    return _lib


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
