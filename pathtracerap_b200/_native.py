"""ctypes binding of libptap.so (C ABI in include/ptap.h).

The library is the product: there is no Python or CPU fallback.  Importing this module fails
loudly when the shared library has not been built (`python -c "import __graft_entry__ as g; g.build()"`
or `make -C pathtracerap_b200/csrc`), and every compute entry point raises when no B200 is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PTAP_LIB") or os.path.join(HERE, "libptap.so")      # PTAP_LIB: a variant build (tools/build_variants.sh), for A/B measurements

# PODs with the reference's layouts (Primitive.h:23-178), see include/ptap.h
MATERIAL = np.dtype([("type", "<i4"), ("refractive_index", "<f4"), ("reflectivity", "<f4"), ("color", "<f4", 3)])
MODEL = np.dtype([("grid_index", "<i4"), ("mesh_index", "<i4"), ("model_to_world", "<f4", 16),
                  ("world_to_model", "<f4", 16), ("mat", MATERIAL)])
MESH = np.dtype([("v_start", "<i4"), ("v_end", "<i4"), ("t_start", "<i4"), ("t_end", "<i4"),
                 ("bb_min", "<f4", 3), ("bb_max", "<f4", 3)])
VERTEX = np.dtype([("position", "<f4", 3), ("normal", "<f4", 3), ("uv", "<f4", 2)])
TRIANGLE = np.dtype([("v", "<i4", 3)])
GRID = np.dtype([("v_start", "<i4"), ("v_end", "<i4"), ("width", "<f4", 3), ("entity_type", "<i4"), ("entity_index", "<i4")])
VOXEL = np.dtype([("start", "<i4"), ("end", "<i4"), ("entity_type", "<i4")])
HIT = np.dtype([("model", "<i4"), ("tri", "<i4"), ("t_model", "<f4"), ("dist", "<f4"), ("u", "<f4"), ("v", "<f4"),
                ("normal", "<f4", 3), ("mat_type", "<i4")])
PATH_IN = np.dtype([("orig", "<f4", 3), ("dir", "<f4", 3), ("color", "<f4", 3), ("ipixel", "<i4"),
                    ("model", "<i4"), ("tri", "<i4"), ("dist", "<f4")])
PATH_OUT = np.dtype([("orig", "<f4", 3), ("dir", "<f4", 3), ("color", "<f4", 3), ("ipixel", "<i4"), ("alive", "<i4")])
assert MODEL.itemsize == 160 and MESH.itemsize == 40 and VERTEX.itemsize == 32 and TRIANGLE.itemsize == 12
assert GRID.itemsize == 28 and VOXEL.itemsize == 12 and HIT.itemsize == 40 and PATH_IN.itemsize == 52 and PATH_OUT.itemsize == 44

FLOAT_MAX = np.float32(9999999.0)
DIFFUSE, SPECULAR, REFLECTIVE, REFRACTIVE, EMISSIVE, COAT, METAL = range(7)
ACCEL_GRID_COMPAT, ACCEL_BVH, ACCEL_BVH_DEVICE, ACCEL_GRID_EMULATED = 0, 1, 2, 3
E_UNSUPPORTED = -7
FLAG_FIRST_HIT_CACHE, FLAG_PROFILE, FLAG_COUNT, FLAG_STAMP, FLAG_ITER_TIMES = 1, 2, 4, 8, 16


class SceneView(C.Structure):
    _fields_ = [("models", C.c_void_p), ("nmodels", C.c_int32), ("meshes", C.c_void_p), ("nmeshes", C.c_int32),
                ("vertices", C.c_void_p), ("nvertices", C.c_int32), ("triangles", C.c_void_p), ("ntriangles", C.c_int32),
                ("grids", C.c_void_p), ("ngrids", C.c_int32), ("voxels", C.c_void_p), ("nvoxels", C.c_int32),
                ("refs", C.c_void_p), ("nrefs", C.c_int32), ("grid_dim", C.c_int32 * 3),
                ("bvh_nodes", C.c_void_p), ("n_bvh_nodes", C.c_int32), ("bvh_tri_id", C.c_void_p), ("n_bvh_tris", C.c_int32),
                ("bvh_mesh_root", C.c_void_p), ("n_bvh_roots", C.c_int32), ("bvh_depth", C.c_int32),
                ("tri_recs", C.c_void_p), ("n_tri_recs", C.c_int32)]


class Camera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("plane_min", C.c_float * 3), ("span", C.c_float * 2), ("jitter", C.c_int32), ("jitter_seed", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("rays_traced", C.c_int64), ("paths", C.c_int64), ("kernel_launches", C.c_int64),
                ("active_per_round", C.c_int64 * 16), ("ms_render", C.c_float), ("ms_trace", C.c_float),
                ("ms_shade", C.c_float), ("ms_generate", C.c_float), ("avg_nodes", C.c_float), ("avg_tris", C.c_float),
                ("avg_cells", C.c_float), ("avg_refs", C.c_float), ("trace_launches", C.c_int64), ("scene_bytes", C.c_int64),
                ("ms_build", C.c_float), ("bvh_nodes", C.c_int32), ("bvh_depth", C.c_int32), ("lanes", C.c_int32),
                ("ms_trace_inflight", C.c_float), ("ms_trace_sum", C.c_float), ("rays_walked", C.c_int64), ("rays_reemulated", C.c_int64)]


EXPORTS = [
    "ptap_scene_create_builtin", "ptap_scene_create_from_config", "ptap_scene_create_empty", "ptap_scene_create_from_view",
    "ptap_scene_add_obj", "ptap_scene_add_mesh", "ptap_scene_add_icosphere", "ptap_scene_add_model", "ptap_compose_trs",
    "ptap_scene_build_grids", "ptap_scene_build_bvh", "ptap_scene_pack_triangles", "ptap_scene_validate_bvh", "ptap_scene_view", "ptap_scene_models", "ptap_scene_destroy", "ptap_scene_last_error",
    "ptap_scene_config_params", "ptap_scene_config_camera", "ptap_set_camera",
    "ptap_create", "ptap_destroy", "ptap_last_error", "ptap_upload_scene", "ptap_build_accel", "ptap_build_grids_device", "ptap_read_grids", "ptap_set_render_params",
    "ptap_render", "ptap_timer_start", "ptap_timer_stop", "ptap_frame_begin", "ptap_film_reset", "ptap_sync", "ptap_read_film", "ptap_film_device_ptr", "ptap_film_add",
    "ptap_write_bmp", "ptap_read_film_resolved", "ptap_write_bmp_resolved", "ptap_get_stats", "ptap_stream", "ptap_trace", "ptap_trace_count", "ptap_shade", "ptap_bench_trace", "ptap_render_probe", "ptap_get_iteration_times",
    "ptap_query_closest", "ptap_query_occluded", "ptap_update_models",
    "ptap_reduce_peer", "ptap_nccl_unique_id", "ptap_nccl_init", "ptap_reduce", "ptap_nccl_finalize",
]

_lib = None


class PtapError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PtapError(f"{LIB_PATH} is missing: build it with `make -C pathtracerap_b200/csrc` "
                            "(there is no Python/CPU fallback for the render path)")
        L = C.CDLL(LIB_PATH)
        vp, ci, cu = C.c_void_p, C.c_int32, C.c_uint32
        pp = C.POINTER(C.c_void_p)
        L.ptap_scene_create_builtin.argtypes = [C.c_char_p, pp]
        L.ptap_scene_create_from_config.argtypes = [C.c_char_p, pp]
        L.ptap_scene_create_empty.argtypes = [pp]
        L.ptap_scene_create_from_view.argtypes = [C.POINTER(SceneView), pp]
        L.ptap_scene_add_obj.argtypes = [vp, C.c_char_p, C.POINTER(ci)]
        L.ptap_scene_add_mesh.argtypes = [vp, vp, ci, vp, ci, C.POINTER(ci)]
        L.ptap_scene_add_icosphere.argtypes = [vp, ci, C.c_float, C.c_float, cu, C.POINTER(ci)]
        L.ptap_scene_add_model.argtypes = [vp, ci, vp, vp, vp, C.POINTER(ci)]
        L.ptap_compose_trs.argtypes = [vp, C.c_float, vp, vp, vp]; L.ptap_compose_trs.restype = None
        L.ptap_scene_build_grids.argtypes = [vp, ci, ci, ci]
        L.ptap_scene_view.argtypes = [vp, C.POINTER(SceneView)]
        L.ptap_scene_build_bvh.argtypes = [vp]
        L.ptap_scene_pack_triangles.argtypes = [vp]
        L.ptap_scene_validate_bvh.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(ci)]
        L.ptap_scene_models.argtypes = [vp]; L.ptap_scene_models.restype = vp
        L.ptap_scene_destroy.argtypes = [vp]; L.ptap_scene_destroy.restype = None
        L.ptap_scene_last_error.argtypes = [vp]; L.ptap_scene_last_error.restype = C.c_char_p
        L.ptap_scene_config_params.argtypes = [vp, vp]
        L.ptap_scene_config_camera.argtypes = [vp, C.POINTER(Camera)]
        L.ptap_set_camera.argtypes = [vp, C.POINTER(Camera)]
        L.ptap_create.argtypes = [C.c_int, C.c_size_t, pp]
        L.ptap_destroy.argtypes = [vp]; L.ptap_destroy.restype = None
        L.ptap_last_error.argtypes = [vp]; L.ptap_last_error.restype = C.c_char_p
        L.ptap_upload_scene.argtypes = [vp, C.POINTER(SceneView)]
        L.ptap_build_accel.argtypes = [vp, C.c_int]
        L.ptap_build_grids_device.argtypes = [vp, C.POINTER(SceneView), ci, ci, ci]
        L.ptap_read_grids.argtypes = [vp, vp, vp, vp]
        L.ptap_set_render_params.argtypes = [vp, ci, ci, ci, cu]
        L.ptap_render.argtypes = [vp, ci, ci]
        L.ptap_film_reset.argtypes = [vp]
        L.ptap_frame_begin.argtypes = [vp]
        L.ptap_timer_start.argtypes = [vp]
        L.ptap_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
        L.ptap_sync.argtypes = [vp]
        L.ptap_read_film.argtypes = [vp, vp]
        L.ptap_film_device_ptr.argtypes = [vp, pp, C.POINTER(C.c_size_t)]
        L.ptap_film_add.argtypes = [vp, vp]
        L.ptap_write_bmp.argtypes = [vp, C.c_char_p, ci]
        L.ptap_read_film_resolved.argtypes = [vp, ci, ci, vp]
        L.ptap_write_bmp_resolved.argtypes = [vp, C.c_char_p, ci, ci, ci]
        L.ptap_get_stats.argtypes = [vp, C.POINTER(Stats)]
        L.ptap_stream.argtypes = [vp]; L.ptap_stream.restype = vp
        L.ptap_trace.argtypes = [vp, vp, ci, vp]
        L.ptap_trace_count.argtypes = [vp, vp, ci, vp, vp]
        L.ptap_shade.argtypes = [vp, vp, ci, ci, ci, vp, vp, C.POINTER(ci)]
        L.ptap_bench_trace.argtypes = [vp, vp, ci, ci, C.POINTER(C.c_float)]
        L.ptap_render_probe.argtypes = [vp, ci, ci, vp, vp, vp, ci, C.POINTER(ci)]
        L.ptap_get_iteration_times.argtypes = [vp, vp, ci, C.POINTER(ci)]
        L.ptap_query_closest.argtypes = [vp, vp, vp, ci, vp, vp]
        L.ptap_query_occluded.argtypes = [vp, vp, vp, ci, vp, vp]
        L.ptap_update_models.argtypes = [vp, vp, ci, ci]
        L.ptap_reduce_peer.argtypes = [vp, vp]
        L.ptap_nccl_unique_id.argtypes = [vp]
        L.ptap_nccl_init.argtypes = [vp, vp, ci, ci]
        L.ptap_reduce.argtypes = [vp, ci]
        L.ptap_nccl_finalize.argtypes = [vp]
        _lib = L
    return _lib


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
