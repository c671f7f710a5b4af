"""ctypes binding of libgsplat_b200.so (include/gsplat_b200.h).

This is the only door to the compute path.  There is no Python/NumPy implementation of any stage here:
if the CUDA library is missing or no GPU is visible, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

GS_MAX_SCENES = 32

_LIB_PATH = Path(__file__).resolve().parent / "csrc" / "libgsplat_b200.so"


class GsError(RuntimeError):
    def __init__(self, code: int, where: str, msg: str):
        super().__init__(f"{where}: [{code}] {msg}")
        self.code = code


# ---- status codes -------------------------------------------------------------------------------------------
GS_OK, GS_ERR_BAD_ARG, GS_ERR_NO_DEVICE, GS_ERR_CUDA, GS_ERR_DEGENERATE, GS_ERR_BUCKET_RANGE, GS_ERR_NOT_READY, GS_ERR_CAPACITY = range(8)
GS_COV_F32, GS_COV_F16 = 0, 1
GS_SH_NONE, GS_SH_F16, GS_SH_U8, GS_SH_F32 = 0, 1, 2, 3
GS_FRAME_RGBA32F, GS_FRAME_RGBA8 = 0, 1
GS_BUF_SORTED_INDEXES, GS_BUF_FRAME, GS_BUF_CENTERS, GS_BUF_DISTANCES, GS_BUF_SPLAT_RECORDS, GS_BUF_INDEXES_TO_SORT, GS_BUF_CENTERS_COLORS, GS_BUF_COVARIANCES, GS_BUF_SH, GS_BUF_SCALE_ROTATIONS, \
    GS_BUF_TILE_RECTS, GS_BUF_TILE_RANGES, GS_BUF_TILE_LIST, GS_BUF_TILE_ORDER, GS_BUF_TILE_INFO = range(15)
GS_RENDER_MODE_3D, GS_RENDER_MODE_2D = 0, 1


class gs_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("max_splat_count", C.c_uint32),
        ("distance_map_range", C.c_uint32), ("integer_based_sort", C.c_uint8), ("dynamic_mode", C.c_uint8),
        ("splat_render_mode", C.c_uint8), ("reserved0", C.c_uint8), ("max_width", C.c_uint32), ("max_height", C.c_uint32),
        ("rank", C.c_uint32), ("world_size", C.c_uint32),
    ]


class gs_sort_params(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("model_view_proj", C.c_float * 16), ("sort_count", C.c_uint32),
        ("render_count", C.c_uint32), ("indexes_to_sort", C.c_void_p), ("indexes_to_sort_dev", C.c_void_p),
        ("transforms", C.c_void_p), ("precomputed_distances", C.c_void_p), ("use_precomputed_distances", C.c_uint8),
        ("reserved", C.c_uint8 * 3),
    ]


class gs_splat_data(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("from_", C.c_uint32), ("count", C.c_uint32), ("centers_colors", C.c_void_p),
        ("covariances", C.c_void_p), ("cov_format", C.c_int32), ("spherical_harmonics", C.c_void_p),
        ("sh_format", C.c_int32), ("sh_degree", C.c_uint32), ("scene_indexes", C.c_void_p), ("scale_rotations", C.c_void_p),
    ]


class gs_uniforms(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("model_view", C.c_float * 16), ("projection", C.c_float * 16),
        ("camera_position", C.c_float * 3), ("focal", C.c_float * 2), ("viewport", C.c_float * 2),
        ("inverse_focal_adjustment", C.c_float), ("ortho_zoom", C.c_float), ("orthographic_mode", C.c_int32),
        ("splat_scale", C.c_float), ("point_cloud_mode", C.c_int32), ("sh_degree", C.c_int32),
        ("antialiased", C.c_int32), ("kernel_2d_size", C.c_float), ("max_screen_space_splat_size", C.c_float),
        ("sh8_min", C.c_float * GS_MAX_SCENES), ("sh8_max", C.c_float * GS_MAX_SCENES), ("scene_count", C.c_uint32),
        ("scene_transforms", C.c_float * (16 * GS_MAX_SCENES)), ("view_matrix", C.c_float * 16),
        ("scene_opacity", C.c_float * GS_MAX_SCENES), ("scene_visibility", C.c_int32 * GS_MAX_SCENES),
        ("enable_optional_effects", C.c_int32), ("dynamic_mode", C.c_int32), ("fade_in_complete", C.c_int32),
        ("scene_center", C.c_float * 3), ("visible_region_fade_start_radius", C.c_float),
    ]


class gs_render_params(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32), ("render_count", C.c_uint32),
        ("sorted_indexes", C.c_void_p), ("sorted_indexes_dev", C.c_void_p), ("frame_format", C.c_int32),
        ("flip_y", C.c_int32),
    ]


class gs_projected_splat(C.Structure):
    _fields_ = [
        ("cx", C.c_float), ("cy", C.c_float), ("b1x", C.c_float), ("b1y", C.c_float), ("b2x", C.c_float),
        ("b2y", C.c_float), ("r", C.c_float), ("g", C.c_float), ("b", C.c_float), ("a", C.c_float),
        ("ndc_z", C.c_float), ("valid", C.c_uint32),
    ]


PROJECTED_DTYPE = np.dtype([(n, np.float32) for n in ("cx", "cy", "b1x", "b1y", "b2x", "b2y", "r", "g", "b", "a", "ndc_z")] + [("valid", np.uint32)])


class gs_projected_surfel(C.Structure):
    _fields_ = [("T", C.c_float * 9)] + [(n, C.c_float) for n in ("qcx", "qcy", "cx", "cy", "h1x", "h1y", "h2x", "h2y", "r", "g", "b", "a", "ndc_z")] + \
        [("branch", C.c_uint32), ("valid", C.c_uint32)]


PROJECTED_SURFEL_DTYPE = np.dtype([("T", np.float32, (9,))] + [(n, np.float32) for n in ("qcx", "qcy", "cx", "cy", "h1x", "h1y", "h2x", "h2y", "r", "g", "b", "a", "ndc_z")]
                                  + [("branch", np.uint32), ("valid", np.uint32)])


class gs_timings(C.Structure):
    _fields_ = [
        ("depth_ms", C.c_float), ("bucket_ms", C.c_float), ("scatter_ms", C.c_float), ("sort_total_ms", C.c_float),
        ("project_ms", C.c_float), ("bin_ms", C.c_float), ("blend_ms", C.c_float), ("render_total_ms", C.c_float),
        ("h2d_ms", C.c_float), ("d2h_ms", C.c_float), ("tile_instances", C.c_uint64), ("kernel_launches", C.c_uint32),
        ("visible_splats", C.c_uint32),
    ]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class gs_ksplat_options(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("minimum_alpha", C.c_uint32), ("half_covariances", C.c_uint8), ("upload_sort_centers", C.c_uint8),
                ("has_transform", C.c_uint8), ("reserved", C.c_uint8 * 1), ("transform", C.c_double * 16)]


class gs_ksplat_info(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("splat_count", C.c_uint32), ("sh_degree", C.c_uint32), ("compression_level", C.c_uint32),
                ("section_count", C.c_uint32), ("scene_center", C.c_float * 3), ("min_sh_coeff", C.c_float), ("max_sh_coeff", C.c_float)]


class gs_kernel_time(C.Structure):
    _fields_ = [("name", C.c_char * 40), ("ms", C.c_float)]


EXPORTED_SYMBOLS = [
    "gs_abi_version", "gs_status_string", "gs_last_error_message", "gs_device_count", "gs_sort_indexes", "sortIndexes", "gs_dropin_release",
    "gs_create", "gs_destroy", "gs_upload_centers", "gs_sort", "gs_compute_distances", "gs_upload_splat_data",
    "gs_render", "gs_frame", "gs_buffer_dev", "gs_stream", "gs_synchronize", "gs_host_alloc", "gs_host_free",
    "gs_read_projected", "gs_read_projected_2d", "gs_last_timings", "gs_frame_async", "gs_frame_begin", "gs_frame_end", "gs_upload_splat_tree", "gs_gather_for_sort", "gs_flush_l2", "gs_event_create", "gs_event_record",
    "gs_event_elapsed_ms", "gs_event_destroy", "gs_set_profiling", "gs_kernel_timings", "gs_set_graph_enabled", "gs_upload_ksplat", "gs_read_buffer", "gs_peer_export", "gs_peer_attach",
    "gs_shard_export", "gs_shard_attach", "gs_shard_attach_local", "gs_sort_sharded", "gs_sort_sharded_async", "gs_sort_sharded_finish",
]

_lib = None


def lib_path() -> Path:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load the CUDA library.  Raises if it has not been built: the product has no other compute path."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise GsError(GS_ERR_NO_DEVICE, "load", f"{_LIB_PATH} is missing: run `python -m gaussiansplats3d_b200.build` "
                      "(nvcc, sm_100a). gaussiansplats3d_b200 has no CPU fallback.")
    lib = C.CDLL(str(_LIB_PATH))
    vp, u32, i32 = C.c_void_p, C.c_uint32, C.c_int32
    lib.gs_abi_version.restype = C.c_int
    lib.gs_status_string.restype = C.c_char_p
    lib.gs_status_string.argtypes = [C.c_int]
    lib.gs_last_error_message.restype = C.c_char_p
    lib.gs_device_count.restype = C.c_int
    lib.gs_sort_indexes.restype = C.c_int
    lib.gs_sort_indexes.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, u32, u32, u32, u32, C.c_bool, C.c_bool, C.c_bool]
    lib.sortIndexes.restype = None
    lib.sortIndexes.argtypes = lib.gs_sort_indexes.argtypes
    lib.gs_create.restype = C.c_int
    lib.gs_create.argtypes = [C.POINTER(gs_config), C.POINTER(vp)]
    lib.gs_destroy.restype = None
    lib.gs_destroy.argtypes = [vp]
    lib.gs_upload_centers.restype = C.c_int
    lib.gs_upload_centers.argtypes = [vp, vp, vp, u32, u32]
    lib.gs_sort.restype = C.c_int
    lib.gs_sort.argtypes = [vp, C.POINTER(gs_sort_params), vp, C.POINTER(C.c_float)]
    lib.gs_compute_distances.restype = C.c_int
    lib.gs_compute_distances.argtypes = [vp, vp, vp, u32, vp]
    lib.gs_upload_splat_data.restype = C.c_int
    lib.gs_upload_splat_data.argtypes = [vp, C.POINTER(gs_splat_data)]
    lib.gs_render.restype = C.c_int
    lib.gs_render.argtypes = [vp, C.POINTER(gs_uniforms), C.POINTER(gs_render_params), vp]
    lib.gs_frame.restype = C.c_int
    lib.gs_frame.argtypes = [vp, C.POINTER(gs_sort_params), C.POINTER(gs_uniforms), C.POINTER(gs_render_params), vp, vp]
    lib.gs_buffer_dev.restype = C.c_int
    lib.gs_buffer_dev.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.gs_stream.restype = C.c_int
    lib.gs_stream.argtypes = [vp, C.POINTER(vp)]
    lib.gs_synchronize.restype = C.c_int
    lib.gs_synchronize.argtypes = [vp]
    lib.gs_host_alloc.restype = C.c_int
    lib.gs_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    lib.gs_host_free.restype = C.c_int
    lib.gs_host_free.argtypes = [vp]
    lib.gs_read_projected.restype = C.c_int
    lib.gs_read_projected.argtypes = [vp, vp, u32]
    lib.gs_read_projected_2d.restype = C.c_int
    lib.gs_read_projected_2d.argtypes = [vp, vp, u32]
    lib.gs_last_timings.restype = C.c_int
    lib.gs_last_timings.argtypes = [vp, C.POINTER(gs_timings)]
    lib.gs_upload_splat_tree.restype = C.c_int
    lib.gs_upload_splat_tree.argtypes = [vp, vp, vp, vp, vp, vp, C.c_uint32]
    lib.gs_gather_for_sort.restype = C.c_int
    lib.gs_gather_for_sort.argtypes = [vp, vp, C.c_double, C.c_double, C.c_int, C.POINTER(C.c_uint32)]
    lib.gs_dropin_release.restype = None
    lib.gs_dropin_release.argtypes = []
    lib.gs_frame_begin.restype = C.c_int
    lib.gs_frame_begin.argtypes = [vp, C.POINTER(gs_sort_params), C.POINTER(gs_uniforms), C.POINTER(gs_render_params), vp]
    lib.gs_frame_end.restype = C.c_int
    lib.gs_frame_end.argtypes = [vp]
    lib.gs_frame_async.restype = C.c_int
    lib.gs_frame_async.argtypes = [vp, C.POINTER(gs_sort_params), C.POINTER(gs_uniforms), C.POINTER(gs_render_params)]
    lib.gs_flush_l2.restype = C.c_int
    lib.gs_flush_l2.argtypes = [vp]
    lib.gs_event_create.restype = C.c_int
    lib.gs_event_create.argtypes = [C.POINTER(vp)]
    lib.gs_event_record.restype = C.c_int
    lib.gs_event_record.argtypes = [vp, vp]
    lib.gs_event_elapsed_ms.restype = C.c_int
    lib.gs_event_elapsed_ms.argtypes = [vp, vp, C.POINTER(C.c_float)]
    lib.gs_event_destroy.restype = C.c_int
    lib.gs_event_destroy.argtypes = [vp]
    lib.gs_set_profiling.restype = C.c_int
    lib.gs_set_profiling.argtypes = [vp, C.c_int]
    lib.gs_upload_ksplat.restype = C.c_int
    lib.gs_upload_ksplat.argtypes = [vp, vp, C.c_size_t, C.POINTER(gs_ksplat_options), C.POINTER(gs_ksplat_info)]
    lib.gs_read_buffer.restype = C.c_int
    lib.gs_read_buffer.argtypes = [vp, C.c_int, vp, C.c_size_t, C.c_size_t]
    lib.gs_peer_export.restype = C.c_int
    lib.gs_peer_export.argtypes = [vp, vp, vp]
    lib.gs_peer_attach.restype = C.c_int
    lib.gs_peer_attach.argtypes = [vp, vp, vp]
    lib.gs_shard_export.restype = C.c_int
    lib.gs_shard_export.argtypes = [vp, vp, vp]
    lib.gs_shard_attach.restype = C.c_int
    lib.gs_shard_attach.argtypes = [vp, u32, vp, vp]
    lib.gs_shard_attach_local.restype = C.c_int
    lib.gs_shard_attach_local.argtypes = [vp, u32, C.POINTER(vp)]
    lib.gs_sort_sharded.restype = C.c_int
    lib.gs_sort_sharded.argtypes = [vp, C.POINTER(gs_sort_params), vp, C.POINTER(C.c_float)]
    lib.gs_sort_sharded_async.restype = C.c_int
    lib.gs_sort_sharded_async.argtypes = [vp, C.POINTER(gs_sort_params)]
    lib.gs_sort_sharded_finish.restype = C.c_int
    lib.gs_sort_sharded_finish.argtypes = [vp, vp, C.POINTER(C.c_float)]
    lib.gs_set_graph_enabled.restype = C.c_int
    lib.gs_set_graph_enabled.argtypes = [vp, C.c_int]
    lib.gs_kernel_timings.restype = C.c_int
    lib.gs_kernel_timings.argtypes = [vp, C.POINTER(gs_kernel_time), u32, C.POINTER(u32)]
    _ = i32
    _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code != GS_OK:
        lib = load()
        msg = lib.gs_last_error_message().decode("utf-8", "replace")
        raise GsError(code, where, msg or lib.gs_status_string(code).decode())


def ptr(a) -> int | None:
    """Host pointer of a C-contiguous numpy array (None stays NULL)."""
    if a is None:
        return None
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("array must be C-contiguous")
    return a.ctypes.data


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array backed by page-locked memory from gs_host_alloc (freed when the array is collected)."""
    lib = load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    check(lib.gs_host_alloc(C.byref(p), max(n, 1)), "gs_host_alloc")
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    class _Owner:
        def __init__(self, addr):
            self.addr = addr

        def __del__(self):
            try:
                lib.gs_host_free(C.c_void_p(self.addr))
            except Exception:
                pass

    _PINNED_OWNERS[arr.__array_interface__["data"][0]] = _Owner(p.value)
    return arr


_PINNED_OWNERS: dict[int, object] = {}
_ = os
