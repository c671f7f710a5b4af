"""Thin object wrapper over the C ABI (include/gsplat_b200.h): one Engine = one gs_engine on one GPU.

Host-side glue only (argument marshalling).  Every computation happens in libgsplat_b200.so's CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _native as N


@dataclass
class Uniforms:
    """Python view of gs_uniforms: what SplatMesh.updateUniforms (SplatMesh.js:1248-1280) + three.js hand the shaders."""
    model_view: np.ndarray
    projection: np.ndarray
    camera_position: np.ndarray
    focal: tuple[float, float]
    viewport: tuple[float, float]
    inverse_focal_adjustment: float = 1.0
    ortho_zoom: float = 1.0
    orthographic_mode: int = 0
    splat_scale: float = 1.0
    point_cloud_mode: int = 0
    sh_degree: int = 0
    antialiased: int = 0
    kernel_2d_size: float = 0.3
    max_screen_space_splat_size: float = 1024.0
    sh8_min: np.ndarray = field(default_factory=lambda: np.full(N.GS_MAX_SCENES, -1.5, np.float32))
    sh8_max: np.ndarray = field(default_factory=lambda: np.full(N.GS_MAX_SCENES, 1.5, np.float32))
    scene_count: int = 1
    scene_transforms: np.ndarray | None = None
    view_matrix: np.ndarray | None = None
    scene_opacity: np.ndarray | None = None
    scene_visibility: np.ndarray | None = None
    enable_optional_effects: int = 0
    dynamic_mode: int = 0
    fade_in_complete: int = 1
    scene_center: tuple[float, float, float] = (0.0, 0.0, 0.0)
    visible_region_fade_start_radius: float = 0.0

    def to_c(self) -> N.gs_uniforms:
        u = N.gs_uniforms()
        u.struct_size = C.sizeof(N.gs_uniforms)
        u.model_view[:] = np.asarray(self.model_view, np.float32).reshape(16).tolist()
        u.projection[:] = np.asarray(self.projection, np.float32).reshape(16).tolist()
        u.camera_position[:] = np.asarray(self.camera_position, np.float32).reshape(3).tolist()
        u.focal[:] = [float(np.float32(self.focal[0])), float(np.float32(self.focal[1]))]
        u.viewport[:] = [float(self.viewport[0]), float(self.viewport[1])]
        u.inverse_focal_adjustment = self.inverse_focal_adjustment
        u.ortho_zoom = self.ortho_zoom
        u.orthographic_mode = self.orthographic_mode
        u.splat_scale = self.splat_scale
        u.point_cloud_mode = self.point_cloud_mode
        u.sh_degree = self.sh_degree
        u.antialiased = self.antialiased
        u.kernel_2d_size = self.kernel_2d_size
        u.max_screen_space_splat_size = self.max_screen_space_splat_size
        u.sh8_min[:] = np.asarray(self.sh8_min, np.float32).tolist()
        u.sh8_max[:] = np.asarray(self.sh8_max, np.float32).tolist()
        u.scene_count = self.scene_count
        tr = self.scene_transforms
        if tr is None:
            tr = np.tile(np.eye(4, dtype=np.float32).reshape(16), N.GS_MAX_SCENES)
        u.scene_transforms[:] = np.asarray(tr, np.float32).reshape(-1).tolist()
        vm = self.view_matrix if self.view_matrix is not None else np.eye(4, dtype=np.float32)
        u.view_matrix[:] = np.asarray(vm, np.float32).reshape(16).tolist()
        op = self.scene_opacity if self.scene_opacity is not None else np.ones(N.GS_MAX_SCENES, np.float32)
        u.scene_opacity[:] = np.asarray(op, np.float32).tolist()
        vis = self.scene_visibility if self.scene_visibility is not None else np.ones(N.GS_MAX_SCENES, np.int32)
        u.scene_visibility[:] = np.asarray(vis, np.int32).tolist()
        u.enable_optional_effects = self.enable_optional_effects
        u.dynamic_mode = self.dynamic_mode
        u.fade_in_complete = self.fade_in_complete
        u.scene_center[:] = [float(v) for v in self.scene_center]
        u.visible_region_fade_start_radius = self.visible_region_fade_start_radius
        return u


class Engine:
    """Device-resident sorter + rasteriser for one GPU."""

    def __init__(self, max_splat_count: int, *, device: int = 0, distance_map_range: int = 1 << 16,
                 integer_based_sort: bool = True, dynamic_mode: bool = False, max_width: int = 0, max_height: int = 0,
                 rank: int = 0, world_size: int = 1, splat_render_mode: int = N.GS_RENDER_MODE_3D):
        """`splat_render_mode`: SplatRenderMode.ThreeD (0) or TwoD (1, 2D Gaussian surfels), fixed for the engine's lifetime."""
        self._lib = N.load()
        cfg = N.gs_config()
        cfg.struct_size = C.sizeof(N.gs_config)
        cfg.device = device
        cfg.max_splat_count = max_splat_count
        cfg.distance_map_range = distance_map_range
        cfg.integer_based_sort = 1 if integer_based_sort else 0
        cfg.dynamic_mode = 1 if dynamic_mode else 0
        cfg.max_width, cfg.max_height = max_width, max_height
        cfg.rank, cfg.world_size = rank, world_size
        cfg.splat_render_mode = int(splat_render_mode)
        self.cfg = cfg
        self._h = C.c_void_p()
        N.check(self._lib.gs_create(C.byref(cfg), C.byref(self._h)), "gs_create")
        self.max_splat_count = max_splat_count
        self.integer_based_sort = integer_based_sort
        self.dynamic_mode = dynamic_mode
        self.rank, self.world_size = rank, world_size
        self.splat_render_mode = int(splat_render_mode)
        self._keep: list = []

    # -- lifetime -------------------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.gs_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- sorter ------------------------------------------------------------------------------------------------
    def upload_centers(self, centers: np.ndarray, scene_indexes: np.ndarray | None = None, start: int = 0) -> None:
        want = np.int32 if self.integer_based_sort else np.float32
        c = np.ascontiguousarray(centers, dtype=want).reshape(-1, 4)
        si = None if scene_indexes is None else np.ascontiguousarray(scene_indexes, dtype=np.uint32)
        N.check(self._lib.gs_upload_centers(self._h, N.ptr(c), N.ptr(si), start, c.shape[0]), "gs_upload_centers")

    def _sort_params(self, mvp, sort_count, render_count, indexes, transforms, precomputed, indexes_dev=None) -> N.gs_sort_params:
        p = N.gs_sort_params()
        p.struct_size = C.sizeof(N.gs_sort_params)
        p.model_view_proj[:] = np.asarray(mvp, np.float32).reshape(16).tolist()
        p.sort_count, p.render_count = int(sort_count), int(render_count)
        keep = []
        if indexes is not None:
            idx = indexes if (isinstance(indexes, np.ndarray) and indexes.dtype == np.uint32 and indexes.flags["C_CONTIGUOUS"]) else np.ascontiguousarray(indexes, dtype=np.uint32)
            keep.append(idx)
            p.indexes_to_sort = N.ptr(idx)
        if indexes_dev is not None:
            p.indexes_to_sort_dev = int(indexes_dev)
        if transforms is not None:
            t = np.zeros(16 * N.GS_MAX_SCENES, np.float32)
            tt = np.asarray(transforms, np.float32).reshape(-1)
            t[: tt.size] = tt
            keep.append(t)
            p.transforms = N.ptr(t)
        if precomputed is not None:
            want = np.int32 if self.integer_based_sort else np.float32
            pd = np.ascontiguousarray(precomputed, dtype=want)
            keep.append(pd)
            p.precomputed_distances = N.ptr(pd)
            p.use_precomputed_distances = 1
        self._keep = keep
        return p

    def sort(self, mvp, sort_count: int, render_count: int, indexes: np.ndarray | None = None, *, transforms=None,
             precomputed=None, out: np.ndarray | None = None, download: bool = True):
        """'sort' message -> 'sortDone'.  Returns (sortedIndexes or None, sort_time_ms)."""
        p = self._sort_params(mvp, sort_count, render_count, indexes, transforms, precomputed)
        if download and out is None:
            out = np.empty(render_count, np.uint32)
        ms = C.c_float(0)
        N.check(self._lib.gs_sort(self._h, C.byref(p), N.ptr(out) if download else None, C.byref(ms)), "gs_sort")
        return (out if download else None), ms.value

    # -- sort-only on N GPUs (include/gsplat_b200.h "Sort-only on N GPUs") --------------------------------------------
    def shard_export(self) -> tuple[bytes, bytes]:
        """CUDA-IPC handles of this rank's exchange block and of its sortedIndexes buffer."""
        a, b = C.create_string_buffer(64), C.create_string_buffer(64)
        N.check(self._lib.gs_shard_export(self._h, a, b), "gs_shard_export")
        return a.raw, b.raw

    def shard_attach(self, block_handles: list[bytes], root_sorted_handle: bytes) -> None:
        """All ranks: map every rank's exchange block (list index = rank) and rank 0's sortedIndexes."""
        blob = C.create_string_buffer(b"".join(block_handles), 64 * len(block_handles))
        N.check(self._lib.gs_shard_attach(self._h, len(block_handles), blob, C.create_string_buffer(root_sorted_handle, 64)), "gs_shard_attach")

    def shard_attach_local(self, engines: list["Engine"]) -> None:
        """Engines of this process on one device (list index = rank): plain pointers instead of IPC mappings."""
        arr = (C.c_void_p * len(engines))(*[en._h for en in engines])
        N.check(self._lib.gs_shard_attach_local(self._h, len(engines), arr), "gs_shard_attach_local")

    def sort_sharded_async(self, mvp, sort_count: int, render_count: int, indexes: np.ndarray | None = None, *, transforms=None, precomputed=None) -> None:
        p = self._sort_params(mvp, sort_count, render_count, indexes, transforms, precomputed)
        self._shard_keep = p
        N.check(self._lib.gs_sort_sharded_async(self._h, C.byref(p)), "gs_sort_sharded_async")

    def sort_sharded_finish(self, out: np.ndarray | None = None):
        """Waits for this rank's part; on rank 0 `out` (render_count u32) receives the assembled order.  Returns (out, ms)."""
        ms = C.c_float(0)
        N.check(self._lib.gs_sort_sharded_finish(self._h, N.ptr(out), C.byref(ms)), "gs_sort_sharded_finish")
        return out, ms.value

    def sort_sharded(self, mvp, sort_count: int, render_count: int, indexes: np.ndarray | None = None, *, transforms=None, precomputed=None,
                     out: np.ndarray | None = None):
        """One sortIndexes call spread over the ranks of the group; every rank calls it with the same arguments."""
        self.sort_sharded_async(mvp, sort_count, render_count, indexes, transforms=transforms, precomputed=precomputed)
        return self.sort_sharded_finish(out)

    # -- SplatTree cull -> indexesToSort (gs_upload_splat_tree / gs_gather_for_sort) --------------------------------------------
    def upload_splat_tree(self, leaves) -> None:
        """`leaves`: splat_tree.SplatTreeLeaves (nodesWithIndexes of the tree)."""
        c = np.ascontiguousarray(leaves.node_center, dtype=np.float64)
        mn = np.ascontiguousarray(leaves.node_min, dtype=np.float64)
        mx = np.ascontiguousarray(leaves.node_max, dtype=np.float64)
        off = np.ascontiguousarray(leaves.offsets, dtype=np.uint32)
        idx = np.ascontiguousarray(leaves.indexes, dtype=np.uint32)
        N.check(self._lib.gs_upload_splat_tree(self._h, N.ptr(c), N.ptr(mn), N.ptr(mx), N.ptr(off), N.ptr(idx) if idx.size else None, leaves.count), "gs_upload_splat_tree")

    def gather_for_sort(self, model_view64, cos_fov_x_over_2: float, cos_fov_y_over_2: float, gather_all: bool = False) -> int:
        """Viewer.gatherSceneNodesForSort on the GPU: fills the engine's indexesToSort, returns splatRenderCount."""
        mv = np.ascontiguousarray(model_view64, dtype=np.float64).reshape(16)
        rc = C.c_uint32(0)
        N.check(self._lib.gs_gather_for_sort(self._h, N.ptr(mv), float(cos_fov_x_over_2), float(cos_fov_y_over_2), 1 if gather_all else 0, C.byref(rc)), "gs_gather_for_sort")
        return int(rc.value)

    def sort_gathered(self, mvp, sort_count: int, render_count: int, *, out: np.ndarray | None = None, download: bool = True, transforms=None):
        """gs_sort over the index list gs_gather_for_sort left on the device."""
        ptr, _ = self.buffer_dev(N.GS_BUF_INDEXES_TO_SORT)
        p = self._sort_params(mvp, sort_count, render_count, None, transforms, None, indexes_dev=ptr)
        if download and out is None:
            out = np.empty(render_count, np.uint32)
        ms = C.c_float(0)
        N.check(self._lib.gs_sort(self._h, C.byref(p), N.ptr(out) if download else None, C.byref(ms)), "gs_sort")
        return (out if download else None), ms.value

    def compute_distances(self, mvp64, count: int, scene_transforms64=None) -> np.ndarray:
        m = np.ascontiguousarray(mvp64, dtype=np.float64).reshape(16)
        st = None if scene_transforms64 is None else np.ascontiguousarray(scene_transforms64, dtype=np.float64).reshape(-1)
        out = np.empty(count, np.int32 if self.integer_based_sort else np.float32)
        N.check(self._lib.gs_compute_distances(self._h, N.ptr(m), N.ptr(st), count, N.ptr(out)), "gs_compute_distances")
        return out

    # -- rasteriser --------------------------------------------------------------------------------------------
    def upload_splat_data(self, centers_colors: np.ndarray, covariances: np.ndarray | None, sh: np.ndarray | None = None,
                          sh_degree: int = 0, scene_indexes: np.ndarray | None = None, start: int = 0, *,
                          scale_rotations: np.ndarray | None = None) -> None:
        """`scale_rotations` (f32 [n, 6] = sx sy sz qx qy qz): the data a TwoD engine renders from; it ignores `covariances`."""
        cc = np.ascontiguousarray(centers_colors, dtype=np.uint32).reshape(-1, 4)
        d = N.gs_splat_data()
        d.struct_size = C.sizeof(N.gs_splat_data)
        d.from_, d.count = start, cc.shape[0]
        d.centers_colors = N.ptr(cc)
        keep = [cc]
        if covariances is not None:
            cov = np.ascontiguousarray(covariances)
            if cov.dtype == np.float16:
                d.cov_format = N.GS_COV_F16
            else:
                cov = np.ascontiguousarray(cov, dtype=np.float32)
                d.cov_format = N.GS_COV_F32
            d.covariances = N.ptr(cov)
            keep.append(cov)
        if scale_rotations is not None:
            sr = np.ascontiguousarray(scale_rotations, dtype=np.float32).reshape(-1, 6)
            d.scale_rotations = N.ptr(sr)
            keep.append(sr)
        d.sh_degree = sh_degree if sh is not None else 0
        d.sh_format = N.GS_SH_NONE
        if sh is not None and sh_degree > 0:
            s = np.ascontiguousarray(sh)
            if s.dtype == np.float16:
                d.sh_format = N.GS_SH_F16
            elif s.dtype == np.uint8:
                d.sh_format = N.GS_SH_U8
            else:
                s = np.ascontiguousarray(s, dtype=np.float32)
                d.sh_format = N.GS_SH_F32
            d.spherical_harmonics = N.ptr(s)
            keep.append(s)
        if scene_indexes is not None:
            si = np.ascontiguousarray(scene_indexes, dtype=np.uint32)
            d.scene_indexes = N.ptr(si)
            keep.append(si)
        N.check(self._lib.gs_upload_splat_data(self._h, C.byref(d)), "gs_upload_splat_data")

    def upload_ksplat(self, data: bytes, *, minimum_alpha: int = 1, half_covariances: bool = False, upload_sort_centers: bool = True,
                      transform16=None) -> dict:
        """Decode a .ksplat buffer on the GPU into the splat data AND the sorter's centres (gs_upload_ksplat).
        `transform16` (column-major 4x4): static scene transform baked into centres, covariances and spherical harmonics."""
        o = N.gs_ksplat_options()
        o.struct_size = C.sizeof(N.gs_ksplat_options)
        o.minimum_alpha, o.half_covariances, o.upload_sort_centers = minimum_alpha, 1 if half_covariances else 0, 1 if upload_sort_centers else 0
        if transform16 is not None:
            o.has_transform = 1
            o.transform[:] = [float(v) for v in np.asarray(transform16, np.float64).reshape(16)]
        info = N.gs_ksplat_info()
        buf = np.frombuffer(data, dtype=np.uint8)
        N.check(self._lib.gs_upload_ksplat(self._h, N.ptr(buf), buf.size, C.byref(o), C.byref(info)), "gs_upload_ksplat")
        return dict(splat_count=info.splat_count, sh_degree=info.sh_degree, compression_level=info.compression_level, section_count=info.section_count,
                    scene_center=tuple(info.scene_center), min_sh_coeff=info.min_sh_coeff, max_sh_coeff=info.max_sh_coeff)

    def read_buffer(self, buffer_id: int, dtype, count: int, offset_bytes: int = 0) -> np.ndarray:
        out = np.empty(count, dtype)
        N.check(self._lib.gs_read_buffer(self._h, buffer_id, N.ptr(out), offset_bytes, out.nbytes), "gs_read_buffer")
        return out

    @staticmethod
    def _render_params(width, height, render_count, sorted_indexes, fmt, flip_y):
        p = N.gs_render_params()
        p.struct_size = C.sizeof(N.gs_render_params)
        p.width, p.height, p.render_count = width, height, render_count
        keep = None
        if sorted_indexes is not None:
            keep = np.ascontiguousarray(sorted_indexes, dtype=np.uint32)
            p.sorted_indexes = N.ptr(keep)
        p.frame_format = fmt
        p.flip_y = 1 if flip_y else 0
        return p, keep

    def _frame_shape(self, width, height, fmt):
        return (height, width, 4), (np.uint8 if fmt == N.GS_FRAME_RGBA8 else np.float32)

    def render(self, uniforms: Uniforms, width: int, height: int, render_count: int, sorted_indexes=None, *,
               frame_format: int = N.GS_FRAME_RGBA32F, flip_y: bool = False, out: np.ndarray | None = None, download: bool = True):
        """renderer.render(splatMesh, camera).  Returns the frame (rows, width, 4); row 0 = bottom unless flip_y."""
        p, keep = self._render_params(width, height, render_count, sorted_indexes, frame_format, flip_y)
        u = uniforms.to_c()
        shape, dt = self._frame_shape(width, height, frame_format)
        if download and out is None:
            out = np.empty(shape, dt)
        N.check(self._lib.gs_render(self._h, C.byref(u), C.byref(p), N.ptr(out) if download else None), "gs_render")
        del keep
        return out if download else None

    def frame(self, mvp, uniforms: Uniforms, width: int, height: int, render_count: int, indexes=None, *,
              frame_format: int = N.GS_FRAME_RGBA8, flip_y: bool = True, frame_out: np.ndarray | None = None,
              sorted_out: np.ndarray | None = None, download: bool = True, transforms=None):
        """One viewer frame: full depth sort + render (Viewer.update + Viewer.render).  `transforms`: per-scene matrices of a dynamic mesh."""
        sp = self._sort_params(mvp, render_count, render_count, indexes, transforms, None)
        rp, _ = self._render_params(width, height, render_count, None, frame_format, flip_y)
        u = uniforms.to_c()
        shape, dt = self._frame_shape(width, height, frame_format)
        if download and frame_out is None:
            frame_out = np.empty(shape, dt)
        N.check(self._lib.gs_frame(self._h, C.byref(sp), C.byref(u), C.byref(rp), N.ptr(sorted_out), N.ptr(frame_out) if download else None), "gs_frame")
        return frame_out if download else None

    def frame_async(self, mvp, uniforms: Uniforms, width: int, height: int, render_count: int, *, frame_format: int = N.GS_FRAME_RGBA8,
                    flip_y: bool = True, prepared=None):
        """Enqueue one frame without waiting (gs_frame_async).  `prepared` = a tuple from prepare_frame() to skip re-marshalling."""
        if prepared is None:
            prepared = self.prepare_frame(mvp, uniforms, width, height, render_count, frame_format=frame_format, flip_y=flip_y)
        sp, u, rp = prepared
        N.check(self._lib.gs_frame_async(self._h, C.byref(sp), C.byref(u), C.byref(rp)), "gs_frame_async")

    def prepare_frame(self, mvp, uniforms: Uniforms, width: int, height: int, render_count: int, *, frame_format: int = N.GS_FRAME_RGBA8,
                      flip_y: bool = True):
        sp = self._sort_params(mvp, render_count, render_count, None, None, None)
        rp, _ = self._render_params(width, height, render_count, None, frame_format, flip_y)
        return sp, uniforms.to_c(), rp

    def frame_prepared(self, prepared, frame_out: np.ndarray | None, sorted_out: np.ndarray | None = None) -> None:
        """gs_frame with pre-marshalled arguments (host buffers: frame_out / sorted_out may be pinned arrays)."""
        sp, u, rp = prepared
        N.check(self._lib.gs_frame(self._h, C.byref(sp), C.byref(u), C.byref(rp), N.ptr(sorted_out), N.ptr(frame_out)), "gs_frame")

    def frame_begin(self, prepared, frame_out: np.ndarray | None) -> None:
        """Pipelined frame (gs_frame_begin): enqueue the frame and the copy of its picture into `frame_out` (pinned host array);
        at most three frames in flight, each with its own `frame_out`.  `prepared` = prepare_frame(...)."""
        sp, u, rp = prepared
        N.check(self._lib.gs_frame_begin(self._h, C.byref(sp), C.byref(u), C.byref(rp), N.ptr(frame_out)), "gs_frame_begin")

    def frame_end(self) -> None:
        """Wait for the oldest pipelined frame: its frame_out is complete on return."""
        N.check(self._lib.gs_frame_end(self._h), "gs_frame_end")

    def peer_export(self) -> tuple[bytes, bytes]:
        """Rank 0: CUDA-IPC handles (frame buffer, handshake block) for the fused tile gather."""
        a, b = C.create_string_buffer(64), C.create_string_buffer(64)
        N.check(self._lib.gs_peer_export(self._h, a, b), "gs_peer_export")
        return a.raw, b.raw

    def peer_attach(self, frame_handle: bytes, sync_handle: bytes) -> None:
        """Ranks > 0: blend straight into rank 0's frame over NVLink from now on."""
        N.check(self._lib.gs_peer_attach(self._h, C.create_string_buffer(frame_handle, 64), C.create_string_buffer(sync_handle, 64)), "gs_peer_attach")

    def set_graph_enabled(self, on: bool) -> None:
        N.check(self._lib.gs_set_graph_enabled(self._h, 1 if on else 0), "gs_set_graph_enabled")

    def set_profiling(self, on: bool) -> None:
        N.check(self._lib.gs_set_profiling(self._h, 1 if on else 0), "gs_set_profiling")

    def kernel_timings(self) -> list[tuple[str, float]]:
        """[(kernel name, device ms)] of the last sort / render / frame, in launch order (needs set_profiling(True))."""
        buf = (N.gs_kernel_time * 64)()
        n = C.c_uint32(0)
        N.check(self._lib.gs_kernel_timings(self._h, buf, 64, C.byref(n)), "gs_kernel_timings")
        return [(buf[i].name.decode(), buf[i].ms) for i in range(min(n.value, 64))]

    def flush_l2(self) -> None:
        N.check(self._lib.gs_flush_l2(self._h), "gs_flush_l2")

    def event(self) -> "DeviceEvent":
        return DeviceEvent(self)

    def read_projected(self, count: int) -> np.ndarray:
        out = np.empty(count, N.PROJECTED_DTYPE)
        N.check(self._lib.gs_read_projected(self._h, N.ptr(out), count), "gs_read_projected")
        return out

    def read_projected_2d(self, count: int) -> np.ndarray:
        """TwoD engines: the vertex-stage output of every splat for the last frame's camera (gs_read_projected_2d)."""
        out = np.empty(count, N.PROJECTED_SURFEL_DTYPE)
        N.check(self._lib.gs_read_projected_2d(self._h, N.ptr(out), count), "gs_read_projected_2d")
        return out

    # -- device access -------------------------------------------------------------------------------------------
    def buffer_dev(self, buffer_id: int) -> tuple[int, int]:
        p, b = C.c_void_p(), C.c_size_t()
        N.check(self._lib.gs_buffer_dev(self._h, buffer_id, C.byref(p), C.byref(b)), "gs_buffer_dev")
        return int(p.value or 0), int(b.value)

    def stream(self) -> int:
        s = C.c_void_p()
        N.check(self._lib.gs_stream(self._h, C.byref(s)), "gs_stream")
        return int(s.value or 0)

    def synchronize(self) -> None:
        N.check(self._lib.gs_synchronize(self._h), "gs_synchronize")

    def timings(self) -> dict:
        t = N.gs_timings()
        N.check(self._lib.gs_last_timings(self._h, C.byref(t)), "gs_last_timings")
        return t.as_dict()


class DeviceEvent:
    """CUDA event recorded on the engine's stream (gs_event_*)."""

    def __init__(self, engine: Engine):
        self._e = engine
        self._ev = C.c_void_p()
        N.check(engine._lib.gs_event_create(C.byref(self._ev)), "gs_event_create")

    def record(self) -> None:
        N.check(self._e._lib.gs_event_record(self._e._h, self._ev), "gs_event_record")

    def elapsed_ms(self, later: "DeviceEvent") -> float:
        ms = C.c_float(0)
        N.check(self._e._lib.gs_event_elapsed_ms(self._ev, later._ev, C.byref(ms)), "gs_event_elapsed_ms")
        return ms.value

    def __del__(self):
        try:
            self._e._lib.gs_event_destroy(self._ev)
        except Exception:
            pass


def sort_indexes(indexes, centers, precomputed, mvp, scene_indexes, transforms, distance_map_range, sort_count, render_count,
                 splat_count, use_precomputed, integer_sort, dynamic_mode, *, want_scratch: bool = False):
    """Call the stateless drop-in gs_sort_indexes exactly as a test would call the reference's sortIndexes().

    Returns indexesOut (and mappedDistances, frequencies when want_scratch)."""
    lib = N.load()
    idx = np.ascontiguousarray(indexes, dtype=np.uint32)
    cen = None if centers is None else np.ascontiguousarray(centers)
    pre = None if precomputed is None else np.ascontiguousarray(precomputed)
    m = np.ascontiguousarray(mvp, dtype=np.float32).reshape(16)
    si = None if scene_indexes is None else np.ascontiguousarray(scene_indexes, dtype=np.uint32)
    tr = None
    if transforms is not None:
        tr = np.zeros(16 * N.GS_MAX_SCENES, np.float32)
        t = np.asarray(transforms, np.float32).reshape(-1)
        tr[: t.size] = t
    out = np.full(max(render_count, 1), 0xFFFFFFFF, np.uint32)
    mapped = np.zeros(max(render_count, 1), np.int32) if want_scratch else None
    freq = np.zeros(distance_map_range, np.uint32) if want_scratch else None
    rc = lib.gs_sort_indexes(N.ptr(idx), N.ptr(cen), N.ptr(pre), N.ptr(mapped), N.ptr(freq), N.ptr(m), N.ptr(out), N.ptr(si), N.ptr(tr),
                             distance_map_range, sort_count, render_count, splat_count, bool(use_precomputed), bool(integer_sort), bool(dynamic_mode))
    N.check(rc, "gs_sort_indexes")
    out = out[:render_count]
    if want_scratch:
        return out, mapped[:render_count], freq
    return out
