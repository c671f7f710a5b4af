"""Host-side mirror of the slice of the reference's Viewer / SplatMesh that drives the hot path.

    SplatMesh.build(...)                  src/splatmesh/SplatMesh.js:306-405    -> SplatMesh.build
    SplatMesh.getIntegerCenters/Float...  :1912-1948                            -> SplatMesh.getIntegerCenters / getFloatCenters
    SplatMesh.updateRenderIndexes         :1228-1235                            -> SplatMesh.updateRenderIndexes
    SplatMesh.updateUniforms              :1248-1280                            -> SplatMesh.updateUniforms
    Viewer.runSplatSort                   src/Viewer.js:1833-1964               -> Viewer.runSplatSort
    Viewer.updateSplatMesh                :651-677                              -> Viewer.updateSplatMesh
    Viewer.render                         :1599-1623                            -> Viewer.render
    Viewer.update                         :1625-1644                            -> Viewer.update

Only the arithmetic-free orchestration lives here (matrix set-up in float64 like three.js, message passing, option
bag).  Sorting and rasterisation run in libgsplat_b200.so through Engine / SortWorker.  Everything the reference does
around the path (loading UI, controls, octree culling, WebXR ...) is out of scope (SURVEY.md section 2).
"""
from __future__ import annotations

import numpy as np

from . import _native as N
from . import three_math as TM
from .engine import Engine, Uniforms
from .scenes import PackedScene, RawScene, float_centers, integer_centers, pack_scene
from .sort_worker import DefaultSplatSortDistanceMapPrecision, createSortWorker, start
from .splat_tree import SplatTree, fov_cosines

THREE_CAMERA_FOV = 50  # Viewer.js:30


class SplatRenderMode:
    """src/SplatRenderMode.js: the Viewer option `splatRenderMode` (Viewer.js:199-202)."""
    ThreeD = 0
    TwoD = 1


class SplatMesh:
    """Owns the GPU-side splat data of one (static) scene and the uniforms of the splat material."""

    def __init__(self, *, dynamicMode=False, halfPrecisionCovariancesOnGPU=False, devicePixelRatio=1.0, antialiased=False,
                 maxScreenSpaceSplatSize=1024, splatScale=1.0, pointCloudModeEnabled=False, sphericalHarmonicsDegree=0,
                 kernel2DSize=0.3, enableOptionalEffects=False, splatRenderMode=SplatRenderMode.ThreeD):
        self.dynamicMode = dynamicMode
        self.splatRenderMode = int(splatRenderMode)
        self.halfPrecisionCovariancesOnGPU = halfPrecisionCovariancesOnGPU
        self.devicePixelRatio = devicePixelRatio
        self.antialiased = antialiased
        self.maxScreenSpaceSplatSize = maxScreenSpaceSplatSize
        self.splatScale = splatScale
        self.pointCloudModeEnabled = pointCloudModeEnabled
        self.sphericalHarmonicsDegree = sphericalHarmonicsDegree
        self.kernel2DSize = kernel2DSize
        self.enableOptionalEffects = enableOptionalEffects
        self.matrixWorld = TM.identity()
        self.packed: PackedScene | None = None
        self.raw: RawScene | None = None
        self.uniforms: dict = {}
        self.renderIndexes: np.ndarray | None = None
        self.instanceCount = 0
        self.engine: Engine | None = None
        self.visibleRegionFadeStartRadius = 0.0
        self.fadeInComplete = True
        self.sceneCenter = (0.0, 0.0, 0.0)
        # per-scene transforms of a dynamic mesh (SplatScene.transform, SplatScene.js:28-36; uploaded every frame by
        # fillTransformsArray, SplatMesh.js:1660-1673): column-major f64, scene 0 = the one scene this mirror holds
        self.sceneTransforms = np.tile(TM.identity(), (N.GS_MAX_SCENES, 1))
        self.splatTree: SplatTree | None = None

    def build(self, raw_scene: RawScene, *, sh_format: str = "f16", transform16=None) -> None:
        """Decode + pack the scene like refreshGPUDataFromSplatBuffers (SplatMesh.js:588-603) and keep it for upload.
        `transform16` (column-major 4x4, the SplatScene's position/quaternion/scale): baked into centres, covariances and SH when
        the mesh is static (fillSplatDataArrays' applySceneTransform default, SplatMesh.js:1872-1883); a dynamic mesh keeps the
        data untouched and applies its transforms per frame in the sorter and the vertex stage."""
        if transform16 is not None and self.dynamicMode:
            self.sceneTransforms[0] = np.asarray(transform16, np.float64).reshape(16)     # applied per frame, not baked
            transform16 = None
        if transform16 is not None:
            from .scenes import transform_scene
            self.raw = transform_scene(raw_scene, transform16)[0]      # what the sorter's centres are taken from
        else:
            self.raw = raw_scene
        degree = min(self.sphericalHarmonicsDegree, raw_scene.sh_degree)
        if degree < raw_scene.sh_degree:  # minSphericalHarmonicsDegree clamp (SplatMesh.js:680-683)
            ncoef = 0 if degree == 0 else (3 if degree == 1 else 8)
            raw_scene = RawScene(raw_scene.centers, raw_scene.scales, raw_scene.rotations, raw_scene.colors,
                                 None if degree == 0 else raw_scene.sh[:, :ncoef], degree)
        self.packed = pack_scene(raw_scene, half_covariances=self.halfPrecisionCovariancesOnGPU, sh_format=sh_format, transform16=transform16,
                                 render_mode=self.splatRenderMode)

    def fillTransformsArray(self) -> np.ndarray:  # noqa: N802  SplatMesh.js:1660-1673
        """f32[32 x 16] for the sorter ('transforms' of the sort message) and the vertex stage (`transforms` uniform)."""
        return self.sceneTransforms.astype(np.float32)

    def buildSplatTree(self, minAlpha: int = 1) -> SplatTree:  # noqa: N802,N803  SplatMesh.js:231-279
        """new SplatTree(8, 1000).processSplatMesh(this, alpha >= minAlpha): the octree over the (transformed) centres."""
        tree = SplatTree(8, 1000)
        tree.processSplatMesh(self.raw.centers, self.raw.colors[:, 3], minAlpha)
        self.splatTree = tree
        return tree

    def getSplatTree(self):  # noqa: N802  SplatMesh.js:557-559
        return self.splatTree

    def getSplatCount(self) -> int:  # noqa: N802
        return 0 if self.packed is None else self.packed.count

    def getIntegerCenters(self, start: int, end: int, padFour: bool = False) -> np.ndarray:  # noqa: N802,N803
        c = integer_centers(self.raw.centers[start:end + 1])
        return c if padFour else c[:, :3].copy()

    def getFloatCenters(self, start: int, end: int, padFour: bool = False) -> np.ndarray:  # noqa: N802,N803
        c = float_centers(self.raw.centers[start:end + 1])
        return c if padFour else c[:, :3].copy()

    def setRenderer(self, engine: Engine) -> None:  # noqa: N802
        """The WebGL renderer of the reference (SplatMesh.js:1300-1340) becomes the CUDA engine; uploads the 'textures'."""
        self.engine = engine
        p = self.packed
        engine.upload_splat_data(p.centers_colors, p.covariances, p.sh, p.sh_degree, scale_rotations=p.scale_rotations)

    def updateRenderIndexes(self, globalIndexes: np.ndarray | None, renderSplatCount: int) -> None:  # noqa: N802,N803
        """SplatMesh.js:1228-1235.  globalIndexes None = keep the order the engine's last sort left on the device."""
        self.renderIndexes = globalIndexes
        self.instanceCount = int(renderSplatCount)

    def updateUniforms(self, renderDimensions, cameraFocalLengthX, cameraFocalLengthY, orthographicMode, orthographicZoom,  # noqa: N802,N803
                       inverseFocalAdjustment) -> None:
        vw, vh = renderDimensions[0] * self.devicePixelRatio, renderDimensions[1] * self.devicePixelRatio
        self.uniforms.update(viewport=(vw, vh), basisViewport=(1.0 / vw, 1.0 / vh), focal=(cameraFocalLengthX, cameraFocalLengthY),
                             orthographicMode=1 if orthographicMode else 0, orthoZoom=orthographicZoom,
                             inverseFocalAdjustment=inverseFocalAdjustment)


class Viewer:
    """Frame loop of the reference's Viewer reduced to the hot path: update() -> runSplatSort + updateSplatMesh, render()."""

    def __init__(self, options: dict | None = None):
        o = dict(options or {})
        self.cameraUp = np.asarray(o.get("cameraUp", (0, 1, 0)), np.float64)            # Viewer.js:51
        self.initialCameraPosition = np.asarray(o.get("initialCameraPosition", (0, 10, 15)), np.float64)
        self.initialCameraLookAt = np.asarray(o.get("initialCameraLookAt", (0, 0, 0)), np.float64)
        self.renderWidth = int(o.get("width", 1920))
        self.renderHeight = int(o.get("height", 1080))
        self.devicePixelRatio = float(o.get("devicePixelRatio", 1.0))
        self.gpuAcceleratedSort = bool(o.get("gpuAcceleratedSort", False))                  # Viewer.js:90
        self.integerBasedSort = bool(o.get("integerBasedSort", True))                       # Viewer.js:95-98
        self.sharedMemoryForWorkers = bool(o.get("sharedMemoryForWorkers", True))
        self.enableSIMDInSort = bool(o.get("enableSIMDInSort", True))
        self.dynamicScene = bool(o.get("dynamicScene", False))
        self.antialiased = bool(o.get("antialiased", False))
        self.kernel2DSize = float(o.get("kernel2DSize", 0.3))
        self.sphericalHarmonicsDegree = int(o.get("sphericalHarmonicsDegree", 0))
        self.focalAdjustment = float(o.get("focalAdjustment", 1.0))
        self.maxScreenSpaceSplatSize = float(o.get("maxScreenSpaceSplatSize", 1024))
        self.halfPrecisionCovariancesOnGPU = bool(o.get("halfPrecisionCovariancesOnGPU", False))
        self.splatRenderMode = int(o.get("splatRenderMode", SplatRenderMode.ThreeD))      # Viewer.js:199-202
        if self.splatRenderMode not in (SplatRenderMode.ThreeD, SplatRenderMode.TwoD):
            raise ValueError(f"splatRenderMode {self.splatRenderMode} is neither SplatRenderMode.ThreeD nor TwoD")
        prec = int(o.get("splatSortDistanceMapPrecision", DefaultSplatSortDistanceMapPrecision))
        self.splatSortDistanceMapPrecision = int(np.clip(prec, 10, 20 if self.integerBasedSort else 24))  # Viewer.js:207-210
        self.device = int(o.get("device", 0))
        self.rank, self.world_size = int(o.get("rank", 0)), int(o.get("world_size", 1))
        self.camera = TM.PerspectiveCamera(THREE_CAMERA_FOV, self.renderWidth / self.renderHeight, 0.1, 1000)  # Viewer.js:338
        self.camera.position = self.initialCameraPosition.copy()
        self.camera.up = self.cameraUp / np.linalg.norm(self.cameraUp)
        self.camera.look_at(self.initialCameraLookAt)
        self.splatMesh: SplatMesh | None = None
        self.engine: Engine | None = None
        self.sortWorker = None
        self.sortRunning = False
        self.splatRenderCount = 0
        self.splatSortCount = 0
        self.lastSortTime = 0.0
        self.sortWorkerIndexesToSort: np.ndarray | None = None
        self.sortWorkerSortedIndexes: np.ndarray | None = None
        self._sorted_on_device = False
        self.enableSplatTree = bool(o.get("splatTree", False))   # the reference always builds its tree; the benchmark configs sort all splats, so opt-in
        # runSplatSort's closure state (Viewer.js:1835-1841)
        self._lastSortViewDir = np.array([0.0, 0.0, -1.0])
        self._lastSortViewPos = np.zeros(3)
        self._queuedSorts: list[int] = []
        self._gathered = False

    # -- scene set-up (addSplatBuffers / setupSortWorker, Viewer.js:1094-1300) ------------------------------------------------
    def addSplatScene(self, raw_scene: RawScene, *, separate_sort_worker: bool = False, position=(0.0, 0.0, 0.0),  # noqa: N802
                      rotation=(0.0, 0.0, 0.0, 1.0), scale=(1.0, 1.0, 1.0)) -> None:
        """Viewer.addSplatScene's `position` / `rotation` (quaternion x, y, z, w) / `scale` options (Viewer.js:736-760): the
        SplatScene transform, baked at load for a static mesh."""
        self.splatMesh = SplatMesh(dynamicMode=self.dynamicScene, halfPrecisionCovariancesOnGPU=self.halfPrecisionCovariancesOnGPU,
                                   devicePixelRatio=self.devicePixelRatio, antialiased=self.antialiased,
                                   maxScreenSpaceSplatSize=self.maxScreenSpaceSplatSize, sphericalHarmonicsDegree=self.sphericalHarmonicsDegree,
                                   kernel2DSize=self.kernel2DSize, splatRenderMode=self.splatRenderMode)
        identity = tuple(position) == (0.0, 0.0, 0.0) and tuple(rotation) == (0.0, 0.0, 0.0, 1.0) and tuple(scale) == (1.0, 1.0, 1.0)
        self.splatMesh.build(raw_scene, transform16=None if identity else TM.compose(position, rotation, scale))
        n = self.splatMesh.getSplatCount()
        self.engine = Engine(n, device=self.device, distance_map_range=1 << self.splatSortDistanceMapPrecision,
                             integer_based_sort=self.integerBasedSort, dynamic_mode=self.dynamicScene,
                             max_width=self.renderWidth, max_height=self.renderHeight, rank=self.rank, world_size=self.world_size,
                             splat_render_mode=self.splatRenderMode)
        self.splatMesh.setRenderer(self.engine)
        centers = (self.splatMesh.getIntegerCenters(0, n - 1, True) if self.integerBasedSort else self.splatMesh.getFloatCenters(0, n - 1, True))
        if separate_sort_worker:
            # the reference's topology: a worker with its own memory, sorted indexes travel back through the host
            self.sortWorker = createSortWorker(n, self.sharedMemoryForWorkers, self.enableSIMDInSort, self.integerBasedSort,
                                               self.dynamicScene, self.splatSortDistanceMapPrecision, device=self.device)
            self.sortWorker.onmessage = self._on_worker_message
            start(self.sortWorker)
            self.sortWorker.postMessage({"centers": centers, "sceneIndexes": None, "range": {"from": 0, "to": n - 1, "count": n}})
        else:
            self.engine.upload_centers(centers, np.zeros(n, np.uint32) if self.dynamicScene else None)
        self.splatRenderCount = n
        if self.enableSplatTree:
            self.engine.upload_splat_tree(self.splatMesh.buildSplatTree().leaves)

    def addSplatSceneFromKSplat(self, data: bytes, *, position=(0.0, 0.0, 0.0), rotation=(0.0, 0.0, 0.0, 1.0), scale=(1.0, 1.0, 1.0)) -> dict:  # noqa: N802
        """Viewer.addSplatScene for a `.ksplat` buffer (KSplatLoader.loadFromFileData -> new SplatBuffer -> SplatMesh.build ->
        'centers' message, Viewer.js:736-868, 1094-1167): header parsing on the host, every per-splat decode on the GPU.
        position / rotation (x, y, z, w) / scale: the SplatScene transform, baked by the decode kernel (static mesh)."""
        from . import ksplat as K
        hdr = K.parse(data)
        n = hdr.max_splat_count
        self.splatMesh = SplatMesh(dynamicMode=False, halfPrecisionCovariancesOnGPU=self.halfPrecisionCovariancesOnGPU,
                                   devicePixelRatio=self.devicePixelRatio, antialiased=self.antialiased,
                                   maxScreenSpaceSplatSize=self.maxScreenSpaceSplatSize, sphericalHarmonicsDegree=self.sphericalHarmonicsDegree,
                                   kernel2DSize=self.kernel2DSize, splatRenderMode=self.splatRenderMode)
        self.engine = Engine(n, device=self.device, distance_map_range=1 << self.splatSortDistanceMapPrecision,
                             integer_based_sort=self.integerBasedSort, dynamic_mode=False, max_width=self.renderWidth, max_height=self.renderHeight,
                             rank=self.rank, world_size=self.world_size, splat_render_mode=self.splatRenderMode)
        identity = tuple(position) == (0.0, 0.0, 0.0) and tuple(rotation) == (0.0, 0.0, 0.0, 1.0) and tuple(scale) == (1.0, 1.0, 1.0)
        info = self.engine.upload_ksplat(data, half_covariances=self.halfPrecisionCovariancesOnGPU,
                                         transform16=None if identity else TM.compose(position, rotation, scale))
        self.splatMesh.engine = self.engine
        degree = min(self.sphericalHarmonicsDegree, info["sh_degree"])
        self.splatMesh.packed = PackedScene(None, None, None, degree, None, info["splat_count"])
        self.splatMesh.sceneCenter = info["scene_center"]
        self._ksplat_info = info
        self.splatRenderCount = info["splat_count"]
        return info

    def _on_worker_message(self, e) -> None:  # Viewer.js:1243-1298
        d = e.data
        if d.get("sortDone"):
            self.sortRunning = False
            self.lastSortTime = d["sortTime"]
            sorted_idx = self.sortWorkerSortedIndexes if self.sharedMemoryForWorkers else d["sortedIndexes"]
            self.splatMesh.updateRenderIndexes(sorted_idx[: d["splatRenderCount"]], d["splatRenderCount"])
        elif d.get("sortSetupPhase1Complete"):
            if self.sharedMemoryForWorkers:
                self.sortWorkerIndexesToSort = d["indexesToSortBuffer"]
                self.sortWorkerSortedIndexes = d["sortedIndexesBuffer"]
                self.sortWorkerIndexesToSort[:] = np.arange(self.sortWorkerIndexesToSort.shape[0], dtype=np.uint32)  # Viewer.js:1282-1284

    # -- matrices ----------------------------------------------------------------------------------------------------------------
    def mvp_matrix(self) -> np.ndarray:
        """Viewer.js:1888-1891 in float64: projection * inverse(camera.matrixWorld) * splatMesh.matrixWorld."""
        m = TM.invert(self.camera.matrixWorld)
        m = TM.multiply(self.camera.projectionMatrix, m)
        if not self.splatMesh.dynamicMode:
            m = TM.multiply(m, self.splatMesh.matrixWorld)
        return m

    def updateSplatMesh(self) -> None:  # noqa: N802  Viewer.js:651-677
        w, h = self.renderWidth, self.renderHeight
        fx = self.camera.projectionMatrix[0] * 0.5 * self.devicePixelRatio * w
        fy = self.camera.projectionMatrix[5] * 0.5 * self.devicePixelRatio * h
        fa = self.focalAdjustment * (1.0 / self.devicePixelRatio if self.camera.isOrthographicCamera else 1.0)
        self.splatMesh.updateUniforms((w, h), fx * fa, fy * fa, self.camera.isOrthographicCamera, self.camera.zoom or 1.0, 1.0 / fa)

    def uniforms(self) -> Uniforms:
        """What three.js + SplatMesh hand the splat shaders for the current camera."""
        sm = self.splatMesh
        mv = TM.multiply(self.camera.matrixWorldInverse, sm.matrixWorld)
        u = sm.uniforms
        dyn = {}
        if sm.dynamicMode:      # SplatMaterial.js:136-146: transformModelViewMatrix = viewMatrix * transforms[sceneIndex]
            dyn = dict(dynamic_mode=1, scene_transforms=sm.fillTransformsArray(), view_matrix=self.camera.matrixWorldInverse.astype(np.float32), scene_count=1)
        return Uniforms(**dyn, model_view=mv.astype(np.float32), projection=self.camera.projectionMatrix.astype(np.float32),
                        camera_position=np.asarray(self.camera.position, np.float32), focal=u["focal"], viewport=u["viewport"],
                        inverse_focal_adjustment=u["inverseFocalAdjustment"], ortho_zoom=u["orthoZoom"], orthographic_mode=u["orthographicMode"],
                        splat_scale=sm.splatScale, point_cloud_mode=1 if sm.pointCloudModeEnabled else 0,
                        sh_degree=sm.packed.sh_degree, antialiased=1 if sm.antialiased else 0, kernel_2d_size=sm.kernel2DSize,
                        max_screen_space_splat_size=sm.maxScreenSpaceSplatSize, fade_in_complete=1 if sm.fadeInComplete else 0,
                        sh8_min=np.full(N.GS_MAX_SCENES, getattr(self, "_ksplat_info", {}).get("min_sh_coeff", -1.5), np.float32),
                        sh8_max=np.full(N.GS_MAX_SCENES, getattr(self, "_ksplat_info", {}).get("max_sh_coeff", 1.5), np.float32),
                        scene_center=sm.sceneCenter, visible_region_fade_start_radius=sm.visibleRegionFadeStartRadius)

    # -- the per-frame path --------------------------------------------------------------------------------------------------------
    def gatherSceneNodesForSort(self, gatherAllNodes: bool = False) -> tuple[int, bool]:  # noqa: N802,N803  Viewer.js:1969-2077
        """(splatRenderCount, shouldSortAll).  With a SplatTree: every leaf is culled against the frustum and the kept leaves' indexes are
        laid out nearest-last in the sorter's indexesToSort -- on the GPU (gs_gather_for_sort); without one: identity, sort all."""
        tree = self.splatMesh.getSplatTree()
        if tree is None or tree.leaves is None:
            self._gathered = False
            return self.splatMesh.getSplatCount(), True
        base = TM.invert(self.camera.matrixWorld)
        if not self.splatMesh.dynamicMode:
            base = TM.multiply(base, self.splatMesh.matrixWorld)
        cx, cy = fov_cosines(self.renderWidth * self.devicePixelRatio, self.renderHeight * self.devicePixelRatio, self.camera.fov)
        count = self.engine.gather_for_sort(base, cx, cy, gatherAllNodes)
        self._gathered = True
        return count, False

    def runSplatSort(self, force: bool = False, forceSortAll: bool = False) -> bool:  # noqa: N802,N803  Viewer.js:1833-1964
        """The reference's scheduling: skip while the view has barely changed, gather the visible leaves, and after a large rotation queue
        partial sorts of the nearest 12.5 % / 33 % / 75 % ... before the full one (Viewer.js:1843-1856, 1899-1913)."""
        if self.sortRunning:
            return True
        if self.splatMesh.getSplatCount() <= 0:
            self.splatRenderCount = 0
            return False
        view_dir = -np.asarray(self.camera.matrixWorld[8:11], np.float64)     # (0, 0, -1).applyQuaternion(camera.quaternion)
        angle_diff = float(np.dot(view_dir, self._lastSortViewDir))
        position_diff = float(np.linalg.norm(np.asarray(self.camera.position, np.float64) - self._lastSortViewPos))
        if not force and not self.splatMesh.dynamicMode and not self._queuedSorts:
            if not (angle_diff <= 0.99 or position_diff >= 1.0):
                return False
        render_count, should_sort_all = self.gatherSceneNodesForSort()
        should_sort_all = should_sort_all or forceSortAll
        self.splatRenderCount = render_count
        mvp = self.mvp_matrix()
        if not self._queuedSorts:
            if self.splatMesh.dynamicMode or should_sort_all:
                self._queuedSorts.append(render_count)
            else:
                for threshold, fractions in ((0.55, (0.125, 0.33333, 0.75)), (0.65, (0.33333, 0.66667)), (0.8, (0.5,))):
                    if angle_diff < threshold:
                        self._queuedSorts.extend(int(np.floor(render_count * f)) for f in fractions)
                        break
                self._queuedSorts.append(render_count)
        sort_count = min(self._queuedSorts.pop(0), render_count)
        self.splatSortCount = sort_count
        n = render_count
        if self.sortWorker is not None:
            self.sortRunning = True
            msg = {"modelViewProj": mvp.astype(np.float32), "cameraPosition": list(self.camera.position), "splatRenderCount": n,
                   "splatSortCount": sort_count, "usePrecomputedDistances": False}
            if not self.sharedMemoryForWorkers:
                msg["indexesToSort"] = np.arange(n, dtype=np.uint32)
                msg["transforms"] = self.splatMesh.fillTransformsArray() if self.splatMesh.dynamicMode else None
            self.sortWorker.postMessage({"sort": msg})
        else:
            tr = self.splatMesh.fillTransformsArray() if self.splatMesh.dynamicMode else None
            if self._gathered:
                _, ms = self.engine.sort_gathered(mvp.astype(np.float32), sort_count, n, download=False, transforms=tr)
            else:
                _, ms = self.engine.sort(mvp.astype(np.float32), sort_count, n, None, download=False, transforms=tr)
            self.lastSortTime = ms
            self.splatMesh.updateRenderIndexes(None, n)
        if not self._queuedSorts:
            self._lastSortViewPos = np.asarray(self.camera.position, np.float64).copy()
            self._lastSortViewDir = view_dir.copy()
        return True

    def update(self, force_sort: bool = True) -> None:  # Viewer.js:1625-1644
        """force_sort=True sorts on every call (what the tests and the benchmark want); False applies the reference's view-change
        thresholds like its frame loop does."""
        self.camera.update()
        self.runSplatSort(force=force_sort, forceSortAll=force_sort and self.splatMesh.getSplatTree() is None)
        self.updateSplatMesh()

    def render(self, *, frame_format: int = N.GS_FRAME_RGBA8, flip_y: bool = True, download: bool = True):  # Viewer.js:1599-1623
        sm = self.splatMesh
        return self.engine.render(self.uniforms(), self.renderWidth, self.renderHeight, sm.instanceCount, sm.renderIndexes,
                                  frame_format=frame_format, flip_y=flip_y, download=download)

    def frame(self, *, frame_format: int = N.GS_FRAME_RGBA8, flip_y: bool = True, download: bool = True, frame_out=None):
        """update() + render() fused into one engine call (sort order never leaves the device)."""
        self.camera.update()
        self.updateSplatMesh()
        n = self.splatMesh.getSplatCount()
        return self.engine.frame(self.mvp_matrix().astype(np.float32), self.uniforms(), self.renderWidth, self.renderHeight, n, None,
                                 frame_format=frame_format, flip_y=flip_y, download=download, frame_out=frame_out,
                                 transforms=self.splatMesh.fillTransformsArray() if self.splatMesh.dynamicMode else None)

    def dispose(self) -> None:
        if self.sortWorker is not None:
            self.sortWorker.terminate()
        if self.engine is not None:
            self.engine.close()
