"""GPU parity: CUDA projection + tile-binned front-to-back compositing vs the CPU restatement of the reference's
shaders (oracle/raster_oracle.c).  Tolerances (SURVEY 8c): per-splat projection within 1e-3 px / 1e-4 relative on
the basis vectors / 2e-4 on colour; frames max abs err <= 2/255 on >= 99.9 % of channels and <= 8/255 everywhere
(edge pixels where A ~ 8 may flip coverage), measured on float accumulators."""
import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu

TOL_MOST, TOL_WORST, FRAC = 2.0 / 255.0, 8.0 / 255.0, 0.999


def _viewer(gs, raw, width, height, cam="bonsai", **opts):
    from gaussiansplats3d_b200.viewer import Viewer
    from gaussiansplats3d_b200.scenes import CAMERAS
    c = CAMERAS[cam]
    v = Viewer(dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=width, height=height, **opts))
    v.addSplatScene(raw)
    return v


def _oracle_frame(oracle_mod, v, order, quantize8=False):
    p = v.splatMesh.packed
    return oracle_mod.render(v.uniforms(), p.centers_colors, p.covariances, order, v.renderWidth, v.renderHeight, sh=p.sh, sh_degree=p.sh_degree, quantize8=quantize8)


def _check_frame(got, want):
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    assert err.max() <= TOL_WORST, f"worst channel error {err.max() * 255:.2f}/255"
    frac = (err <= TOL_MOST).mean()
    assert frac >= FRAC, f"only {frac * 100:.3f}% of channels within 2/255"
    return err


@pytest.mark.parametrize("sh_degree,fmt", [(0, "f16"), (1, "f16"), (2, "f16"), (2, "u8"), (2, "f32")])
def test_projection_matches_vertex_shader(gs, oracle_mod, sh_degree, fmt):
    from gaussiansplats3d_b200.scenes import synthetic_scene
    from gaussiansplats3d_b200.viewer import Viewer
    raw = synthetic_scene(60_000, seed=4, kind="bonsai", sh_degree=sh_degree)
    v = Viewer(dict(width=640, height=360, sphericalHarmonicsDegree=sh_degree, initialCameraPosition=(1.5, 2.7, -6.4), initialCameraLookAt=(0.4, 0.3, 0.2), cameraUp=(0, -1, -0.6)))
    v.splatMesh = None
    from gaussiansplats3d_b200.viewer import SplatMesh
    v.addSplatScene(raw)
    if fmt != "f16" and sh_degree:
        from gaussiansplats3d_b200.scenes import pack_scene
        v.splatMesh.packed = pack_scene(raw, sh_format=fmt)
        v.splatMesh.setRenderer(v.engine)
    v.update()
    v.render(download=False)
    got = v.engine.read_projected(raw.count)
    p = v.splatMesh.packed
    want = oracle_mod.project(v.uniforms(), p.centers_colors, p.covariances, p.sh, p.sh_degree)
    assert np.array_equal(got["valid"], want["valid"]) or (got["valid"] != want["valid"]).mean() < 1e-4
    m = (got["valid"] == 1) & (want["valid"] == 1)
    assert m.sum() > 1000
    for k in ("cx", "cy"):
        assert np.abs(got[k][m] - want[k][m]).max() < 2e-3, k
    for k in ("b1x", "b1y", "b2x", "b2y"):
        scale = np.maximum(np.hypot(want["b1x"][m], want["b1y"][m]), 1.0)
        # e1 flips sign freely (a quad is symmetric): compare outer products instead of vectors
    q_got = np.stack([got["b1x"] * got["b1x"] + got["b2x"] * got["b2x"], got["b1x"] * got["b1y"] + got["b2x"] * got["b2y"], got["b1y"] * got["b1y"] + got["b2y"] * got["b2y"]], 1)[m]
    q_want = np.stack([want["b1x"] * want["b1x"] + want["b2x"] * want["b2x"], want["b1x"] * want["b1y"] + want["b2x"] * want["b2y"], want["b1y"] * want["b1y"] + want["b2y"] * want["b2y"]], 1)[m]
    rel = np.abs(q_got - q_want).max(1) / np.maximum(np.abs(q_want).max(1), 1e-6)
    assert np.quantile(rel, 0.999) < 2e-3 and rel.max() < 5e-2, (np.quantile(rel, 0.999), rel.max())
    for k in ("r", "g", "b", "a"):
        assert np.abs(got[k][m] - want[k][m]).max() < 5e-4, k
    assert np.abs(got["ndc_z"][m] - want["ndc_z"][m]).max() < 1e-4


@pytest.mark.parametrize("n,w,h,sh_degree", [(20_000, 320, 200, 0), (200_000, 1000, 600, 1), (150_000, 801, 455, 2)])
def test_frame_matches_reference_blend(gs, oracle_mod, n, w, h, sh_degree):
    from gaussiansplats3d_b200.scenes import synthetic_scene
    raw = synthetic_scene(n, seed=7, kind="bonsai", sh_degree=sh_degree)
    v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=sh_degree)
    v.update()
    got = v.render(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False)
    order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None)
    want, _ = _oracle_frame(oracle_mod, v, order)
    _check_frame(got, want)
    assert got[..., 3].max() > 0.5, "frame is empty"
    # canvas format + image orientation
    got8 = v.render(frame_format=gs._native.GS_FRAME_RGBA8, flip_y=True)
    want8 = np.floor(np.clip(want[::-1], 0, 1) * 255.0 + 0.5)
    assert np.abs(got8.astype(np.int32) - want8.astype(np.int32)).max() <= 9
    assert (np.abs(got8.astype(np.int32) - want8.astype(np.int32)) <= 2).mean() >= FRAC
    t = v.engine.timings()
    assert t["tile_instances"] > 0 and t["visible_splats"] > 0
    v.dispose()


def test_full_hd_bonsai_frame(gs, oracle_mod):
    """BASELINE config 2: 1.2M splats, SH0, 1920x1080, bonsai camera; whole frame vs the oracle."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n = 1_200_000
    raw = synthetic_scene(n, seed=1, kind="bonsai", sh_degree=0)
    v = _viewer(gs, raw, 1920, 1080)
    got = v.frame(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False)
    order = np.empty(n, np.uint32)
    order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None)
    want, _ = _oracle_frame(oracle_mod, v, order)
    err = _check_frame(got, want)
    print(f"1080p bonsai: max err {err.max() * 255:.3f}/255, mean {err.mean() * 255:.5f}/255, timings {v.engine.timings()}")
    v.dispose()


def test_explicit_sorted_indexes_and_worker_topology(gs, oracle_mod):
    """updateRenderIndexes(sortedIndexes) path: order comes from the host (separate sort worker), as in the reference."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    from gaussiansplats3d_b200.viewer import Viewer
    raw = synthetic_scene(50_000, seed=12, kind="uniform")
    v = Viewer(dict(width=400, height=300, sharedMemoryForWorkers=True))
    v.addSplatScene(raw, separate_sort_worker=True)
    v.update()
    assert v.splatMesh.renderIndexes is not None and not v.sortRunning
    got = v.render(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False)
    want, _ = _oracle_frame(oracle_mod, v, v.splatMesh.renderIndexes)
    _check_frame(got, want)
    # a deliberately different (front-to-back) order must give a different picture: order is honoured
    rev = v.splatMesh.renderIndexes[::-1].copy()
    got_rev = v.engine.render(v.uniforms(), 400, 300, raw.count, rev, flip_y=False)
    want_rev, _ = _oracle_frame(oracle_mod, v, rev)
    _check_frame(got_rev, want_rev)
    assert np.abs(got_rev - got).max() > 0.05
    v.dispose()


def test_render_options(gs, oracle_mod):
    """antialiased compensation, point-cloud mode, half covariances, splatScale, fade-in."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    raw = synthetic_scene(40_000, seed=3, kind="bonsai")
    for opts, tweak in ((dict(antialiased=True), None), (dict(halfPrecisionCovariancesOnGPU=True), None), (dict(), "point"), (dict(), "scale"), (dict(), "fade")):
        v = _viewer(gs, raw, 480, 270, **opts)
        if tweak == "point":
            v.splatMesh.pointCloudModeEnabled = True
        if tweak == "scale":
            v.splatMesh.splatScale = 0.6
        if tweak == "fade":
            v.splatMesh.fadeInComplete = False
            v.splatMesh.visibleRegionFadeStartRadius = 2.0
        v.update()
        got = v.render(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False)
        order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), raw.count, raw.count, None)
        want, _ = _oracle_frame(oracle_mod, v, order)
        _check_frame(got, want)
        v.dispose()


def test_dynamic_scenes_and_optional_effects(gs, oracle_mod):
    """SURVEY 8f N3: per-scene transforms in the vertex stage (SplatMaterial.js:136-146, :181-183), scene opacity / visibility
    (SplatMaterial.js:124-133, SplatMaterial3D.js:198-202), 3 scenes, SH1 so the per-scene camera transform matters."""
    from gaussiansplats3d_b200 import three_math as TM
    from gaussiansplats3d_b200.engine import Engine, Uniforms
    from gaussiansplats3d_b200.scenes import pack_scene, synthetic_scene
    n, w, h = 60_000, 512, 300
    raw = synthetic_scene(n, seed=6, kind="uniform", sh_degree=1)
    p = pack_scene(raw)
    rng = np.random.default_rng(3)
    scene_idx = rng.integers(0, 3, n, dtype=np.uint32)
    transforms = np.tile(np.eye(4, dtype=np.float64).T.reshape(16), (32, 1))
    transforms[1] = TM.compose((1.5, 0.0, -1.0), (0.0, np.sin(0.3), 0.0, np.cos(0.3)), (1.2, 1.2, 1.2))
    transforms[2] = TM.compose((-2.0, 0.5, 0.5), (np.sin(0.2), 0.0, 0.0, np.cos(0.2)), (0.7, 0.7, 0.7))
    cam = TM.PerspectiveCamera(50, w / h, 0.1, 1000)
    cam.position = np.array([0.0, 4.0, 12.0]); cam.look_at((0, 0, 0))
    opacity = np.ones(32, np.float32); opacity[1] = 0.6
    vis = np.ones(32, np.int32)
    for effects, hide in ((0, False), (1, False), (1, True)):
        v = vis.copy()
        if hide:
            v[2] = 0
        u = Uniforms(model_view=cam.matrixWorldInverse.astype(np.float32), projection=cam.projectionMatrix.astype(np.float32),
                     camera_position=cam.position.astype(np.float32), focal=(cam.projectionMatrix[0] * 0.5 * w, cam.projectionMatrix[5] * 0.5 * h),
                     viewport=(w, h), sh_degree=1, scene_count=3, scene_transforms=transforms.astype(np.float32), view_matrix=cam.matrixWorldInverse.astype(np.float32),
                     scene_opacity=opacity, scene_visibility=v, enable_optional_effects=effects, dynamic_mode=1)
        order = rng.permutation(n).astype(np.uint32)     # any order: the blend must honour it
        with Engine(n, max_width=w, max_height=h, dynamic_mode=True) as e:
            e.upload_splat_data(p.centers_colors, p.covariances, p.sh, p.sh_degree, scene_indexes=scene_idx)
            got = e.render(u, w, h, n, order, flip_y=False)
            proj = e.read_projected(n)
        want, wproj = oracle_mod.render(u, p.centers_colors, p.covariances, order, w, h, sh=p.sh, sh_degree=p.sh_degree, scene_indexes=scene_idx)
        assert (proj["valid"] != wproj["valid"]).mean() < 1e-4
        m = (proj["valid"] == 1) & (wproj["valid"] == 1)
        assert np.abs(proj["cx"][m] - wproj["cx"][m]).max() < 5e-3 and np.abs(proj["a"][m] - wproj["a"][m]).max() < 5e-4
        _check_frame(got, want)
        if hide:
            assert (wproj["valid"][scene_idx == 2] == 0).all()


def test_precision_20bit_and_float_sort_feed_the_same_frame(gs, oracle_mod):
    """splatSortDistanceMapPrecision 20 (3 radix passes) and the float sort mode drive the renderer like the default."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    raw = synthetic_scene(80_000, seed=13, kind="bonsai")
    for opts in (dict(splatSortDistanceMapPrecision=20), dict(integerBasedSort=False, splatSortDistanceMapPrecision=22)):
        v = _viewer(gs, raw, 480, 270, **opts)
        got = v.frame(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False)
        order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), raw.count, raw.count, None)
        centers = v.splatMesh.getIntegerCenters(0, raw.count - 1, True) if v.integerBasedSort else v.splatMesh.getFloatCenters(0, raw.count - 1, True)
        want_order = oracle_mod.port_sort_indexes(np.arange(raw.count, dtype=np.uint32), centers, None, v.mvp_matrix().astype(np.float32), None, None,
                                                  1 << v.splatSortDistanceMapPrecision, raw.count, raw.count, raw.count, False, v.integerBasedSort, False)
        assert np.array_equal(order, want_order)
        want, _ = _oracle_frame(oracle_mod, v, order)
        _check_frame(got, want)
        v.dispose()


@pytest.mark.parametrize("name", ["bonsai-sh0-160x100", "bonsai-sh2-128x96", "garden-sh1-200x120"])
def test_frame_and_order_match_committed_fixture(gs, name):
    """Against tests/golden/raster_golden.npz (no oracle call at run time): the Viewer-driven sort must reproduce the stored draw
    order bit for bit (that order is the compiled reference sorter's) and the frame must meet the stated tolerance."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
    import raster_cases
    from gaussiansplats3d_b200.scenes import synthetic_scene
    gold = np.load(Path(__file__).resolve().parent / "golden" / "raster_golden.npz")
    n, seed, kind, sh, w, h, cam = raster_cases.CASES[name]
    raw = synthetic_scene(n, seed=seed, kind=kind, sh_degree=sh)
    v = _viewer(gs, raw, w, h, cam=cam, sphericalHarmonicsDegree=sh)
    v.update()
    got = v.render(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False)
    order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None)
    assert np.array_equal(order, gold[name + "|order"])
    _check_frame(got, gold[name + "|frame"])
    v.dispose()


@pytest.mark.parametrize("w,h", [(1000, 600), (2600, 1500)])
def test_blend_and_binning_generations_agree(gs, oracle_mod, monkeypatch, w, h):
    """The round-1 kernels (radix-sorted instances, column blend: GS_BIN=1 GS_BLEND=1) and the current ones (counting-sort binning, block
    blend with exact block masks) must draw the same picture: same instance count, frames equal to rounding.  The larger frame exceeds 256
    coarse tiles of 128x64 px and so runs with 32-px tiles (16 warps per tile) in the current path."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n = 200_000
    raw = synthetic_scene(n, seed=7, kind="bonsai", sh_degree=1)
    frames, inst = {}, {}
    for mode in ("1", "2"):
        monkeypatch.setenv("GS_BIN", mode)
        monkeypatch.setenv("GS_BLEND", mode)
        v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=1)
        v.update()
        frames[mode] = v.render(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False).copy()
        inst[mode] = v.engine.timings()["tile_instances"]
        if mode == "2":
            order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None)
            want, _ = _oracle_frame(oracle_mod, v, order)
            _check_frame(frames[mode], want)
        v.dispose()
    assert inst["1"] == inst["2"]      # both generations bin exactly as oracle/bin_oracle.py restates (tests/test_binning_gpu.py)
    d = np.abs(frames["1"] - frames["2"])
    # the two blends round differently (forward differences over 4-px columns vs direct evaluation, opacity inside the exponent)
    assert d.max() <= 4.0 / 255 and (d <= 1.0 / 255).mean() >= 0.9995, (d.max() * 255, (d <= 1.0 / 255).mean())


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1280, 720), (3840, 2160)])
def test_blend_list_prefetch_variants_are_bit_identical(gs, monkeypatch, w, h):
    """GS_BLEND_TMA=1 fetches the coarse-tile list batches with bulk asynchronous copies (cp.async.bulk + mbarrier, double buffered)
    instead of plain loads: same batches, same arithmetic, so the frame must be bit-identical (a protocol error paints magenta).
    GS_BLEND_ROUNDS=2 halves the batch; that shifts which records share a loop iteration, and a warp stops at the first ITERATION after
    which all of its pixels are below the 1/512 transmittance cutoff, so it may composite one more (invisible) record: <= 1/255.
    16-px tiles (720p) and 32-px tiles (4K)."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n = 150_000
    raw = synthetic_scene(n, seed=11, kind="bonsai", sh_degree=0)
    frames = {}
    for name, env in (("plain", {}), ("tma", {"GS_BLEND_TMA": "1"}), ("rounds2", {"GS_BLEND_ROUNDS": "2"}), ("tma_rounds2", {"GS_BLEND_TMA": "1", "GS_BLEND_ROUNDS": "2"})):
        for k in ("GS_BLEND_TMA", "GS_BLEND_ROUNDS"):
            monkeypatch.delenv(k, raising=False)
        for k, val in env.items():
            monkeypatch.setenv(k, val)
        v = _viewer(gs, raw, w, h)
        v.update()
        frames[name] = v.render(frame_format=gs._native.GS_FRAME_RGBA8, flip_y=True).copy()
        v.dispose()
    assert frames["plain"][..., 3].max() > 0
    assert np.array_equal(frames["tma"], frames["plain"])
    assert np.array_equal(frames["tma_rounds2"], frames["rounds2"])
    d = np.abs(frames["rounds2"].astype(np.int16) - frames["plain"].astype(np.int16))
    assert d.max() <= 1 and (d != 0).mean() < 1e-3, (d.max(), (d != 0).mean())


def test_dynamic_scene_applies_its_transform(gs, oracle_mod):
    """Viewer(dynamicScene=True).addSplatScene(position, rotation, scale): the transform is NOT baked; the sorter (sorter.cpp:44-50) and the
    vertex stage (SplatMaterial.js:136-146) apply it every frame.  The picture must match (a) the restatement driven with the same
    dynamic uniforms and order, and (b) the static viewer that bakes the same transform at load, up to the sort's tie-breaking."""
    from gaussiansplats3d_b200 import three_math as TM
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, w, h = 60_000, 480, 270
    raw = synthetic_scene(n, seed=21, kind="bonsai", sh_degree=0)
    q = np.array([0.1, 0.35, -0.2, 0.9]); q /= np.linalg.norm(q)
    kw = dict(position=(0.6, -0.4, 0.8), rotation=tuple(q), scale=(1.4, 1.4, 1.4))
    frames = {}
    for dynamic in (False, True):
        v = _viewer(gs, raw, w, h, dynamicScene=dynamic) if False else None
        from gaussiansplats3d_b200.viewer import Viewer
        from gaussiansplats3d_b200.scenes import CAMERAS
        c = CAMERAS["bonsai"]
        v = Viewer(dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=w, height=h, dynamicScene=dynamic))
        v.addSplatScene(raw, **kw)
        frames[dynamic] = v.frame(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False).copy()
        if dynamic:
            u = v.uniforms()
            assert u.dynamic_mode == 1 and not np.allclose(u.scene_transforms[0], TM.identity())
            tr = v.splatMesh.fillTransformsArray()
            order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None, transforms=tr)
            centers = v.splatMesh.getIntegerCenters(0, n - 1, True)
            want_order = oracle_mod.port_sort_indexes(np.arange(n, dtype=np.uint32), centers, None, v.mvp_matrix().astype(np.float32), np.zeros(n, np.uint32), tr,
                                                      1 << 16, n, n, n, False, True, True)
            assert np.array_equal(order, want_order)
            p = v.splatMesh.packed
            want, _ = oracle_mod.render(u, p.centers_colors, p.covariances, order, w, h, scene_indexes=None)
            _check_frame(frames[True], want)
        v.dispose()
    assert frames[True][..., 3].max() > 0.5
    d = np.abs(frames[True] - frames[False])
    assert (d <= 2.0 / 255).mean() >= 0.995, (d <= 2.0 / 255).mean()          # same picture; ties in the two sorts may resolve differently


def test_pipelined_frames_equal_blocking_frames(gs):
    """gs_frame_begin / gs_frame_end (two or three frames in flight, alternating device frame buffers, copies on a second stream) must deliver
    exactly the pictures gs_frame delivers, in order, for a moving camera."""
    from gaussiansplats3d_b200 import _native as N
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, w, h = 150_000, 640, 360
    raw = synthetic_scene(n, seed=8, kind="bonsai", sh_degree=1)
    v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=1)
    e = v.engine
    cams = []
    for k in range(6):
        v.camera.position = np.asarray(v.initialCameraPosition) + np.array([0.15 * k, -0.05 * k, 0.1 * k])
        v.camera.look_at(v.initialCameraLookAt)
        v.camera.update(); v.updateSplatMesh()
        cams.append(e.prepare_frame(v.mvp_matrix().astype(np.float32), v.uniforms(), w, h, n, frame_format=N.GS_FRAME_RGBA8, flip_y=True))
    want = []
    for prep in cams:
        out = N.pinned_empty((h, w, 4), np.uint8)
        e.frame_prepared(prep, out)
        want.append(out.copy())
    bufs = [N.pinned_empty((h, w, 4), np.uint8) for _ in range(2)]
    got = []
    e.frame_begin(cams[0], bufs[0])
    for i in range(len(cams)):
        if i + 1 < len(cams):
            e.frame_begin(cams[i + 1], bufs[(i + 1) & 1])
        e.frame_end()
        got.append(bufs[i & 1].copy())
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), f"pipelined frame {i} differs"
    assert not np.array_equal(want[0], want[-1])
    with pytest.raises(RuntimeError):
        e.frame_end()                                   # nothing in flight any more
    # three frames in flight over the two device buffers (begin(i+2) before end(i)); each needs its own host buffer; statistics of the
    # frame that ended come from the blend kernel's status snapshot
    bufs = [N.pinned_empty((h, w, 4), np.uint8) for _ in range(3)]
    got = []
    e.frame_begin(cams[0], bufs[0])
    e.frame_begin(cams[1], bufs[1])
    for i in range(len(cams)):
        if i + 2 < len(cams):
            e.frame_begin(cams[i + 2], bufs[(i + 2) % 3])
        e.frame_end()
        assert e.timings()["visible_splats"] > 0 and e.timings()["tile_instances"] > 0
        got.append(bufs[i % 3].copy())
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), f"3-deep pipelined frame {i} differs"
    e.frame_begin(cams[0], bufs[0]); e.frame_begin(cams[1], bufs[1]); e.frame_begin(cams[2], bufs[2])
    with pytest.raises(RuntimeError):
        e.frame_begin(cams[3], bufs[0])                 # a fourth frame in flight is refused
    with pytest.raises(RuntimeError):
        e.frame_async(None, None, w, h, n, prepared=cams[3])   # so is anything else that would overwrite a frame buffer being copied out
    for _ in range(3):
        e.frame_end()
    v.dispose()
