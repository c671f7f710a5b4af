"""GPU parity of the TwoD (2D Gaussian surfel) render mode: k_project2d + the shared sort / binning + k_blend2d against the CPU
restatement of SplatMaterial2D (oracle/surfel_oracle.c).

Tolerances.  Projection: the kernel evaluates the vertex stage in the shader's own f32 operation order, unfused (the fallback
square's pointImage^2 - temp cancels ~1e6 px^2 down to ~1 px^2), so T is compared at 1e-4 of its largest element per splat, quad centre within 2e-3 px, half-edges within 1e-3 relative, colour 5e-4, quad branch equal on >= 99.99 % of the splats both
draw.  Frames: the 3D tolerances, max abs err <= 2/255 on >= 99.9 % of channels and <= 8/255 everywhere on float accumulators
(observed on a B200: at most 1.45/255 on every frame and crop below).  The kernel evaluates p = k x l in the equivalent linear form
relative to the quad centre and exp with ex2.approx; a pixel centre within rounding of a quad edge may fall on either side."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL_MOST, TOL_WORST, FRAC = 2.0 / 255.0, 8.0 / 255.0, 0.999


def _viewer(gs, raw, width, height, cam="bonsai", position=None, **opts):
    from gaussiansplats3d_b200.scenes import CAMERAS
    from gaussiansplats3d_b200.viewer import SplatRenderMode, Viewer
    c = CAMERAS[cam]
    v = Viewer(dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=width, height=height,
                    splatRenderMode=SplatRenderMode.TwoD, **opts))
    v.addSplatScene(raw, **({} if position is None else position))
    return v


def _oracle(v, order, crop=None):
    import oracle.surfel as S
    p = v.splatMesh.packed
    ps = S.project_2d(v.uniforms(), p.centers_colors, p.scale_rotations, p.sh, p.sh_degree)
    if crop is None:
        return S.blend_2d(ps, order, v.renderWidth, v.renderHeight)
    return S.blend_2d_crop(ps, order, v.renderWidth, v.renderHeight, *crop)


def _check_frame(got, want):
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    frac = (err <= TOL_MOST).mean()
    assert err.max() <= TOL_WORST, f"worst channel error {err.max() * 255:.2f}/255 at {np.unravel_index(err.argmax(), err.shape)}"
    assert frac >= FRAC, f"only {frac * 100:.3f}% of channels within 2/255"
    return err


def _frame(gs, v, fmt=None, flip_y=False):
    v.camera.update(); v.updateSplatMesh()
    return v.frame(frame_format=gs._native.GS_FRAME_RGBA32F if fmt is None else fmt, flip_y=flip_y).copy()


def _order(v):
    n = v.splatMesh.getSplatCount()
    order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None)
    return order


@pytest.mark.parametrize("sh_degree,fmt", [(0, "f16"), (1, "f16"), (2, "f16"), (2, "u8"), (2, "f32")])
def test_projection_matches_vertex_shader(gs, sh_degree, fmt):
    import oracle.surfel as S
    from gaussiansplats3d_b200.scenes import pack_scene, synthetic_scene
    raw = synthetic_scene(60_000, seed=4, kind="bonsai", sh_degree=sh_degree)
    raw.scales[: 20_000] *= 4.0           # a third of the surfels large enough for the eigen-aligned quad
    v = _viewer(gs, raw, 640, 360, sphericalHarmonicsDegree=sh_degree)
    if fmt != "f16" and sh_degree:
        v.splatMesh.packed = pack_scene(raw, sh_format=fmt, render_mode=1)
        v.splatMesh.setRenderer(v.engine)
    _frame(gs, v)
    got = v.engine.read_projected_2d(raw.count)
    p = v.splatMesh.packed
    want = S.project_2d(v.uniforms(), p.centers_colors, p.scale_rotations, p.sh, p.sh_degree)
    assert (got["valid"] != want["valid"]).mean() < 1e-4
    # missingW = sqrt(1 - x^2 - y^2 - z^2) is NaN where rounding makes the argument negative (undefined in GLSL): both give NaN T
    finite = np.isfinite(want["T"]).all(1)
    assert np.array_equal(finite, np.isfinite(got["T"]).all(1))
    m = (got["valid"] == 1) & (want["valid"] == 1) & finite
    assert m.sum() > 1000
    assert (got["branch"][m] == want["branch"][m]).mean() >= 0.9999
    assert 0.05 < (want["branch"][m] == 0).mean() < 0.95, "both quad branches must be exercised"
    tscale = np.abs(want["T"][m]).max(1, keepdims=True)
    assert (np.abs(got["T"][m] - want["T"][m]) / tscale).max() < 1e-4
    for k in ("cx", "cy"):
        assert np.abs(got[k][m] - want[k][m]).max() < 2e-3, k
    b = m & (got["branch"] == want["branch"])
    hscale = np.maximum(np.hypot(want["h1x"][b], want["h1y"][b]), np.hypot(want["h2x"][b], want["h2y"][b]))
    for k in ("h1x", "h1y", "h2x", "h2y"):
        assert np.quantile(np.abs(got[k][b] - want[k][b]) / hscale, 0.999) < 1e-3, k
    e = b & (want["branch"] == 0)
    assert np.abs(got["qcx"][e] - want["qcx"][e]).max() < 1e-5          # NDC units in the eigen branch
    for k in ("r", "g", "b", "a"):
        assert np.abs(got[k][m] - want[k][m]).max() < 5e-4, k
    v.dispose()


@pytest.mark.parametrize("n,w,h,sh_degree", [(20_000, 320, 200, 0), (200_000, 1000, 600, 1), (150_000, 801, 455, 2)])
def test_frame_matches_reference_blend(gs, n, w, h, sh_degree):
    from gaussiansplats3d_b200.scenes import synthetic_scene
    raw = synthetic_scene(n, seed=11, kind="bonsai", sh_degree=sh_degree)
    raw.scales[: n // 3] *= 4.0
    v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=sh_degree)
    got = _frame(gs, v)
    want = _oracle(v, _order(v))
    _check_frame(got, want)
    assert got[..., 3].max() > 0.5 and (got[..., 3] > 0.01).mean() > 0.05
    v.dispose()


def test_quad_centre_filter_near_window_origin(gs):
    """Eigen-branch vQuadCenter is in NDC units (SplatMaterial2D.js:232) while vFragCoord is in pixels, so rho2d is small only within
    a few pixels of the window origin: a large surfel covering the origin must show the rho2d term there, as in the restatement."""
    from gaussiansplats3d_b200.scenes import RawScene
    raw = RawScene(np.array([[0.0, 0.0, 0.0]], np.float32), np.array([[3.0, 3.0, 1.0]], np.float32), np.array([[0.0, 0.0, 0.0, 1.0]], np.float32),
                   np.array([[200, 120, 40, 255]], np.uint8), None, 0)
    v = _viewer(gs, raw, 160, 120, cam="default", position=None)
    got = _frame(gs, v)
    want = _oracle(v, np.zeros(1, np.uint32))
    _check_frame(got, want)
    assert want[0, 0, 3] < 0.98 * want[60, 80, 3], "the restatement must show the rho2d filter at the window origin"
    v.dispose()


def test_full_hd_and_4k_crops(gs):
    """1.2 M surfels at 1920x1080 (16-px tiles) and 3840x2160 (32-px tiles), checked on crops of the full-size frames."""
    from gaussiansplats3d_b200.scenes import synthetic_scene
    raw = synthetic_scene(1_200_000, seed=3, kind="bonsai", sh_degree=0)
    for w, h in ((1920, 1080), (3840, 2160)):
        v = _viewer(gs, raw, w, h)
        got = _frame(gs, v)
        order = _order(v)
        for x0, y0 in ((w // 2 - 128, h // 2 - 128), (w // 4, h // 3)):
            want = _oracle(v, order, (x0, y0, 256, 256))
            _check_frame(got[y0:y0 + 256, x0:x0 + 256], want)
        v.dispose()


def test_rgba8_flip_and_explicit_sorted_indexes(gs):
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, w, h = 80_000, 480, 270
    raw = synthetic_scene(n, seed=5, kind="bonsai", sh_degree=1)
    raw.scales[: n // 4] *= 4.0
    v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=1)
    f8 = _frame(gs, v, fmt=gs._native.GS_FRAME_RGBA8, flip_y=True)
    order = _order(v)
    want = _oracle(v, order)
    want8 = np.floor(np.clip(want, 0, 1) * 255.0 + 0.5)[::-1]
    _check_frame(f8 / 255.0, want8 / 255.0)
    # an explicit draw order (here: a shuffled one) replaces the engine's sort
    rng = np.random.default_rng(2)
    perm = rng.permutation(n).astype(np.uint32)
    got = v.engine.render(v.uniforms(), w, h, n, sorted_indexes=perm)
    _check_frame(got, _oracle(v, perm))
    v.dispose()


def test_dynamic_transform_and_fade_in(gs):
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, w, h = 60_000, 480, 270
    raw = synthetic_scene(n, seed=21, kind="bonsai", sh_degree=0)
    raw.scales[: n // 3] *= 4.0
    q = np.array([0.1, 0.35, -0.2, 0.9]); q /= np.linalg.norm(q)
    kw = dict(position=(0.6, -0.4, 0.8), rotation=tuple(q), scale=(1.4, 1.4, 1.4))
    frames = {}
    for dynamic in (False, True):
        v = _viewer(gs, raw, w, h, position=kw, dynamicScene=dynamic)
        frames[dynamic] = _frame(gs, v)
        tr = v.splatMesh.fillTransformsArray() if dynamic else None
        order, _ = v.engine.sort(v.mvp_matrix().astype(np.float32), n, n, None, transforms=tr)
        _check_frame(frames[dynamic], _oracle(v, order))
        v.dispose()
    assert frames[True][..., 3].max() > 0.5
    d = np.abs(frames[True] - frames[False])
    assert (d <= 2.0 / 255).mean() >= 0.99, (d <= 2.0 / 255).mean()   # baked (decomposed) and per-frame transforms draw the same scene
    # fade-in (SplatMaterial.js:347-363)
    v = _viewer(gs, raw, w, h)
    v.splatMesh.fadeInComplete = False
    v.splatMesh.visibleRegionFadeStartRadius = 1.0
    got = _frame(gs, v)
    u = v.uniforms()
    assert u.fade_in_complete == 0
    _check_frame(got, _oracle(v, _order(v)))
    v.dispose()


def test_pipelined_frames_equal_blocking_frames(gs):
    from gaussiansplats3d_b200 import _native as N
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, w, h = 150_000, 640, 360
    raw = synthetic_scene(n, seed=8, kind="bonsai", sh_degree=1)
    raw.scales[: n // 3] *= 4.0
    v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=1)
    e = v.engine
    cams = []
    for k in range(5):
        v.camera.position = np.asarray(v.initialCameraPosition) + np.array([0.15 * k, -0.05 * k, 0.1 * k])
        v.camera.look_at(v.initialCameraLookAt)
        v.camera.update(); v.updateSplatMesh()
        cams.append(e.prepare_frame(v.mvp_matrix().astype(np.float32), v.uniforms(), w, h, n, frame_format=N.GS_FRAME_RGBA8, flip_y=True))
    want = []
    for prep in cams:
        out = N.pinned_empty((h, w, 4), np.uint8)
        e.frame_prepared(prep, out)
        want.append(out.copy())
    bufs = [N.pinned_empty((h, w, 4), np.uint8) for _ in range(3)]
    got = []
    e.frame_begin(cams[0], bufs[0])
    e.frame_begin(cams[1], bufs[1])
    for i in range(len(cams)):
        if i + 2 < len(cams):
            e.frame_begin(cams[i + 2], bufs[(i + 2) % 3])
        e.frame_end()
        got.append(bufs[i % 3].copy())
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), f"pipelined frame {i} differs"
    assert not np.array_equal(want[0], want[-1])
    v.dispose()


def test_3d_and_2d_engines_alternate(gs):
    """Captured frame graphs are keyed by the render mode: engines of both modes alternating in one process each keep their picture."""
    from gaussiansplats3d_b200.scenes import CAMERAS, synthetic_scene
    from gaussiansplats3d_b200.viewer import Viewer
    raw = synthetic_scene(50_000, seed=9, kind="bonsai", sh_degree=0)
    raw.scales[:10_000] *= 4.0
    c = CAMERAS["bonsai"]
    opts = dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=400, height=240)
    v3, v2 = Viewer(opts), Viewer(dict(opts, splatRenderMode=1))
    v3.addSplatScene(raw); v2.addSplatScene(raw)
    first = {}
    for it in range(3):
        for name, v in (("3d", v3), ("2d", v2)):
            f = _frame(gs, v, fmt=gs._native.GS_FRAME_RGBA8)
            if it == 0:
                first[name] = f
            else:
                assert np.array_equal(f, first[name]), f"{name} frame changed after the other mode rendered"
    assert not np.array_equal(first["3d"], first["2d"])
    v3.dispose(); v2.dispose()


def test_errors(gs):
    from gaussiansplats3d_b200 import Engine, GsError
    from gaussiansplats3d_b200.scenes import pack_scene, synthetic_scene
    raw = synthetic_scene(1000, seed=1)
    p = pack_scene(raw, render_mode=1)
    assert p.covariances is None and p.scale_rotations.shape == (1000, 6)
    e = Engine(1000, max_width=64, max_height=64, splat_render_mode=1)
    with pytest.raises(GsError) as ei:
        e.upload_splat_data(p.centers_colors, pack_scene(raw).covariances)
    assert ei.value.code == 1 and "scale_rotations" in str(ei.value)
    e.upload_splat_data(p.centers_colors, None, scale_rotations=p.scale_rotations)
    back = e.read_buffer(gs._native.GS_BUF_SCALE_ROTATIONS, np.float32, 6000)
    assert np.array_equal(back.reshape(-1, 6), p.scale_rotations)
    with pytest.raises(GsError) as ei:
        e.read_projected(10)              # a TwoD engine has no 3D records: refused before anything is launched
    assert ei.value.code == 1 and "read_projected_2d" in str(ei.value)
    with pytest.raises(GsError):
        e.read_buffer(gs._native.GS_BUF_COVARIANCES, np.float32, 6)   # nor covariances
    e.close()
    e3 = Engine(1000, max_width=64, max_height=64)
    with pytest.raises(GsError):
        e3.read_projected_2d(10)          # a ThreeD engine has no surfel projection
    with pytest.raises(GsError):
        e3.read_buffer(gs._native.GS_BUF_SCALE_ROTATIONS, np.float32, 6)
    e3.close()
    with pytest.raises(GsError):
        Engine(10, max_width=8, max_height=8, splat_render_mode=2)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_frames_sum_to_single_engine_frame(gs, world):
    from gaussiansplats3d_b200.parallel import combine_frames, ownership_map
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, w, h = 120_000, 801, 455
    raw = synthetic_scene(n, seed=8, kind="bonsai", sh_degree=1)
    raw.scales[: n // 3] *= 4.0
    v1 = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=1)
    want = _frame(gs, v1, fmt=gs._native.GS_FRAME_RGBA8)
    v1.dispose()
    own = ownership_map(w, h, world)
    frames = []
    for r in range(world):
        v = _viewer(gs, raw, w, h, sphericalHarmonicsDegree=1, rank=r, world_size=world)
        f = _frame(gs, v, fmt=gs._native.GS_FRAME_RGBA8)
        assert not f[own != r].any(), "a rank wrote pixels outside its own coarse tiles"
        frames.append(f)
        v.dispose()
    assert np.array_equal(combine_frames(frames), want), "sharded TwoD frames do not sum to the single-GPU frame bit for bit"


def _peer_worker_2d(rank, world, port, q):
    """One process per GPU, TwoD engines: rank 0 exports its frame through CUDA IPC, the other rank's k_blend2d stores its tiles into it."""
    import os
    import sys
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import gaussiansplats3d_b200 as gs
    from gaussiansplats3d_b200 import _native as N
    from gaussiansplats3d_b200.parallel import PeerGather
    from gaussiansplats3d_b200.scenes import CAMERAS, synthetic_scene
    from gaussiansplats3d_b200.viewer import Viewer
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    n, w, h = 100_000, 801, 455
    raw = synthetic_scene(n, seed=8, kind="bonsai", sh_degree=0)
    raw.scales[: n // 3] *= 4.0
    c = CAMERAS["bonsai"]
    opts = dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=w, height=h, device=rank,
                splatRenderMode=1)
    v = Viewer(dict(opts, rank=rank, world_size=world))
    v.addSplatScene(raw)
    e = v.engine
    cams = []
    for k in range(5):
        v.camera.position = np.asarray(v.initialCameraPosition) + np.array([0.12 * k, -0.04 * k, 0.08 * k])
        v.camera.look_at(v.initialCameraLookAt)
        v.camera.update(); v.updateSplatMesh()
        cams.append(e.prepare_frame(v.mvp_matrix().astype(np.float32), v.uniforms(), w, h, n, frame_format=N.GS_FRAME_RGBA8, flip_y=True))
    wants = []
    if rank == 0:
        v1 = Viewer(opts)
        v1.addSplatScene(raw)
        for prep in cams:
            out = N.pinned_empty((h, w, 4), np.uint8)
            v1.engine.frame_prepared(prep, out)
            wants.append(out.copy())
        v1.dispose()
    PeerGather(e, rank, world)
    ok = True
    for prep_i, prep in enumerate(cams):   # blocking frames (graph replay across frames)
        out = N.pinned_empty((h, w, 4), np.uint8) if rank == 0 else None
        e.frame_prepared(prep, out)
        if rank == 0:
            ok = ok and bool(np.array_equal(out, wants[prep_i]))
    dist.barrier()
    if rank == 0:                          # pipelined frames: the peer stores frame f+1 into the other half of rank 0's allocation
        bufs = [N.pinned_empty((h, w, 4), np.uint8) for _ in range(3)]
        e.frame_begin(cams[0], bufs[0]); e.frame_begin(cams[1], bufs[1])
        for i in range(len(cams)):
            if i + 2 < len(cams):
                e.frame_begin(cams[i + 2], bufs[(i + 2) % 3])
            e.frame_end()
            ok = ok and bool(np.array_equal(bufs[i % 3], wants[i]))
    else:
        for prep in cams:
            e.frame_async(None, None, w, h, n, prepared=prep)
        e.synchronize()
    dist.barrier()
    q.put((rank, ok))
    v.dispose()
    dist.destroy_process_group()


def test_fused_peer_gather_two_gpus_2d(gs):
    """Needs 2 GPUs (skipped on a 1-GPU box): rank 0's TwoD picture assembled by the fused peer gather equals the single-GPU TwoD frame."""
    if gs._native.load().gs_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from test_multi_gpu import _free_port
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_peer_worker_2d, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]
