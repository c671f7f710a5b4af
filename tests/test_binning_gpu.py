"""GPU: tile binning read back from the engine (GS_BUF_TILE_*) and compared bit for bit with the restatement in oracle/bin_oracle.py,
on every binning path: the counting sort (<= 256 coarse tiles, 16- and 32-px fine tiles, with and without the warp compaction, both
k_bin_place configurations), the older emit + radix path (two-pass 9- and 10-bit tile sorts), sharded ranks with and without the subset
sort, and both render modes.  Binning is integer work, so the check is equality.  Also: the device rects contain every pixel the
splat's quad covers, frames on the larger-frame paths against the blend oracles, tile-instance overflow, and the sharded diagonal limit."""
import re

import numpy as np
import pytest

from oracle import bin_oracle as B

pytestmark = pytest.mark.gpu

SIZES = [(320, 200), (801, 455), (1920, 1080), (1921, 1080), (3840, 2160), (4096, 2160), (7680, 4320),
         (4096, 256), (4112, 256), (8192, 256), (256, 8192), (24576, 64)]
TOL_MOST, TOL_WORST, FRAC = 2.0 / 255.0, 8.0 / 255.0, 0.999
ADV_CAMERA = dict(cameraUp=(0.0, 1.0, 0.0), initialCameraPosition=(0.0, 0.0, 10.0), initialCameraLookAt=(0.0, 0.0, 0.0))


# ---- scenes ---------------------------------------------------------------------------------------------------------------------
def _adversarial_scene(v, w, h, seed=3):
    """Splats on the plane z = 0, seen face-on from z = 10, placed in pixels: centres on fine- and coarse-tile corners and on the frame
    edges with extents that end near tile boundaries, splats over many coarse tiles (up to the whole screen), culled splats (behind the
    camera, far off screen) and exact duplicates."""
    from gaussiansplats3d_b200.scenes import RawScene
    rng = np.random.default_rng(seed)
    P = np.asarray(v.camera.projectionMatrix, np.float64).reshape(16)
    f = P[0] * 0.5 * w                                   # focal length in px; the camera sits 10 units from the plane

    def world(px, py):                                   # GL window pixel coordinates -> point on z = 0
        return (2.0 * px / w - 1.0) * 10.0 / P[0], (2.0 * py / h - 1.0) * 10.0 / P[5]

    def scale_for(extent_px):                            # quad half-extent ~ sqrt(8) * sigma_px
        return np.maximum(extent_px, 0.05) * 10.0 / (2.8284271 * f)

    t = B.geometry(w, h).tile_px
    k = 12_000
    step = np.where(rng.uniform(size=k) < 0.5, t, 8 * t)
    px = rng.integers(0, w // t + 2, k) * t
    py = rng.integers(0, h // t + 2, k) * t
    px = np.where(step > t, (px // (8 * t)) * 8 * t, px) + rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0], k)
    py = np.where(step > t, (py // (4 * t)) * 4 * t, py) + rng.choice([-1.0, -0.5, 0.0, 0.5, 1.0], k)
    edge = rng.uniform(size=k) < 0.15                    # on the frame's last row / column
    px[edge] = w - rng.choice([0.0, 0.5, 1.0, t / 2], edge.sum())
    py[edge[::-1]] = h - rng.choice([0.0, 0.5, 1.0, t / 2], edge[::-1].sum())
    ext = t * rng.integers(0, 6, k) + rng.choice([0.2, 0.5, 1.0, 2.0, -0.5], k)
    kb = 400                                             # many coarse tiles: > 32 coarse tiles walks the whole warp
    bx, by = rng.uniform(0, w, kb), rng.uniform(0, h, kb)
    bext = rng.uniform(300, 3000, kb)
    bx[:20], by[:20], bext[:20] = w / 2, h / 2, 5000.0   # as large as the size cap allows: the whole screen of smaller frames
    xs, ys = world(np.concatenate([px, bx]), np.concatenate([py, by]))
    centers = np.stack([xs, ys, np.zeros_like(xs)], 1)
    s = scale_for(np.concatenate([ext, bext]))
    scales = np.stack([s, s * rng.uniform(0.3, 1.0, s.size), s * rng.uniform(0.3, 1.0, s.size)], 1)
    kc = 600                                             # culled: behind the camera, far off screen
    cx, cy = world(rng.uniform(0, w, kc), rng.uniform(0, h, kc))
    behind = np.stack([cx, cy, np.full(kc, 15.0)], 1)
    ox, oy = world(rng.choice([-8.0, 9.0], kc) * w, rng.uniform(0, h, kc))
    off = np.stack([ox, oy, np.zeros(kc)], 1)
    centers = np.concatenate([centers, behind, off])
    scales = np.concatenate([scales, np.full((2 * kc, 3), scale_for(np.array([8.0]))[0])])
    q = rng.normal(size=(centers.shape[0], 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[q[:, 3] < 0] *= -1
    colors = np.empty((centers.shape[0], 4), np.uint8)
    colors[:, :3] = rng.integers(0, 256, (centers.shape[0], 3))
    colors[:, 3] = rng.integers(160, 256, centers.shape[0])
    dup = rng.integers(0, k, 800)                        # exact duplicates
    cat = lambda a: np.concatenate([a, a[dup]])          # noqa: E731
    return RawScene(cat(centers).astype(np.float32), cat(scales).astype(np.float32), cat(q).astype(np.float32), cat(colors), None, 0)


def _viewer(scene, w, h, mode=0, n=60_000, seed=7, scale=1.0, **opts):
    from gaussiansplats3d_b200.scenes import CAMERAS, synthetic_scene
    from gaussiansplats3d_b200.viewer import Viewer
    if scene == "adversarial":
        cam = ADV_CAMERA
    else:
        c = CAMERAS["bonsai" if scene == "bonsai" else "default"]
        cam = dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"])
    v = Viewer(dict(cam, width=w, height=h, splatRenderMode=mode, **opts))
    if scene == "adversarial":
        raw = _adversarial_scene(v, w, h)
    else:
        raw = synthetic_scene(n, seed=seed, kind=scene, sh_degree=0)
        raw.scales *= np.float32(scale)
        if mode == 1:
            raw.scales[: n // 3] *= 4.0                  # surfels large enough for the eigen-aligned quad
    v.addSplatScene(raw)
    v.camera.update(); v.updateSplatMesh()
    return v


# ---- read-back and comparison ---------------------------------------------------------------------------------------------------
def _state(e, n_splats):
    from gaussiansplats3d_b200 import _native as N
    cap, ncoarse, tile_px, path = (int(x) for x in e.read_buffer(N.GS_BUF_TILE_INFO, np.uint64, 4))
    t = e.timings()
    total = int(t["tile_instances"])
    stored = min(total, cap)
    return dict(cap=cap, ncoarse=ncoarse, tile_px=tile_px, path=path, total=total, visible=int(t["visible_splats"]),
                rects=e.read_buffer(N.GS_BUF_TILE_RECTS, np.uint16, 4 * n_splats).reshape(-1, 4),
                ranges=e.read_buffer(N.GS_BUF_TILE_RANGES, np.uint32, 2 * ncoarse).reshape(-1, 2),
                tile_order=e.read_buffer(N.GS_BUF_TILE_ORDER, np.uint32, ncoarse),
                list=e.read_buffer(N.GS_BUF_TILE_LIST, np.uint64, stored) if stored else np.zeros(0, np.uint64))


def _device_order(e, count):
    from gaussiansplats3d_b200 import _native as N
    return e.read_buffer(N.GS_BUF_SORTED_INDEXES, np.uint32, count)


def _nonempty(rects):
    r = rects.astype(np.int64)
    return (r[:, 2] >= r[:, 0]) & (r[:, 3] >= r[:, 1])


def _check_binning(e, n_splats, w, h, order, rank=0, world=1, bin_version=2):
    """The engine's binning of its last frame equals the restatement of the lists for `order` (its last element drawn first)."""
    s = _state(e, n_splats)
    want = B.bin_frame(s["rects"], order, w, h, rank, world)
    path = B.binning_path(w, h, bin_version)
    assert (s["ncoarse"], s["tile_px"], s["path"]) == (want.geometry.ncoarse, want.geometry.tile_px, path)
    assert s["visible"] == int(_nonempty(s["rects"]).sum())
    assert s["total"] == want.total, (s["total"], want.total)
    assert s["total"] <= s["cap"]
    assert np.array_equal(s["ranges"], want.ranges(path)), "tile ranges differ"
    if not np.array_equal(s["list"], want.entries):
        bad = int(np.nonzero(s["list"] != want.entries)[0][0])
        tile = int(want.tiles[bad])
        raise AssertionError(f"list entry {bad} (coarse tile {tile}) is {int(s['list'][bad]):#x}, the restatement has {int(want.entries[bad]):#x}")
    assert np.array_equal(s["tile_order"], want.tile_order(path)), "blend schedule differs"
    return s, want


def _env(monkeypatch, **env):
    for k in ("GS_BIN", "GS_BINCFG", "GS_BIN_COMPACT", "GS_BLEND", "GS_BLEND_TMA", "GS_SUBSET_MIN", "GS_INSTANCE_FACTOR"):
        monkeypatch.delenv(k, raising=False)
    for k, val in env.items():
        monkeypatch.setenv(k, str(val))


# ---- exact binning --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
@pytest.mark.parametrize("scene", ["bonsai", "uniform", "adversarial"])
@pytest.mark.parametrize("w,h", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_binning_matches_restatement(gs, monkeypatch, w, h, scene, mode):
    _env(monkeypatch, GS_INSTANCE_FACTOR=64)      # the adversarial scene's large splats need more than 4 instances per splat on a strip
    v = _viewer(scene, w, h, mode)
    e, n = v.engine, v.splatMesh.getSplatCount()
    v.frame(frame_format=gs._native.GS_FRAME_RGBA8)
    s, want = _check_binning(e, n, w, h, _device_order(e, n))
    assert want.total > 0
    g = want.geometry
    r = s["rects"][_nonempty(s["rects"])].astype(np.int64)
    if scene == "adversarial":      # the scene does reach what it is meant to reach
        assert (r[:, 2] == g.tiles_x - 1).any() and (r[:, 3] == g.tiles_y - 1).any()
        assert ((r[:, 2] % 8 == 7) & (r[:, 2] < g.tiles_x - 1)).sum() > 20 and ((r[:, 0] % 8 == 0) & (r[:, 0] > 0)).sum() > 20
        if g.ncoarse > 32 and g.coarse_y >= 3:      # (the size cap keeps a splat within 2048 px: 16 coarse tiles of a single row)
            assert ((r[:, 2] // 8 - r[:, 0] // 8 + 1) * (r[:, 3] // 4 - r[:, 1] // 4 + 1) > 32).sum() > 0
        assert (~_nonempty(s["rects"])).sum() >= 1200
    v.dispose()


@pytest.mark.parametrize("w,h", [(801, 455), (4096, 2160)])
def test_binning_render_counts(gs, monkeypatch, w, h):
    """render_count at and around the 2048-rank chunk of the counting sort, and below the number of uploaded splats; explicit orders."""
    _env(monkeypatch)
    v = _viewer("adversarial", w, h)
    e, n = v.engine, v.splatMesh.getSplatCount()
    perm = np.random.default_rng(5).permutation(n).astype(np.uint32)
    for rc in (1, 2047, 2048, 2049, 4097, n - 1000):
        order = perm[:rc].copy()
        e.render(v.uniforms(), w, h, rc, order, frame_format=gs._native.GS_FRAME_RGBA8)
        assert np.array_equal(_device_order(e, rc), order)
        _check_binning(e, n, w, h, order)
    v.dispose()


CONFIGS = [("default", {}), ("bincfg1", {"GS_BINCFG": 1}), ("nocompact", {"GS_BIN_COMPACT": 0}), ("bin1", {"GS_BIN": 1}),
           ("tma", {"GS_BLEND_TMA": 1})]


@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
@pytest.mark.parametrize("w,h", [(801, 455), (1920, 1080), (3840, 2160), (4096, 256), (8192, 256), (4096, 2160)])
def test_binning_configurations_agree(gs, monkeypatch, w, h, mode):
    """GS_BINCFG=1 (8 warps x 8 items in k_bin_count / k_bin_place), GS_BIN_COMPACT=0 (no warp compaction), GS_BIN=1 (emit + radix sort
    everywhere) and GS_BLEND_TMA=1 (bulk-copied list batches) all bin exactly as restated; since the lists are equal, so are the frames."""
    frames = {}
    for name, env in CONFIGS:
        _env(monkeypatch, **env)
        v = _viewer("adversarial" if mode == 0 else "bonsai", w, h, mode)
        e, n = v.engine, v.splatMesh.getSplatCount()
        frames[name] = v.frame(frame_format=gs._native.GS_FRAME_RGBA8).copy()
        _check_binning(e, n, w, h, _device_order(e, n), bin_version=int(env.get("GS_BIN", 2)))
        v.dispose()
    assert frames["default"][..., 3].max() > 0
    for name, _ in CONFIGS[1:]:
        assert np.array_equal(frames[name], frames["default"]), name


@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
@pytest.mark.parametrize("subset", [False, True], ids=["replicated", "subset"])
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("w,h", [(801, 455), (4096, 2160)])
def test_sharded_binning(gs, monkeypatch, w, h, world, subset, mode):
    """Each rank's lists are the GLOBAL draw order restricted to its coarse tiles, also when the rank sorted only its own subset."""
    from gaussiansplats3d_b200.parallel import combine_frames
    _env(monkeypatch, GS_SUBSET_MIN=1 if subset else 4_000_000_000)
    v1 = _viewer("bonsai", w, h, mode)
    n = v1.splatMesh.getSplatCount()
    single = v1.frame(frame_format=gs._native.GS_FRAME_RGBA8, flip_y=False).copy()
    order = _device_order(v1.engine, n)
    v1.dispose()
    frames = []
    for r in range(world):
        v = _viewer("bonsai", w, h, mode, rank=r, world_size=world)
        frames.append(v.frame(frame_format=gs._native.GS_FRAME_RGBA8, flip_y=False).copy())
        if not subset:
            assert np.array_equal(_device_order(v.engine, n), order)
        _check_binning(v.engine, n, w, h, order, r, world)
        v.dispose()
    assert np.array_equal(combine_frames(frames), single)


# ---- rects ------------------------------------------------------------------------------------------------------------------------
def _rect_coverage(rects, cx, cy, hx, hy, ok, w, h, tile):
    """(splats whose rect misses a fine tile holding a pixel centre inside the AABB c +- h, more than 1e-3 px from its edge;
    fraction of rects wider than the AABB's fine tiles by at least one whole fine tile)."""
    lo_x, hi_x = np.ceil(cx - hx - 0.5 + 1e-3), np.floor(cx + hx - 0.5 - 1e-3)
    lo_y, hi_y = np.ceil(cy - hy - 0.5 + 1e-3), np.floor(cy + hy - 0.5 - 1e-3)
    lo_x, lo_y = np.maximum(lo_x, 0), np.maximum(lo_y, 0)
    hi_x, hi_y = np.minimum(hi_x, w - 1), np.minimum(hi_y, h - 1)
    need = ok & (lo_x <= hi_x) & (lo_y <= hi_y)
    need &= np.isfinite(lo_x) & np.isfinite(lo_y) & np.isfinite(hi_x) & np.isfinite(hi_y)
    r = rects.astype(np.int64)
    tx0, tx1 = np.where(need, lo_x, 0).astype(np.int64) // tile, np.where(need, hi_x, 0).astype(np.int64) // tile
    ty0, ty1 = np.where(need, lo_y, 0).astype(np.int64) // tile, np.where(need, hi_y, 0).astype(np.int64) // tile
    ne = _nonempty(rects)
    miss = need & (~ne | (r[:, 0] > tx0) | (r[:, 1] > ty0) | (r[:, 2] < tx1) | (r[:, 3] < ty1))
    # the whole AABB (no margin, not clipped to pixel centres) in fine tiles: a rect tile outside it is pure cost
    ax0, ax1 = np.floor(np.maximum(cx - hx, 0) / tile), np.floor(np.minimum(cx + hx, w - 1) / tile)
    ay0, ay1 = np.floor(np.maximum(cy - hy, 0) / tile), np.floor(np.minimum(cy + hy, h - 1) / tile)
    wider = need & ne & ((r[:, 0] < ax0) | (r[:, 2] > ax1) | (r[:, 1] < ay0) | (r[:, 3] > ay1))
    return np.nonzero(miss)[0], wider.sum() / max(int(need.sum()), 1)


@pytest.mark.parametrize("scene", ["bonsai", "adversarial"])
@pytest.mark.parametrize("w,h", [(801, 455), (4096, 2160)])
def test_rects_are_conservative_3d(gs, oracle_mod, monkeypatch, w, h, scene):
    _env(monkeypatch)
    v = _viewer(scene, w, h, 0)
    e, n = v.engine, v.splatMesh.getSplatCount()
    v.frame(frame_format=gs._native.GS_FRAME_RGBA8)
    s = _state(e, n)
    dev = e.read_projected(n)
    p = v.splatMesh.packed
    want = oracle_mod.project(v.uniforms(), p.centers_colors, p.covariances, p.sh, p.sh_degree)
    hx = np.hypot(want["b1x"].astype(np.float64), want["b2x"])
    hy = np.hypot(want["b1y"].astype(np.float64), want["b2y"])
    ok = (want["valid"] == 1) & (dev["valid"] == 1)
    assert ok.sum() > 1000
    miss, wider = _rect_coverage(s["rects"], want["cx"].astype(np.float64), want["cy"].astype(np.float64), hx, hy, ok, w, h, s["tile_px"])
    print(f"3D {scene} {w}x{h}: {ok.sum()} splats, rect wider than the quad's AABB by a whole fine tile: {wider * 100:.2f} %")
    assert miss.size == 0, f"{miss.size} rects miss covered fine tiles, e.g. splat {miss[0]}: rect {s['rects'][miss[0]]}, " \
                           f"centre {want['cx'][miss[0]]:.3f},{want['cy'][miss[0]]:.3f} half {hx[miss[0]]:.3f},{hy[miss[0]]:.3f}"
    assert s["visible"] == int(_nonempty(s["rects"]).sum())
    v.dispose()


@pytest.mark.parametrize("scene", ["bonsai", "adversarial"])
@pytest.mark.parametrize("w,h", [(801, 455), (4096, 2160)])
def test_rects_are_conservative_2d(gs, monkeypatch, w, h, scene):
    import oracle.surfel as S
    _env(monkeypatch)
    v = _viewer(scene, w, h, 1)
    e, n = v.engine, v.splatMesh.getSplatCount()
    v.frame(frame_format=gs._native.GS_FRAME_RGBA8)
    dev = e.read_projected_2d(n)          # re-projects with the same parameters: same rects
    s = _state(e, n)
    p = v.splatMesh.packed
    want = S.project_2d(v.uniforms(), p.centers_colors, p.scale_rotations, p.sh, p.sh_degree)
    f64 = lambda k: want[k].astype(np.float64)      # noqa: E731
    hx, hy = np.abs(f64("h1x")) + np.abs(f64("h2x")), np.abs(f64("h1y")) + np.abs(f64("h2y"))
    ok = (want["valid"] == 1) & (dev["valid"] == 1) & (want["a"] > 0) & (dev["branch"] == want["branch"])
    assert ok.sum() > 1000
    miss, wider = _rect_coverage(s["rects"], f64("cx"), f64("cy"), hx, hy, ok, w, h, s["tile_px"])
    print(f"2D {scene} {w}x{h}: {ok.sum()} surfels, rect wider than the quad's AABB by a whole fine tile: {wider * 100:.2f} %")
    assert miss.size == 0, f"{miss.size} rects miss covered fine tiles, e.g. surfel {miss[0]}: rect {s['rects'][miss[0]]}"
    assert s["visible"] == int(_nonempty(s["rects"]).sum())
    v.dispose()


# ---- frames on the larger-frame paths ----------------------------------------------------------------------------------------------
def _check_frame(got, want):
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    assert err.max() <= TOL_WORST, f"worst channel error {err.max() * 255:.2f}/255"
    assert (err <= TOL_MOST).mean() >= FRAC, f"only {(err <= TOL_MOST).mean() * 100:.3f}% of channels within 2/255"
    return err.max()


def _crops(w, h, c=256):
    # right + bottom edges (GL rows: row 0 is the bottom), right + top edges, a coarse-tile corner of the 32-px tiling (256 x 128 px)
    return [(w - c, 0), (w - c, h - c), (1024 - c // 2, 1024 - c // 2), (0, h - c)]


@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
@pytest.mark.parametrize("w,h", [(4096, 2160), (7680, 4320)])
def test_radix_path_frames_match_oracle(gs, oracle_mod, monkeypatch, w, h, mode):
    import oracle.surfel as S
    _env(monkeypatch)
    v = _viewer("bonsai", w, h, mode, n=400_000)
    got = v.frame(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False).copy()
    n = v.splatMesh.getSplatCount()
    order = _device_order(v.engine, n)
    p = v.splatMesh.packed
    if mode == 0:
        ps = oracle_mod.project(v.uniforms(), p.centers_colors, p.covariances, p.sh, p.sh_degree)
        crop = lambda x0, y0: oracle_mod.blend_crop(ps, order, w, h, x0, y0, 256, 256)      # noqa: E731
    else:
        ps = S.project_2d(v.uniforms(), p.centers_colors, p.scale_rotations, p.sh, p.sh_degree)
        crop = lambda x0, y0: S.blend_2d_crop(ps, order, w, h, x0, y0, 256, 256)            # noqa: E731
    worst = 0.0
    for x0, y0 in _crops(w, h):
        want = crop(x0, y0)
        worst = max(worst, _check_frame(got[y0:y0 + 256, x0:x0 + 256], want))
    assert got[..., 3].max() > 0.5
    print(f"{'3D' if mode == 0 else '2D'} {w}x{h}: worst crop error {worst * 255:.3f}/255")
    v.dispose()


@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
def test_wide_strip_frame_matches_oracle(gs, oracle_mod, monkeypatch, mode):
    """8192 x 256: 512 fine tiles wide, so k_bin_place runs without its warp compaction; the whole frame against the oracle."""
    import oracle.surfel as S
    _env(monkeypatch)
    w, h = 8192, 256
    v = _viewer("bonsai", w, h, mode, n=200_000)
    got = v.frame(frame_format=gs._native.GS_FRAME_RGBA32F, flip_y=False).copy()
    n = v.splatMesh.getSplatCount()
    order = _device_order(v.engine, n)
    p = v.splatMesh.packed
    if mode == 0:
        want, _ = oracle_mod.render(v.uniforms(), p.centers_colors, p.covariances, order, w, h, sh=p.sh, sh_degree=p.sh_degree)
    else:
        want, _ = S.render_2d(v.uniforms(), p.centers_colors, p.scale_rotations, order, w, h, sh=p.sh, sh_degree=p.sh_degree)
    _check_frame(got, want)
    assert got[..., 3].max() > 0.5
    v.dispose()


@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
def test_radix_path_frame_variants_are_bit_equal(gs, monkeypatch, mode):
    """4096 x 2160 (radix path): gs_render, the graph frame, the frame without a graph and pipelined frames give the same RGBA8 picture
    with flip_y; and the RGBA8 picture is the float picture rounded, upside down."""
    from gaussiansplats3d_b200 import _native as N
    _env(monkeypatch)
    w, h = 4096, 2160
    v = _viewer("bonsai", w, h, mode, n=300_000)
    e, n = v.engine, v.splatMesh.getSplatCount()
    v.update()
    f32 = v.render(frame_format=N.GS_FRAME_RGBA32F, flip_y=False).copy()
    frames = {"render": v.render(frame_format=N.GS_FRAME_RGBA8, flip_y=True).copy(),
              "graph": v.frame(frame_format=N.GS_FRAME_RGBA8, flip_y=True).copy()}
    e.set_graph_enabled(False)
    frames["no_graph"] = v.frame(frame_format=N.GS_FRAME_RGBA8, flip_y=True).copy()
    e.set_graph_enabled(True)
    prep = e.prepare_frame(v.mvp_matrix().astype(np.float32), v.uniforms(), w, h, n, frame_format=N.GS_FRAME_RGBA8, flip_y=True)
    bufs = [N.pinned_empty((h, w, 4), np.uint8) for _ in range(2)]
    e.frame_begin(prep, bufs[0]); e.frame_begin(prep, bufs[1])
    e.frame_end(); e.frame_end()
    frames["pipelined0"], frames["pipelined1"] = bufs[0].copy(), bufs[1].copy()
    for k, f in frames.items():
        assert np.array_equal(f, frames["render"]), k
    want8 = np.floor(np.clip(f32[::-1], 0, 1) * np.float32(255) + np.float32(0.5))
    d = np.abs(frames["render"].astype(np.int32) - want8.astype(np.int32))
    assert d.max() <= 1 and (d == 0).mean() >= 0.9999
    assert frames["render"][..., 3].max() > 128
    v.dispose()


# ---- overflow ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1], ids=["3d", "2d"])
@pytest.mark.parametrize("w,h", [(1000, 600), (4096, 2160)])
def test_instance_overflow_is_reported_and_recovers(gs, monkeypatch, w, h, mode):
    """GS_INSTANCE_FACTOR=0 leaves room for 4 * (16-px tiles) + 65536 instances; a scene needing several times that must fail with
    GS_ERR_CAPACITY from gs_render, gs_frame and gs_frame_end, report the instance count it needed, keep every tile range inside the
    list, and leave the engine able to render a frame that fits, bit-equal to a fresh engine's, blocking and pipelined."""
    from gaussiansplats3d_b200 import _native as N
    _env(monkeypatch, GS_INSTANCE_FACTOR=0)
    n = 600_000

    def make():
        return _viewer("bonsai", w, h, mode, n=n, seed=9, scale=2.0)

    v = make()
    e = v.engine
    cap = int(e.read_buffer(N.GS_BUF_TILE_INFO, np.uint64, 1)[0])
    assert cap == 4 * (-(-w // 16)) * (-(-h // 16)) + 65536
    v.update()
    with pytest.raises(N.GsError) as ei:
        v.render(frame_format=N.GS_FRAME_RGBA8)
    assert ei.value.code == N.GS_ERR_CAPACITY
    m = re.search(r"(\d+) instances needed, capacity (\d+)", str(ei.value))
    assert m and int(m.group(2)) == cap, str(ei.value)
    s = _state(e, n)
    want = B.bin_frame(s["rects"], _device_order(e, n), w, h)
    assert int(m.group(1)) == want.total == s["total"], (m.group(1), want.total, s["total"])
    print(f"overflow {w}x{h} {'3D' if mode == 0 else '2D'}: {want.total} instances needed, capacity {cap} ({want.total / cap:.2f}x)")
    assert want.total >= 2 * cap
    rg = s["ranges"].astype(np.int64)
    used = rg[:, 0] < rg[:, 1]
    assert (rg[used] <= cap).all()
    path = B.binning_path(w, h)
    if path == B.COUNTING:          # slots below the capacity hold exactly the instances that belong there
        assert np.array_equal(s["ranges"], want.ranges(path, capacity=cap))
        assert np.array_equal(s["list"], want.entries[:cap])
    else:
        assert (rg[~used] == B.EMPTY_RANGE).all()
    mvp, u = v.mvp_matrix().astype(np.float32), v.uniforms()
    with pytest.raises(N.GsError) as ei:
        e.frame(mvp, u, w, h, n)
    assert ei.value.code == N.GS_ERR_CAPACITY
    buf = N.pinned_empty((h, w, 4), np.uint8)
    e.frame_begin(e.prepare_frame(mvp, u, w, h, n), buf)
    with pytest.raises(N.GsError) as ei:
        e.frame_end()
    assert ei.value.code == N.GS_ERR_CAPACITY
    # a frame that fits (the first 5 000 splats), after the overflow, equals a fresh engine's frame
    rc = 5_000
    fresh = make()
    want_frame = fresh.engine.frame(mvp, u, w, h, rc).copy()
    fresh.dispose()
    assert want_frame[..., 3].max() > 0
    assert np.array_equal(e.frame(mvp, u, w, h, rc), want_frame)
    assert e.timings()["tile_instances"] <= cap
    with pytest.raises(N.GsError):
        e.frame(mvp, u, w, h, n)
    e.frame_begin(e.prepare_frame(mvp, u, w, h, rc), buf)
    e.frame_end()
    assert np.array_equal(buf, want_frame)
    v.dispose()


# ---- the sharded diagonal limit -------------------------------------------------------------------------------------------------
def test_sharded_frames_beyond_the_diagonal_limit_are_refused(gs, monkeypatch):
    """Sharded ownership covers coarse-tile diagonals cx + cy up to 127.  24576 x 64 (192 coarse tiles in a row, diagonals up to 191)
    is refused on every rank; 16384 x 64 (diagonals up to 127) renders, and its ranks sum to the single-engine frame bit for bit."""
    from gaussiansplats3d_b200 import _native as N
    from gaussiansplats3d_b200.parallel import combine_frames
    _env(monkeypatch)
    world = 3
    for r in range(world):
        v = _viewer("bonsai", 24576, 64, 0, n=20_000, rank=r, world_size=world)
        with pytest.raises(N.GsError) as ei:
            v.frame(frame_format=N.GS_FRAME_RGBA8)
        assert ei.value.code == N.GS_ERR_BAD_ARG and "diagonal" in str(ei.value)
        v.update()
        with pytest.raises(N.GsError) as ei:
            v.render(frame_format=N.GS_FRAME_RGBA8)
        assert ei.value.code == N.GS_ERR_BAD_ARG
        v.dispose()
    w, h = 16384, 64
    assert B.geometry(w, h).max_diagonal == 127
    v1 = _viewer("bonsai", w, h, 0, n=100_000)
    single = v1.frame(frame_format=N.GS_FRAME_RGBA8, flip_y=False).copy()
    order = _device_order(v1.engine, 100_000)
    v1.dispose()
    frames = []
    for r in range(world):
        v = _viewer("bonsai", w, h, 0, n=100_000, rank=r, world_size=world)
        frames.append(v.frame(frame_format=N.GS_FRAME_RGBA8, flip_y=False).copy())
        _check_binning(v.engine, 100_000, w, h, order, r, world)
        v.dispose()
    assert single[..., 3].max() > 0
    assert np.array_equal(combine_frames(frames), single)
