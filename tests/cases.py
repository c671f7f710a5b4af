"""Seeded input generators shared by the CPU (oracle) and GPU (parity) tests.  No reference code, no product code."""
from __future__ import annotations

import numpy as np


def perspective(fov_deg=50.0, aspect=16 / 9, near=0.1, far=1000.0) -> np.ndarray:
    """three.js PerspectiveCamera.updateProjectionMatrix -> Matrix4.makePerspective (column-major, f64)."""
    top = near * np.tan(np.deg2rad(0.5 * fov_deg))
    height = 2 * top
    width = aspect * height
    left = -0.5 * width
    right, bottom = left + width, top - height
    m = np.zeros(16)
    m[0] = 2 * near / (right - left)
    m[5] = 2 * near / (top - bottom)
    m[8] = (right + left) / (right - left)
    m[9] = (top + bottom) / (top - bottom)
    m[10] = -(far + near) / (far - near)
    m[11] = -1.0
    m[14] = -2 * far * near / (far - near)
    return m


def look_at_world(eye, target, up) -> np.ndarray:
    """camera.matrixWorld for position `eye` looking at `target` (three.js Object3D.lookAt for cameras), column-major f64."""
    eye, target, up = (np.asarray(v, np.float64) for v in (eye, target, up))
    z = eye - target
    z /= np.linalg.norm(z)
    x = np.cross(up, z)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    m = np.eye(4)
    m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = x, y, z, eye
    return m.T.reshape(16).copy()  # column-major flat


def mat(colmajor16) -> np.ndarray:
    return np.asarray(colmajor16, np.float64).reshape(4, 4).T


def flat(m4) -> np.ndarray:
    return np.asarray(m4, np.float64).T.reshape(16).copy()


def camera_mvp(eye=(0, 10, 15), target=(0, 0, 0), up=(0, 1, 0), aspect=16 / 9):
    """(mvp f64[16], view f64[16], proj f64[16]) like Viewer.runSplatSort (Viewer.js:1888-1891), mesh at identity."""
    world = mat(look_at_world(eye, target, up))
    view = np.linalg.inv(world)
    proj = mat(perspective(aspect=aspect))
    return flat(proj @ view), flat(view), flat(proj)


def sort_case(seed: int, n: int, *, integer=True, dynamic=False, precomputed=False, index_kind="shuffled", sort_frac=1.0,
              scale=3.0, ties=False, n_scenes=4):
    """One sortIndexes() argument set (SURVEY 8c matrix)."""
    rng = np.random.default_rng(seed)
    xyz = rng.normal(0.0, scale, (n, 3)).astype(np.float32)
    if ties:  # many splats on a few depth planes -> long equal-bucket runs
        xyz = np.round(xyz / 2.0).astype(np.float32) * 2.0
    if integer:
        centers = np.empty((n, 4), np.int32)
        centers[:, :3] = np.floor(xyz.astype(np.float64) * 1000.0 + 0.5).astype(np.int32)
        centers[:, 3] = 1000
    else:
        centers = np.ones((n, 4), np.float32)
        centers[:, :3] = xyz
    eye = rng.normal(0, 1, 3) * 8 + np.array([0, 4, 12.0])
    mvp64, _, _ = camera_mvp(eye=eye, target=rng.normal(0, 1, 3), up=(0, 1, 0))
    mvp = mvp64.astype(np.float32)
    if index_kind == "identity":
        idx = np.arange(n, dtype=np.uint32)
    elif index_kind == "shuffled":
        idx = rng.permutation(n).astype(np.uint32)
    else:  # "octree": runs of nearby indexes in shuffled block order, a subset of the splats
        blocks = rng.permutation((n + 255) // 256)
        idx = np.concatenate([np.arange(b * 256, min(n, (b + 1) * 256)) for b in blocks]).astype(np.uint32)
    render_count = n if index_kind != "octree" else max(1, int(n * 0.8))
    idx = idx[:render_count] if index_kind == "octree" else idx
    sort_count = max(0, min(render_count, int(round(render_count * sort_frac))))
    scene_indexes = transforms = None
    if dynamic:
        scene_indexes = rng.integers(0, n_scenes, n, dtype=np.uint32)
        if index_kind == "octree":
            scene_indexes = np.sort(scene_indexes)
        transforms = np.zeros((32, 16), np.float32)
        for s in range(32):
            a = rng.normal(0, 1, (3, 3))
            q, _ = np.linalg.qr(a)
            t = np.eye(4)
            t[:3, :3] = q * rng.uniform(0.5, 2.0)
            t[:3, 3] = rng.normal(0, 2, 3)
            transforms[s] = t.T.reshape(16)
    pre = None
    if precomputed:
        if integer:
            pre = rng.integers(-2_000_000, 2_000_000, n, dtype=np.int64).astype(np.int32)
        else:
            pre = rng.normal(0, 40, n).astype(np.float32)
    return dict(indexes=idx, centers=centers, precomputed=pre, mvp=mvp, scene_indexes=scene_indexes, transforms=transforms,
                sort_count=sort_count, render_count=render_count, splat_count=n, use_precomputed=precomputed, integer_sort=integer,
                dynamic_mode=dynamic)


def sort_matrix(n=20000, seeds=(0,)):
    """(name, kwargs) for the six distance branches x ranges x partial sorts x index kinds x adversarial inputs."""
    out = []
    for seed in seeds:
        for integer in (True, False):
            for dynamic, pre in ((False, False), (True, False), (False, True)):
                for kind in ("identity", "shuffled", "octree"):
                    for frac in (1.0, 0.37):
                        name = f"s{seed}-{'int' if integer else 'flt'}-{'dyn' if dynamic else ('pre' if pre else 'sta')}-{kind}-{frac}"
                        out.append((name, dict(seed=seed, n=n, integer=integer, dynamic=dynamic, precomputed=pre, index_kind=kind, sort_frac=frac)))
        out.append((f"s{seed}-ties", dict(seed=seed, n=n, ties=True)))
        out.append((f"s{seed}-ties-flt", dict(seed=seed, n=n, ties=True, integer=False)))
        out.append((f"s{seed}-tiny", dict(seed=seed, n=7)))
        out.append((f"s{seed}-one-tile-edge", dict(seed=seed, n=4096)))
        out.append((f"s{seed}-tile-plus-one", dict(seed=seed, n=4097)))
        out.append((f"s{seed}-sort0", dict(seed=seed, n=1000, sort_frac=0.0)))
        out.append((f"s{seed}-wide", dict(seed=seed, n=n, scale=60.0)))
    return out


def property_case(seed, n, integer, mode, kind, frac, rbits, ties):
    """(case, distance_map_range) of one property example: mode is "static", "dynamic" or "precomputed", the range is 2^rbits."""
    c = sort_case(seed=seed, n=n, integer=integer, dynamic=(mode == "dynamic"), precomputed=(mode == "precomputed"), index_kind=kind,
                  sort_frac=frac, ties=ties and mode != "precomputed")
    return c, 1 << rbits


RANGES = (1 << 10, 1 << 16, 1 << 20)


def call_args(case, R):
    return (case["indexes"], case["centers"], case["precomputed"], case["mvp"], case["scene_indexes"], case["transforms"], R,
            case["sort_count"], case["render_count"], case["splat_count"], case["use_precomputed"], case["integer_sort"], case["dynamic_mode"])
