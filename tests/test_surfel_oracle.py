"""CPU: the C restatement of the TwoD (surfel) material (oracle/surfel_oracle.c) against an independent float64 formulation
(oracle/surfel_independent.py), and the host packing of the scale/rotation texture against a scalar restatement
(oracle/surfel_pack_oracle.py)."""
import numpy as np
import pytest

from oracle import surfel_independent as SI
from oracle import surfel_pack_oracle as SP


def _scene(n, seed, big_fraction):
    from gaussiansplats3d_b200.scenes import synthetic_scene
    raw = synthetic_scene(n, seed=seed, kind="bonsai", sh_degree=0)
    raw.scales[: int(n * big_fraction)] *= 25.0
    return raw


def _uniforms_and_order(raw, w, h, cam):
    from gaussiansplats3d_b200.scenes import CAMERAS, pack_scene
    from gaussiansplats3d_b200.viewer import Viewer
    c = CAMERAS[cam] if isinstance(cam, str) else cam
    v = Viewer(dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=w, height=h))
    v.camera.update()
    # Viewer.updateSplatMesh without a GPU: the uniforms need only the camera and a SplatMesh's options
    from gaussiansplats3d_b200.viewer import SplatMesh
    v.splatMesh = SplatMesh(splatRenderMode=1)
    v.splatMesh.packed = pack_scene(raw, render_mode=1)
    v.updateSplatMesh()
    u = v.uniforms()
    # draw order: farthest first by view depth (the sort itself is tested elsewhere)
    mv = np.asarray(u.model_view, np.float64).reshape(4, 4).T
    z = (np.c_[raw.centers.astype(np.float64), np.ones(raw.count)] @ mv.T)[:, 2]
    return u, v.splatMesh.packed, np.argsort(z, kind="stable").astype(np.uint32)


@pytest.mark.parametrize("seed,cam,w,h,big", [(1, "bonsai", 96, 64, 0.3), (2, "garden", 80, 60, 0.5), (3, "default", 72, 48, 0.2)])
def test_restatement_agrees_with_independent_formulation(seed, cam, w, h, big):
    import oracle.surfel as S
    raw = _scene(400, seed, big)
    u, p, order = _uniforms_and_order(raw, w, h, cam)
    ps = S.project_2d(u, p.centers_colors, p.scale_rotations)
    got = S.blend_2d(ps, order, w, h)
    want, branches = SI.render(u, p.centers_colors, p.scale_rotations, order, w, h)
    drawn = [(s, b) for s, b in zip(order, branches) if b is not None]
    assert {0, 1} <= {b for _, b in drawn}, "both quad branches must be exercised"
    agree = np.mean([ps["branch"][s] == b for s, b in drawn if ps["valid"][s]])
    assert agree >= 0.99, agree
    # f32 against f64: a pixel centre within rounding of a quad edge, or a basis vector within rounding of 1 px (the branch test),
    # may land on the other side.  Everywhere else the two agree within 8/255; every pixel beyond that must be such a case.
    err = np.abs(got - want)
    assert (err <= 2.0 / 255).mean() >= 0.995, (err.max() * 255, (err <= 2.0 / 255).mean())
    disagree = {int(s) for s, b in drawn if ps["valid"][s] and ps["branch"][s] != b}
    for y, x in zip(*np.nonzero((err > 8.0 / 255).any(-1))):
        assert _on_a_quad_edge_or_branch_flip(ps, disagree, x + 0.5, y + 0.5), (x, y, err[y, x] * 255)
    assert got[..., 3].max() > 0.3


def _on_a_quad_edge_or_branch_flip(ps, disagree, fx, fy):
    """Some drawn surfel's quad has the pixel centre on its edge to within the f32 uncertainty of that edge, or its quad branch differs
    between the two formulations and its quad reaches the pixel.  The edge uncertainty is 1e-3 in quad-local units, except for the
    fallback square: its radius comes from pointImage^2 - temp, which cancels terms of order |pointImage|^2 px^2, so in f32 the
    radius is only known to about 8 eps |pointImage|^2 / (2 radius) px."""
    for s in np.nonzero(ps["valid"])[0]:
        q = ps[s]
        h1, h2 = np.array([q["h1x"], q["h1y"]], np.float64), np.array([q["h2x"], q["h2y"]], np.float64)
        det = h1[0] * h2[1] - h2[0] * h1[1]
        if not np.isfinite(det) or det == 0:
            continue
        dx, dy = fx - float(q["cx"]), fy - float(q["cy"])
        u, v = (dx * h2[1] - dy * h2[0]) / det, (dy * h1[0] - dx * h1[1]) / det
        m = max(abs(u), abs(v))
        tol = 1e-3
        if q["branch"] == 1:
            r = max(float(q["h1x"]) / 3.0, 0.01)
            dr = 8.0 * 2.0 ** -23 * (float(q["qcx"]) ** 2 + float(q["qcy"]) ** 2) / (2.0 * r)
            tol = max(tol, dr / r)
        if abs(m - 1.0) < tol or (int(s) in disagree and m <= 1.5):
            return True
    return False


def test_quad_centre_term_is_visible_near_the_window_origin():
    """One large surfel covering the whole window: the eigen branch's vQuadCenter is in NDC units, so rho2d = 2 |qc - pixel|^2 is small
    only within a few pixels of the window origin, and there it lowers alpha below the surfel's own value.  Both formulations agree."""
    import oracle.surfel as S
    from gaussiansplats3d_b200.scenes import RawScene
    raw = RawScene(np.array([[0.0, 0.0, 0.0]], np.float32), np.array([[3.0, 3.0, 1.0]], np.float32),
                   np.array([[0.0, 0.0, 0.0, 1.0]], np.float32), np.array([[200, 120, 40, 255]], np.uint8), None, 0)
    u, p, order = _uniforms_and_order(raw, 40, 30, "default")
    ps = S.project_2d(u, p.centers_colors, p.scale_rotations)
    assert ps["branch"][0] == 0 and ps["valid"][0] == 1
    got = S.blend_2d(ps, order, 40, 30)
    want, _ = SI.render(u, p.centers_colors, p.scale_rotations, order, 40, 30)
    assert np.abs(got - want).max() <= 2.0 / 255
    assert got[0, 0, 3] < 0.9 * got[15, 20, 3]


@pytest.mark.parametrize("with_transform", [False, True])
def test_host_scale_rotations_equal_scalar_restatement(with_transform):
    from gaussiansplats3d_b200 import three_math as TM
    from gaussiansplats3d_b200.scenes import pack_scene, synthetic_scene
    raw = synthetic_scene(2000, seed=7)
    raw.rotations[::3] *= -1.0                         # negative w: ensurePositiveW
    t = None
    if with_transform:
        q = np.array([0.1, 0.35, -0.2, 0.9]); q /= np.linalg.norm(q)
        t = np.asarray(TM.compose((0.6, -0.4, 0.8), tuple(q), (1.4, 0.7, 1.1)), np.float64).reshape(16)
    got = pack_scene(raw, transform16=t, render_mode=1).scale_rotations
    want = np.array([SP.scale_rotation_one(raw.scales[i], raw.rotations[i], t) for i in range(raw.count)], np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    if not with_transform:
        assert np.all(got[:, 2] == 1.0)                # the z scale override
    # a mirrored transform flips the sign of the x scale (Matrix4.decompose)
    m = np.asarray(TM.compose((0, 0, 0), (0, 0, 0, 1), (-1.0, 1.0, 1.0)), np.float64).reshape(16)
    got = pack_scene(raw, transform16=m, render_mode=1).scale_rotations
    want = np.array([SP.scale_rotation_one(raw.scales[i], raw.rotations[i], m) for i in range(raw.count)], np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)) and (got[:, 0] < 0).all()


def test_scale_override_reads_as_half_at_compressed_levels():
    """SplatMesh.js:1856-1863 passes scaleOverride.z = 1 through toUncompressedFloat: a half-float read at levels 1 and 2."""
    assert SP.scale_z_override(0) == 1.0
    assert SP.scale_z_override(1) == SP.scale_z_override(2) == 2.0 ** -24
