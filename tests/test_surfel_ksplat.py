"""`.ksplat` files in the TwoD (surfel) render mode: the scale/rotation texture decoded on the GPU (k_ksplat_decode's SR variant)
against the scalar restatement of SplatBuffer.fillSplatScaleRotationArray (oracle/surfel_pack_oracle.py), on the hand-assembled
fixtures, without and with a scene transform; and the frame of a .ksplat-loaded TwoD viewer against the same data uploaded as arrays."""
import numpy as np
import pytest

from oracle import surfel_pack_oracle as SP

TRANSFORMS = {"none": None, "trs": dict(position=(0.3, -0.2, 0.5), rotation=(0.1, 0.35, -0.2, 0.9), scale=(1.3, 0.8, 1.1))}


def _handmade(name):
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
    import ksplat_handmade as HM
    return HM.fixture(name)


def _names():
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
    import ksplat_handmade as HM
    return list(HM.FIXTURES)


def _transform16(kind):
    from gaussiansplats3d_b200 import three_math as TM
    t = TRANSFORMS[kind]
    if t is None:
        return None
    q = np.asarray(t["rotation"], np.float64)
    q /= np.linalg.norm(q)
    return np.asarray(TM.compose(t["position"], tuple(q), t["scale"]), np.float64).reshape(16), dict(t, rotation=tuple(q))


@pytest.mark.parametrize("kind", list(TRANSFORMS))
@pytest.mark.parametrize("name", _names())
def test_oracle_fill_uses_the_fixture_values(name, kind):
    """The restatement's fill starts from the scales and quaternions the fixture was assembled from (not from a decoder under test)."""
    data, exp = _handmade(name)
    tt = _transform16(kind)
    t = None if tt is None else tt[0]
    n = exp["count"]
    sc = np.array(exp["scales"], np.float32).reshape(n, 3)
    rot = np.array(exp["rot_xyzw"], np.float32).reshape(n, 4)
    sz = SP.scale_z_override(exp["level"])
    want = np.array([SP.scale_rotation_one(sc[i], rot[i], t, sz) for i in range(n)], np.float32)
    got = SP.ksplat_scale_rotations(data, t)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    if exp["level"] and t is None:
        assert np.all(got[:, 2] == np.float32(2.0 ** -24))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(TRANSFORMS))
@pytest.mark.parametrize("name", _names())
def test_gpu_decodes_scale_rotations_and_renders_like_arrays(gs, name, kind):
    from gaussiansplats3d_b200 import _native as N
    from gaussiansplats3d_b200.viewer import Viewer
    from oracle import ksplat_oracle as KO
    data, exp = _handmade(name)
    tt = _transform16(kind)
    t16, pose = (None, {}) if tt is None else tt
    n = exp["count"]
    d = KO.decode(data, transform16=t16)
    centre = d["centers"].astype(np.float64).mean(0)
    extent = max(float(np.abs(d["centers"] - centre).max()), 0.05)
    w = h = 64
    v = Viewer(dict(width=w, height=h, splatRenderMode=1, sphericalHarmonicsDegree=2, cameraUp=(0, 1, 0),
                    initialCameraPosition=tuple(centre + np.array([0.3, 0.4, 4.0]) * extent), initialCameraLookAt=tuple(centre)))
    info = v.addSplatSceneFromKSplat(data, **pose)
    assert info["splat_count"] == n
    sr = SP.ksplat_scale_rotations(data, t16)
    got_sr = v.engine.read_buffer(N.GS_BUF_SCALE_ROTATIONS, np.uint32, 6 * n).reshape(n, 6)
    assert np.array_equal(got_sr, sr.view(np.uint32))
    assert np.array_equal(v.engine.read_buffer(N.GS_BUF_CENTERS_COLORS, np.uint32, 4 * n).reshape(n, 4), d["centers_colors"])
    v.camera.update(); v.updateSplatMesh()
    got = v.frame(frame_format=N.GS_FRAME_RGBA32F, flip_y=False).copy()
    # the same data through the host-packed path: arrays + sorter centres into a fresh TwoD engine, same camera and uniforms
    with gs.Engine(n, max_width=w, max_height=h, splat_render_mode=1) as e:
        e.upload_splat_data(d["centers_colors"], None, d["sh"], d["sh_degree"] if d["sh"] is not None else 0, scale_rotations=sr)
        e.upload_centers(d["int_centers"])
        want = e.frame(v.mvp_matrix().astype(np.float32), v.uniforms(), w, h, n, frame_format=N.GS_FRAME_RGBA32F, flip_y=False)
    assert np.array_equal(got, want)
    assert got[..., 3].max() > 0.0, "the fixture's surfels must be on screen"
    v.dispose()
