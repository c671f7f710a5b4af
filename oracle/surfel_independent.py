"""oracle/surfel_independent.py -- TEST INFRASTRUCTURE ONLY.

An independent formulation of the TwoD (surfel) material that pins oracle/surfel_oracle.c, in the way raster_independent.py pins the
3D restatement.  It shares none of that file's algebra: everything is float64 geometry instead of the shader's matrix chain --
  * rotation from scipy.spatial.transform.Rotation (not the shader's quaternion formula);
  * rho3d from the intersection of the world-space ray through the pixel with the surfel's plane (tangent-frame coordinates of the
    hit point), the pixel mapped to NDC with the reference's (W - 1) / 2 offset of ndc2pix; the near test on the hit point's clip w;
  * the fallback square's centre and radius from the extremes of the projected unit circle (sampled), not from the dual conic;
  * coverage from the software triangle rasteriser of the 4-vertex quad (raster_independent.rasterise_quad_triangles).
"""
from __future__ import annotations

import numpy as np
from scipy.spatial.transform import Rotation

from .raster_independent import rasterise_quad_triangles


def _mat(colmajor16) -> np.ndarray:
    return np.asarray(colmajor16, np.float64).reshape(4, 4).T


def render(uniforms, centers_colors, scale_rotations, order, width, height) -> tuple[np.ndarray, list]:
    """SH degree 0.  Float RGBA frame (rows bottom-up) and the per-splat quad branch (0 eigen, 1 fallback, None not drawn), draw order = `order`."""
    PMV = _mat(uniforms.projection) @ _mat(uniforms.model_view)
    inv = np.linalg.inv(PMV)
    W, H = float(uniforms.viewport[0]), float(uniforms.viewport[1])
    ifa = float(uniforms.inverse_focal_adjustment)
    cc = np.asarray(centers_colors, np.uint32).reshape(-1, 4)
    centers = cc[:, 1:].view(np.float32).astype(np.float64)
    rgba = np.stack([(cc[:, 0] >> (8 * k)) & 255 for k in range(4)], 1).astype(np.float64) / 255.0
    sr = np.asarray(scale_rotations, np.float64).reshape(-1, 6)
    ys, xs = np.mgrid[0:height, 0:width]
    fx, fy = xs + 0.5, ys + 0.5
    # world-space ray of every pixel: NDC with the (W-1)/2 offset, unprojected at the near and far planes
    nx, ny = (fx - (W - 1.0) / 2.0) / (W / 2.0), (fy - (H - 1.0) / 2.0) / (H / 2.0)

    def unproject(z):
        p = np.stack([nx, ny, np.full_like(nx, z), np.ones_like(nx)], -1) @ inv.T
        return p[..., :3] / p[..., 3:]
    o = unproject(-1.0)
    d = unproject(1.0) - o

    def clip(p):
        return PMV @ np.append(p, 1.0)

    def ndc(p):
        c = clip(p)
        return c[:3] / c[3]
    frame = np.zeros((height, width, 4))
    branches = []
    for s in np.asarray(order):
        c0 = centers[s]
        cl = clip(c0)
        if cl[2] < -1.2 * cl[3] or abs(cl[0]) > 1.2 * cl[3] or abs(cl[1]) > 1.2 * cl[3]:
            branches.append(None)
            continue
        q = sr[s, 3:]
        w = np.sqrt(max(0.0, 1.0 - q @ q))
        R = Rotation.from_quat([q[0], q[1], q[2], w]).as_matrix()
        tu, tv = R[:, 0] * sr[s, 0], R[:, 1] * sr[s, 1]
        nc = ndc(c0)
        if not -1.0 <= nc[2] <= 1.0:
            branches.append(None)
            continue
        centre_px = (nc[:2] * 0.5 + 0.5) * np.array([W, H])
        b1 = (ndc(c0 + tu) - nc)[:2] * 0.5 * np.array([W, H])
        b2 = (ndc(c0 + tv) - nc)[:2] * 0.5 * np.array([W, H])
        if np.hypot(*b1) < 1.0 or np.hypot(*b2) < 1.0:
            th = np.linspace(0.0, 2.0 * np.pi, 8192, endpoint=False)
            ring = c0[None] + np.cos(th)[:, None] * tu[None] + np.sin(th)[:, None] * tv[None]
            rc = np.c_[ring, np.ones(len(th))] @ PMV.T
            px = rc[:, 0] / rc[:, 3] * (W / 2.0) + (W - 1.0) / 2.0
            py = rc[:, 1] / rc[:, 3] * (H / 2.0) + (H - 1.0) / 2.0
            qc = np.array([(px.min() + px.max()) / 2.0, (py.min() + py.max()) / 2.0])
            radius = max(0.01, (px.max() - px.min()) / 2.0, (py.max() - py.min()) / 2.0)
            B1, B2 = np.array([3.0 * radius, 0.0]), np.array([0.0, 3.0 * radius])
            branches.append(1)
        else:
            qc = nc[:2]                     # vQuadCenter of the eigen branch: NDC units
            B1, B2 = 3.0 * ifa * b1, 3.0 * ifa * b2
            branches.append(0)
        covered, _ = rasterise_quad_triangles(centre_px, B1, B2, width, height)
        if not covered.any():
            continue
        # ray / plane: o + t d = c0 + u tu + v tv
        dd = d[covered]
        rhs = o[covered] - c0[None]
        A = np.empty((dd.shape[0], 3, 3))
        A[:, :, 0], A[:, :, 1], A[:, :, 2] = tu[None], tv[None], -dd
        with np.errstate(all="ignore"):
            sol = np.linalg.solve(A, rhs[..., None])[..., 0]
        u, v, t = sol[:, 0], sol[:, 1], sol[:, 2]
        hit = o[covered] + t[:, None] * dd
        hw = np.c_[hit, np.ones(len(hit))] @ PMV[3]
        rho3d = u * u + v * v
        rho2d = 2.0 * ((qc[0] - fx[covered]) ** 2 + (qc[1] - fy[covered]) ** 2)
        rho = np.minimum(rho3d, rho2d)
        depth = np.where(rho3d <= rho2d, hw, cl[3])
        alpha = np.minimum(0.99, rgba[s, 3] * np.exp(-0.5 * rho))
        ok = np.isfinite(rho) & (depth >= 0.2) & (alpha >= 1.0 / 255.0)
        a = np.where(ok, alpha, 0.0)[:, None]
        px = frame[covered]
        px[:, :3] = rgba[s, :3][None] * a + px[:, :3] * (1.0 - a)
        px[:, 3:] = a + px[:, 3:] * (1.0 - a)
        frame[covered] = px
    return frame, branches
