"""Seeded synthetic splat scenes standing in for the reference's demo data (bonsai / garden .ksplat files are an
external download that is not on disk: README.md:121) and the packing of raw splat attributes into the arrays the
reference's SplatMesh uploads (the load-time CPU loops of SplatBuffer.js / SplatMesh.js, done here with NumPy).

Sizes, SH degrees and cameras follow BASELINE.json `configs` / SURVEY.md 8(d)."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass
class RawScene:
    """Uncompressed per-splat attributes, the content of a level-0 SplatBuffer (SplatBuffer.js:108-163)."""
    centers: np.ndarray      # f32 [n,3]
    scales: np.ndarray       # f32 [n,3] linear
    rotations: np.ndarray    # f32 [n,4] x,y,z,w (unit)
    colors: np.ndarray       # u8  [n,4] rgba
    sh: np.ndarray | None    # f32 [n, ncoef, 3] coefficient-major RGB triples (the GPU-side order), or None
    sh_degree: int

    @property
    def count(self) -> int:
        return self.centers.shape[0]


def synthetic_scene(n: int, seed: int, kind: str = "bonsai", sh_degree: int = 0) -> RawScene:
    """bonsai: clustered N(0,1.5^2) + 10% shell r=6.  garden: same + ground-plane disc r=12.  uniform: N(0,3^2)."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        centers = rng.normal(0.0, 3.0, (n, 3))
    else:
        n_shell = n // 10
        n_disc = n // 4 if kind == "garden" else 0
        n_core = n - n_shell - n_disc
        core = rng.normal(0.0, 1.5, (n_core, 3))
        d = rng.normal(0, 1, (n_shell, 3))
        shell = 6.0 * d / np.linalg.norm(d, axis=1, keepdims=True)
        parts = [core, shell]
        if n_disc:
            r = 12.0 * np.sqrt(rng.uniform(0, 1, n_disc))
            th = rng.uniform(0, 2 * np.pi, n_disc)
            parts.append(np.stack([r * np.cos(th), rng.normal(-1.5, 0.05, n_disc), r * np.sin(th)], 1))
        centers = np.concatenate(parts, 0)
        centers = centers[rng.permutation(n)]
    log_scales = np.clip(rng.normal(-4.5, 1.2, (n, 3)), -8.0, -1.0)
    scales = np.exp(log_scales)
    q = rng.normal(0, 1, (n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[q[:, 3] < 0] *= -1.0
    colors = np.empty((n, 4), np.uint8)
    colors[:, :3] = rng.integers(0, 256, (n, 3), dtype=np.uint8)
    colors[:, 3] = (255.0 * (1.0 - rng.uniform(0, 1, n) ** 3)).astype(np.uint8)  # skewed high
    sh = None
    if sh_degree > 0:
        ncoef = 3 if sh_degree == 1 else 8
        sh = rng.normal(0.0, 0.15, (n, ncoef, 3)).astype(np.float32)
    return RawScene(centers.astype(np.float32), scales.astype(np.float32), q.astype(np.float32), colors, sh, sh_degree)


def compute_covariances(scales: np.ndarray, rotations_xyzw: np.ndarray, transform3x3: np.ndarray | None = None) -> np.ndarray:
    """SplatBuffer.computeCovariance (SplatBuffer.js:440-486): Sigma = (R S)(R S)^T [then T Sigma T^T], evaluated in
    float64, stored as float32 [m00, m01, m02, m11, m12, m22]."""
    s = scales.astype(np.float64)
    x, y, z, w = (rotations_xyzw[:, k].astype(np.float64) for k in range(4))
    x2, y2, z2 = x + x, y + y, z + z
    xx, xy, xz, yy, yz, zz, wx, wy, wz = x * x2, x * y2, x * z2, y * y2, y * z2, z * z2, w * x2, w * y2, w * z2
    R = np.empty((scales.shape[0], 3, 3))
    R[:, 0, 0], R[:, 0, 1], R[:, 0, 2] = 1 - (yy + zz), xy - wz, xz + wy
    R[:, 1, 0], R[:, 1, 1], R[:, 1, 2] = xy + wz, 1 - (xx + zz), yz - wx
    R[:, 2, 0], R[:, 2, 1], R[:, 2, 2] = xz - wy, yz + wx, 1 - (xx + yy)
    M = R * s[:, None, :]
    cov = M @ np.transpose(M, (0, 2, 1))
    if transform3x3 is not None:
        T = np.asarray(transform3x3, np.float64)
        cov = T @ cov @ T.T
    out = np.stack([cov[:, 0, 0], cov[:, 0, 1], cov[:, 0, 2], cov[:, 1, 1], cov[:, 1, 2], cov[:, 2, 2]], 1)
    return out.astype(np.float32)


# ---- static-scene transform baked at load (SplatMesh.fillSplatDataArrays, SplatMesh.js:1853-1897) ------------------------------------
def rotation_of_transform(transform16) -> np.ndarray:
    """The rotation a scene transform applies to spherical harmonics (SplatBuffer.js:628-632): Matrix4.decompose -> quaternion ->
    normalize -> makeRotationFromQuaternion, in three.js's own operation order (reciprocal multiplies, x2 = x + x products).
    `transform16`: column-major 4x4.  Returns the 3x3 rotation (row, column)."""
    e = [float(v) for v in np.asarray(transform16, np.float64).reshape(16)]
    sx = np.sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2])
    sy = np.sqrt(e[4] * e[4] + e[5] * e[5] + e[6] * e[6])
    sz = np.sqrt(e[8] * e[8] + e[9] * e[9] + e[10] * e[10])
    m = np.array(e).reshape(4, 4).T[:3, :3]
    if np.linalg.det(m) < 0:      # three.js flips the x scale for a mirrored basis
        sx = -sx
    isx, isy, isz = 1.0 / sx, 1.0 / sy, 1.0 / sz
    m11, m21, m31 = e[0] * isx, e[1] * isx, e[2] * isx          # m<row><col>, column-major elements
    m12, m22, m32 = e[4] * isy, e[5] * isy, e[6] * isy
    m13, m23, m33 = e[8] * isz, e[9] * isz, e[10] * isz
    t = m11 + m22 + m33
    if t > 0:                      # Quaternion.setFromRotationMatrix
        k = 0.5 / np.sqrt(t + 1.0)
        w, x, y, z = 0.25 / k, (m32 - m23) * k, (m13 - m31) * k, (m21 - m12) * k
    elif m11 > m22 and m11 > m33:
        k = 2.0 * np.sqrt(1.0 + m11 - m22 - m33)
        w, x, y, z = (m32 - m23) / k, 0.25 * k, (m12 + m21) / k, (m13 + m31) / k
    elif m22 > m33:
        k = 2.0 * np.sqrt(1.0 + m22 - m11 - m33)
        w, x, y, z = (m13 - m31) / k, (m12 + m21) / k, 0.25 * k, (m23 + m32) / k
    else:
        k = 2.0 * np.sqrt(1.0 + m33 - m11 - m22)
        w, x, y, z = (m21 - m12) / k, (m13 + m31) / k, (m23 + m32) / k, 0.25 * k
    ln = np.sqrt(x * x + y * y + z * z + w * w)      # Quaternion.normalize
    if ln == 0:
        x, y, z, w = 0.0, 0.0, 0.0, 1.0
    else:
        ln = 1.0 / ln
        x, y, z, w = x * ln, y * ln, z * ln, w * ln
    x2, y2, z2 = x + x, y + y, z + z                 # Matrix4.makeRotationFromQuaternion = compose(zero, q, one)
    xx, xy, xz, yy, yz, zz, wx, wy, wz = x * x2, x * y2, x * z2, y * y2, y * z2, z * z2, w * x2, w * y2, w * z2
    return np.array([[1 - (yy + zz), xy - wz, xz + wy],
                     [xy + wz, 1 - (xx + zz), yz - wx],
                     [xz - wy, yz + wx, 1 - (xx + yy)]])


def sh_rotation_matrices(rot3x3: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Band-1 (3x3) and band-2 (5x5) coefficient rotations in the reference's coefficient order and sign convention
    (SplatBuffer.js:632-634 for band 1, rotateSphericalHarmonics5 :780-816 for band 2).  Row l holds the weights of the INPUT
    coefficients that make OUTPUT coefficient l."""
    r = np.asarray(rot3x3, np.float64)
    m1 = np.array([[r[1, 1], -r[1, 2], r[1, 0]],
                   [-r[2, 1], r[2, 2], -r[2, 0]],
                   [r[0, 1], -r[0, 2], r[0, 0]]])
    a, b, c = m1[0], m1[1], m1[2]          # tsh11, tsh12, tsh13
    k14, k34, k13, k43, k112 = np.sqrt(1 / 4), np.sqrt(3 / 4), np.sqrt(1 / 3), np.sqrt(4 / 3), np.sqrt(1 / 12)

    def sym(u, v):     # the (u, v) product pattern shared by rows 1, 2 and 4
        return np.array([k14 * ((u[2] * v[0] + u[0] * v[2]) + (v[2] * u[0] + v[0] * u[2])),
                         u[1] * v[0] + v[1] * u[0],
                         k34 * (u[1] * v[1] + v[1] * u[1]),
                         u[1] * v[2] + v[1] * u[2],
                         k14 * ((u[2] * v[2] - u[0] * v[0]) + (v[2] * u[2] - v[0] * u[0]))])

    row3 = np.array([k13 * (b[2] * b[0] + b[0] * b[2]) - k112 * ((c[2] * c[0] + c[0] * c[2]) + (a[2] * a[0] + a[0] * a[2])),
                     k43 * b[1] * b[0] - k13 * (c[1] * c[0] + a[1] * a[0]),
                     b[1] * b[1] - k14 * (c[1] * c[1] + a[1] * a[1]),
                     k43 * b[1] * b[2] - k13 * (c[1] * c[2] + a[1] * a[2]),
                     k13 * (b[2] * b[2] - b[0] * b[0]) - k112 * ((c[2] * c[2] - c[0] * c[0]) + (a[2] * a[2] - a[0] * a[0]))])
    row5 = np.array([k14 * ((c[2] * c[0] + c[0] * c[2]) - (a[2] * a[0] + a[0] * a[2])),
                     c[1] * c[0] - a[1] * a[0],
                     k34 * (c[1] * c[1] - a[1] * a[1]),
                     c[1] * c[2] - a[1] * a[2],
                     k14 * ((c[2] * c[2] - c[0] * c[0]) - (a[2] * a[2] - a[0] * a[0]))])
    m2 = np.stack([sym(c, a), sym(b, a), row3, sym(b, c), row5])
    return m1, m2


def transform_scene(raw: RawScene, transform16) -> tuple[RawScene, np.ndarray]:
    """Centres and spherical harmonics of `raw` under a static scene transform, as the reference bakes them at load:
    centre.applyMatrix4 (SplatBuffer.js:340-342; f64 arithmetic, f32 storage) and the SH rotation above (:684-716).  Scales and
    quaternions stay as they are -- the covariance takes the transform's upper 3x3 instead (computeCovariance :461-466), which is
    returned as the second value for `compute_covariances`."""
    m = np.asarray(transform16, np.float64).reshape(4, 4).T
    c = raw.centers.astype(np.float64)
    w = c @ m[3, :3] + m[3, 3]                               # applyMatrix4 divides by w (1 for affine transforms)
    centers = ((c @ m[:3, :3].T + m[:3, 3]) / w[:, None]).astype(np.float32)
    sh = raw.sh
    if sh is not None and raw.sh_degree >= 1:
        m1, m2 = sh_rotation_matrices(rotation_of_transform(transform16))
        src = sh.astype(np.float64)
        out = np.empty_like(src)
        out[:, 0:3] = np.einsum("lk,nkc->nlc", m1, src[:, 0:3])
        if raw.sh_degree >= 2:
            out[:, 3:8] = np.einsum("lk,nkc->nlc", m2, src[:, 3:8])
        sh = out.astype(np.float32)
    return RawScene(centers, raw.scales, raw.rotations, raw.colors, sh, raw.sh_degree), m[:3, :3].copy()


def _quaternion_from_rotation(m11, m12, m13, m21, m22, m23, m31, m32, m33):
    """Quaternion.setFromRotationMatrix (three r160), vectorised in float64; returns x, y, z, w."""
    t = m11 + m22 + m33
    x, y, z, w = (np.empty_like(t) for _ in range(4))
    a = t > 0
    b = ~a & (m11 > m22) & (m11 > m33)
    c = ~a & ~b & (m22 > m33)
    d = ~a & ~b & ~c
    with np.errstate(divide="ignore", invalid="ignore"):
        k = 0.5 / np.sqrt(t + 1.0)
        w[a], x[a], y[a], z[a] = (0.25 / k)[a], ((m32 - m23) * k)[a], ((m13 - m31) * k)[a], ((m21 - m12) * k)[a]
        k = 2.0 * np.sqrt(1.0 + m11 - m22 - m33)
        w[b], x[b], y[b], z[b] = ((m32 - m23) / k)[b], (0.25 * k)[b], ((m12 + m21) / k)[b], ((m13 + m31) / k)[b]
        k = 2.0 * np.sqrt(1.0 + m22 - m11 - m33)
        w[c], x[c], y[c], z[c] = ((m13 - m31) / k)[c], ((m12 + m21) / k)[c], (0.25 * k)[c], ((m23 + m32) / k)[c]
        k = 2.0 * np.sqrt(1.0 + m33 - m11 - m22)
        w[d], x[d], y[d], z[d] = ((m21 - m12) / k)[d], ((m13 + m31) / k)[d], ((m23 + m32) / k)[d], (0.25 * k)[d]
    return x, y, z, w


def _normalize_quaternion(x, y, z, w):
    """Quaternion.normalize: multiply by 1 / length; a zero quaternion becomes (0, 0, 0, 1)."""
    ln = np.sqrt(x * x + y * y + z * z + w * w)
    zero = ln == 0
    with np.errstate(divide="ignore"):
        il = 1.0 / ln
    x, y, z, w = x * il, y * il, z * il, w * il
    x[zero], y[zero], z[zero], w[zero] = 0.0, 0.0, 0.0, 1.0
    return x, y, z, w


def compute_scale_rotations(scales: np.ndarray, rotations_xyzw: np.ndarray, transform16=None, scale_z: float = 1.0) -> np.ndarray:
    """The TwoD mode's scale/rotation texture: SplatBuffer.fillSplatScaleRotationArray (SplatBuffer.js:349-438) with the z scale
    overridden to `scale_z` (SplatMesh.js:1856-1863), packed 6 x f32 per splat [sx sy sz qx qy qz] like
    SplatMesh.updateScaleRotationsPaddedData (SplatMesh.js:1150-1170).  float64 in three.js's operation order: the quaternion is
    normalised; with a scene transform the matrix transform * R * S is decomposed (Matrix4.decompose) and the quaternion normalised
    again; finally w is made non-negative (ensurePositiveW)."""
    n = scales.shape[0]
    sx, sy = scales[:, 0].astype(np.float64), scales[:, 1].astype(np.float64)
    sz = np.full(n, float(scale_z))
    x, y, z, w = _normalize_quaternion(*(rotations_xyzw[:, k].astype(np.float64) for k in range(4)))
    if transform16 is not None:
        e = [float(v) for v in np.asarray(transform16, np.float64).reshape(16)]
        x2, y2, z2 = x + x, y + y, z + z     # makeRotationFromQuaternion, then the columns times makeScale's diagonal (exact)
        xx, xy, xz, yy, yz, zz, wx, wy, wz = x * x2, x * y2, x * z2, y * y2, y * z2, z * z2, w * x2, w * y2, w * z2
        r = [[1 - (yy + zz), xy - wz, xz + wy], [xy + wz, 1 - (xx + zz), yz - wx], [xz - wy, yz + wx, 1 - (xx + yy)]]
        rs = [[r[i][j] * (sx, sy, sz)[j] for j in range(3)] for i in range(3)]
        t = [[e[0], e[4], e[8]], [e[1], e[5], e[9]], [e[2], e[6], e[10]]]
        # Matrix4.multiplyMatrices(transform, R S): left-to-right sums (the fourth term, t[i][3] * 0, adds an exact zero)
        m = [[(t[i][0] * rs[0][j] + t[i][1] * rs[1][j]) + t[i][2] * rs[2][j] for j in range(3)] for i in range(3)]
        # Matrix4.decompose
        dsx = np.sqrt(m[0][0] * m[0][0] + m[1][0] * m[1][0] + m[2][0] * m[2][0])
        dsy = np.sqrt(m[0][1] * m[0][1] + m[1][1] * m[1][1] + m[2][1] * m[2][1])
        dsz = np.sqrt(m[0][2] * m[0][2] + m[1][2] * m[1][2] + m[2][2] * m[2][2])
        det = (-m[0][2] * m[1][1] * m[2][0] - m[0][0] * m[1][2] * m[2][1] + m[0][0] * m[1][1] * m[2][2]
               + m[0][2] * m[1][0] * m[2][1] - m[0][1] * m[1][0] * m[2][2] + m[0][1] * m[1][2] * m[2][0])
        dsx = np.where(det < 0, -dsx, dsx)
        isx, isy, isz = 1.0 / dsx, 1.0 / dsy, 1.0 / dsz
        x, y, z, w = _quaternion_from_rotation(m[0][0] * isx, m[0][1] * isy, m[0][2] * isz, m[1][0] * isx, m[1][1] * isy, m[1][2] * isz,
                                               m[2][0] * isx, m[2][1] * isy, m[2][2] * isz)
        x, y, z, w = _normalize_quaternion(x, y, z, w)
        sx, sy, sz = dsx, dsy, dsz
    flip = np.where(w < 0, -1.0, 1.0)
    out = np.stack([sx, sy, sz, x * flip, y * flip, z * flip], 1)
    return out.astype(np.float32)


def pack_centers_colors(centers: np.ndarray, colors: np.ndarray, minimum_alpha: int = 1) -> np.ndarray:
    """SplatMesh.updateCenterColorsPaddedData (SplatMesh.js:1143-1153) + fillSplatColorArray's alpha floor
    (SplatBuffer.js:541-542): uvec4 {r | g<<8 | b<<16 | a<<24, bits(x), bits(y), bits(z)}."""
    n = centers.shape[0]
    c = colors.astype(np.uint32)
    a = np.where(c[:, 3] >= minimum_alpha, c[:, 3], 0)
    out = np.empty((n, 4), np.uint32)
    out[:, 0] = c[:, 0] | (c[:, 1] << 8) | (c[:, 2] << 16) | (a << 24)
    out[:, 1:] = np.ascontiguousarray(centers, dtype=np.float32).view(np.uint32)
    return out


def integer_centers(centers: np.ndarray) -> np.ndarray:
    """SplatMesh.getIntegerCenters(padFour=true) (SplatMesh.js:1912-1926): Math.round(f32 * 1000.0) in f64, w = 1000."""
    n = centers.shape[0]
    out = np.empty((n, 4), np.int32)
    out[:, :3] = np.floor(centers.astype(np.float32).astype(np.float64) * 1000.0 + 0.5).astype(np.int32)
    out[:, 3] = 1000
    return out


def float_centers(centers: np.ndarray) -> np.ndarray:
    """SplatMesh.getFloatCenters(padFour=true) (SplatMesh.js:1935-1948): w = 1."""
    out = np.ones((centers.shape[0], 4), np.float32)
    out[:, :3] = centers
    return out


@dataclass
class PackedScene:
    """What SplatMesh keeps on the GPU (setupDataTextures, SplatMesh.js:637-898) + what it sends the sorter."""
    centers_colors: np.ndarray   # u32 [n,4]
    covariances: np.ndarray      # f32 or f16 [n,6]
    sh: np.ndarray | None        # f16 / u8 / f32 [n, ncomp]
    sh_degree: int
    int_centers: np.ndarray      # i32 [n,4]
    count: int
    scale_rotations: np.ndarray | None = None   # f32 [n,6], TwoD render mode only (instead of covariances)


def pack_scene(raw: RawScene, *, half_covariances: bool = False, sh_format: str = "f16", minimum_alpha: int = 1,
               sh8_range: tuple[float, float] = (-1.5, 1.5), transform16=None, render_mode: int = 0) -> PackedScene:
    """`transform16` (column-major 4x4): the static scene transform baked into centres, covariances and SH (non-dynamic meshes).
    `render_mode` 1 (SplatRenderMode.TwoD): the scale/rotation texture is built instead of the covariances (SplatMesh.js:1853-1870)."""
    t3 = None
    srot = None
    if render_mode == 1:
        srot = compute_scale_rotations(raw.scales, raw.rotations, transform16)
    if transform16 is not None:
        raw, t3 = transform_scene(raw, transform16)
    cov = None
    if render_mode != 1:
        cov = compute_covariances(raw.scales, raw.rotations, t3)
    if half_covariances and cov is not None:  # halfPrecisionCovariancesOnGPU
        cov = cov.astype(np.float16)
    sh = None
    if raw.sh is not None and raw.sh_degree > 0:
        flat = raw.sh.reshape(raw.count, -1)
        if sh_format == "f16":  # getTargetSphericalHarmonicsCompressionLevel >= 1 (SplatMesh.js:1064-1066)
            sh = flat.astype(np.float16)
        elif sh_format == "u8":  # SplatBuffer.js:22-26
            lo, hi = sh8_range
            sh = np.floor((np.clip(flat, lo, hi) - lo) / (hi - lo) * 255.0).astype(np.uint8)
        else:
            sh = flat.astype(np.float32)
    return PackedScene(pack_centers_colors(raw.centers, raw.colors, minimum_alpha), cov, sh, raw.sh_degree if sh is not None else 0,
                       integer_centers(raw.centers), raw.count, srot)


# Cameras of the reference's demo pages (demo/bonsai.html:38-41, demo/garden.html:38-41) and the Viewer default
# (Viewer.js:51-55)
CAMERAS = {
    "bonsai": dict(up=(0.01933, -0.75830, -0.65161), position=(1.54163, 2.68515, -6.37228), look_at=(0.45622, 1.95338, 1.51278)),
    "garden": dict(up=(0.0, -1.0, -0.54), position=(-3.15634, -0.16946, -0.51552), look_at=(1.52976, 2.27776, 1.65898)),
    "default": dict(up=(0.0, 1.0, 0.0), position=(0.0, 10.0, 15.0), look_at=(0.0, 0.0, 0.0)),
}
