"""oracle/surfel_pack_oracle.py -- TEST INFRASTRUCTURE ONLY.

Scalar restatement, one splat at a time with Python floats (f64, like JS numbers), of the TwoD mode's scale/rotation fill:
SplatBuffer.fillSplatScaleRotationArray (src/loaders/SplatBuffer.js:349-438 of the reference) as SplatMesh.fillSplatDataArrays calls it
in SplatRenderMode.TwoD (SplatMesh.js:1853-1870, scaleOverride.z = 1):
  scale.set(sx, sy, toUncompressedFloat(1, level))   -- for a file at compression level 1 or 2 the override is read as a half: 2^-24
  rotation.set(x, y, z, w).normalize()
  transform: makeScale, makeRotationFromQuaternion, identity().premultiply(S).premultiply(R).premultiply(transform), decompose,
             rotation.normalize()
  ensurePositiveW
three.js r160 operation order (Matrix4.multiplyMatrices, decompose, Quaternion.setFromRotationMatrix / normalize)."""
import math


def half_to_float(h):
    s = -1.0 if h & 0x8000 else 1.0
    e, m = (h >> 10) & 31, h & 1023
    if e == 0:
        return s * m * 2.0 ** -24
    if e == 31:
        return s * math.inf if m == 0 else math.nan
    return s * (1.0 + m / 1024.0) * 2.0 ** (e - 15)


def scale_z_override(compression_level):
    """toUncompressedFloat(1, level) (SplatBuffer.js:12-20): 1 at level 0, fromHalfFloat(1) = 2^-24 at levels 1 and 2."""
    return 1.0 if compression_level == 0 else half_to_float(1)


def _normalize(x, y, z, w):
    ln = math.sqrt(x * x + y * y + z * z + w * w)
    if ln == 0:
        return 0.0, 0.0, 0.0, 1.0
    ln = 1.0 / ln
    return x * ln, y * ln, z * ln, w * ln


def _mat4_mul(a, b):
    """Matrix4.multiplyMatrices(a, b) on column-major element lists."""
    out = [0.0] * 16
    for i in range(4):
        for j in range(4):
            out[4 * j + i] = a[i] * b[4 * j] + a[4 + i] * b[4 * j + 1] + a[8 + i] * b[4 * j + 2] + a[12 + i] * b[4 * j + 3]
    return out


def _rotation_from_quaternion(x, y, z, w):
    x2, y2, z2 = x + x, y + y, z + z
    xx, xy, xz, yy, yz, zz, wx, wy, wz = x * x2, x * y2, x * z2, y * y2, y * z2, z * z2, w * x2, w * y2, w * z2
    return [(1 - (yy + zz)), (xy + wz), (xz - wy), 0.0, (xy - wz), (1 - (xx + zz)), (yz + wx), 0.0,
            (xz + wy), (yz - wx), (1 - (xx + yy)), 0.0, 0.0, 0.0, 0.0, 1.0]


def _determinant(te):
    n11, n12, n13, n14 = te[0], te[4], te[8], te[12]
    n21, n22, n23, n24 = te[1], te[5], te[9], te[13]
    n31, n32, n33, n34 = te[2], te[6], te[10], te[14]
    n41, n42, n43, n44 = te[3], te[7], te[11], te[15]
    return (n41 * (+n14 * n23 * n32 - n13 * n24 * n32 - n14 * n22 * n33 + n12 * n24 * n33 + n13 * n22 * n34 - n12 * n23 * n34)
            + n42 * (+n11 * n23 * n34 - n11 * n24 * n33 + n14 * n21 * n33 - n13 * n21 * n34 + n13 * n24 * n31 - n14 * n23 * n31)
            + n43 * (+n11 * n24 * n32 - n11 * n22 * n34 - n14 * n21 * n32 + n12 * n21 * n34 + n14 * n22 * n31 - n12 * n24 * n31)
            + n44 * (-n13 * n22 * n31 - n11 * n23 * n32 + n11 * n22 * n33 + n13 * n21 * n32 - n12 * n21 * n33 + n12 * n23 * n31))


def _quaternion_from_rotation(te):
    m11, m12, m13 = te[0], te[4], te[8]
    m21, m22, m23 = te[1], te[5], te[9]
    m31, m32, m33 = te[2], te[6], te[10]
    t = m11 + m22 + m33
    if t > 0:
        s = 0.5 / math.sqrt(t + 1.0)
        return (m32 - m23) * s, (m13 - m31) * s, (m21 - m12) * s, 0.25 / s
    if m11 > m22 and m11 > m33:
        s = 2.0 * math.sqrt(1.0 + m11 - m22 - m33)
        return 0.25 * s, (m12 + m21) / s, (m13 + m31) / s, (m32 - m23) / s
    if m22 > m33:
        s = 2.0 * math.sqrt(1.0 + m22 - m11 - m33)
        return (m12 + m21) / s, 0.25 * s, (m23 + m32) / s, (m13 - m31) / s
    s = 2.0 * math.sqrt(1.0 + m33 - m11 - m22)
    return (m13 + m31) / s, (m23 + m32) / s, 0.25 * s, (m21 - m12) / s


def scale_rotation_one(scale, quat_xyzw, transform_colmajor16=None, scale_z=1.0):
    """One splat -> [sx, sy, sz, qx, qy, qz] as Python floats (the caller stores them as f32)."""
    sx, sy, sz = float(scale[0]), float(scale[1]), float(scale_z)
    x, y, z, w = _normalize(*(float(v) for v in quat_xyzw))
    if transform_colmajor16 is not None:
        S = [sx, 0.0, 0.0, 0.0, 0.0, sy, 0.0, 0.0, 0.0, 0.0, sz, 0.0, 0.0, 0.0, 0.0, 1.0]
        I = [1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0]
        m = _mat4_mul(S, I)                                 # identity().premultiply(scaleMatrix)
        m = _mat4_mul(_rotation_from_quaternion(x, y, z, w), m)
        m = _mat4_mul([float(v) for v in transform_colmajor16], m)
        dsx = math.sqrt(m[0] * m[0] + m[1] * m[1] + m[2] * m[2])
        dsy = math.sqrt(m[4] * m[4] + m[5] * m[5] + m[6] * m[6])
        dsz = math.sqrt(m[8] * m[8] + m[9] * m[9] + m[10] * m[10])
        if _determinant(m) < 0:
            dsx = -dsx
        r = list(m)
        for k, inv in ((0, 1.0 / dsx), (4, 1.0 / dsy), (8, 1.0 / dsz)):
            r[k] *= inv; r[k + 1] *= inv; r[k + 2] *= inv
        x, y, z, w = _normalize(*_quaternion_from_rotation(r))
        sx, sy, sz = dsx, dsy, dsz
    flip = -1.0 if w < 0 else 1.0
    return [sx, sy, sz, x * flip, y * flip, z * flip]


def ksplat_scale_rotations(data: bytes, transform_colmajor16=None):
    """The TwoD scale/rotation texture of a `.ksplat` buffer: every splat's file scale and quaternion (decoded by oracle/ksplat_oracle.py)
    through scale_rotation_one, with the z scale override read at the file's compression level.  f32 [n, 6]."""
    import numpy as np
    from . import ksplat_oracle as KO
    d = KO.decode(data)
    sz = scale_z_override(d["header"].compression_level)
    t = None if transform_colmajor16 is None else [float(v) for v in np.asarray(transform_colmajor16, np.float64).reshape(16)]
    return np.array([scale_rotation_one(d["scales"][i], d["rotations"][i], t, sz) for i in range(d["count"])], np.float32).reshape(-1, 6)
