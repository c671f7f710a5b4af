"""ctypes wrapper of oracle/surfel_oracle.c, the C restatement of the TwoD (surfel) material.  TEST INFRASTRUCTURE ONLY.

Built with the same flags as libgs_oracle.so (f32, no FMA contraction, OpenMP where the compiler has it) into oracle/ by
__graft_entry__.build(); where that directory is read-only and the library is missing it is built into a temporary directory."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from .pyoracle import N

HERE = Path(__file__).resolve().parent
SRC = HERE / "surfel_oracle.c"
LIB = HERE / "libgs_surfel_oracle.so"


def build(out: Path = LIB) -> Path:
    if out.exists() and out.stat().st_mtime >= SRC.stat().st_mtime:
        return out
    cmd = ["/usr/bin/gcc", "-std=c11", "-O2", "-fwrapv", "-ffp-contract=off", "-fPIC", "-shared", str(SRC), "-o", str(out), "-lm"]
    res = subprocess.run(cmd[:-3] + ["-fopenmp"] + cmd[-3:], capture_output=True, text=True)
    if res.returncode != 0:
        res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("surfel oracle build failed:\n" + res.stdout + res.stderr)
    return out


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        try:
            path = build()
        except (OSError, RuntimeError):
            path = build(Path(tempfile.mkdtemp(prefix="gs_surfel_oracle_")) / LIB.name)
        _lib = C.CDLL(str(path))
        _lib.gso_project_2d.restype = None
        _lib.gso_project_2d.argtypes = [C.c_void_p] * 3
        _lib.gso_blend_2d.restype = None
        _lib.gso_blend_2d.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        _lib.gso_blend_2d_crop.restype = None
        _lib.gso_blend_2d_crop.argtypes = [C.c_void_p, C.c_void_p] + [C.c_uint32] * 7 + [C.c_void_p]
    return _lib


def project_2d(uniforms, centers_colors, scale_rotations, sh=None, sh_degree=0, scene_indexes=None) -> np.ndarray:
    """Vertex stage of the TwoD material for every splat (gso_project_2d): N.PROJECTED_SURFEL_DTYPE records."""
    from .pyoracle import _splat_data
    cc = np.ascontiguousarray(centers_colors, dtype=np.uint32).reshape(-1, 4)
    d, keep = _splat_data(cc, np.zeros((cc.shape[0], 6), np.float32), sh, sh_degree, scene_indexes)
    sr = np.ascontiguousarray(scale_rotations, dtype=np.float32).reshape(-1, 6)
    d.scale_rotations = sr.ctypes.data
    u = uniforms.to_c()
    out = np.empty(d.count, N.PROJECTED_SURFEL_DTYPE)
    lib().gso_project_2d(C.addressof(u), C.addressof(d), out.ctypes.data)
    del keep
    return out


def blend_2d(projected: np.ndarray, order: np.ndarray, width: int, height: int) -> np.ndarray:
    """Fragment stage + NormalBlending in draw order; float RGBA, rows bottom-up."""
    ps = np.ascontiguousarray(projected)
    o = np.ascontiguousarray(order, dtype=np.uint32)
    frame = np.empty((height, width, 4), np.float32)
    lib().gso_blend_2d(ps.ctypes.data, o.ctypes.data, o.shape[0], width, height, frame.ctypes.data)
    return frame


def blend_2d_crop(projected: np.ndarray, order: np.ndarray, width: int, height: int, x0: int, y0: int, w: int, h: int) -> np.ndarray:
    ps = np.ascontiguousarray(projected)
    o = np.ascontiguousarray(order, dtype=np.uint32)
    frame = np.empty((h, w, 4), np.float32)
    lib().gso_blend_2d_crop(ps.ctypes.data, o.ctypes.data, o.shape[0], width, height, x0, y0, w, h, frame.ctypes.data)
    return frame


def render_2d(uniforms, centers_colors, scale_rotations, order, width, height, sh=None, sh_degree=0, scene_indexes=None):
    ps = project_2d(uniforms, centers_colors, scale_rotations, sh, sh_degree, scene_indexes)
    return blend_2d(ps, order, width, height), ps
