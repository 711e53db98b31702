"""CPU oracle of distortion, the inverse of Mode C -- TEST INFRASTRUCTURE ONLY, like lmc_oracle.py and lmc_oracle_local.py.
Only tests/ and the profiles may import it, as the checker; the product package never does.

* ``C.distort_slerp_f64`` -- ctypes binding of oracle/lmc_oracle_distort.c, the explicit-op-order definition.
* ``distort_slerp_scipy`` -- an independent restatement with SciPy ``Slerp`` + ``np.interp``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from .lmc_oracle_local import slerp_pose_scipy

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "lmc_oracle_distort.c")
_LIB_PATH = os.path.join(_HERE, "_build", "liblmc_oracle_distort.so")
# the flags of oracle/Makefile (explicit FMAs, no contraction)
_CFLAGS = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-mfma", "-Wall", "-Wextra"]


def build(force: bool = False) -> str:
    """Compile oracle/lmc_oracle_distort.c (gcc, no external deps) into oracle/_build/."""
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_LIB_PATH), exist_ok=True)
        tmp = _LIB_PATH + ".%d.tmp" % os.getpid()
        subprocess.run([os.environ.get("CC", "gcc")] + _CFLAGS + [_SRC, "-o", tmp, "-lm"], check=True)
        os.replace(tmp, _LIB_PATH)
    return _LIB_PATH


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        vp, i64 = ctypes.c_void_p, ctypes.c_int64
        L.orc_distort_slerp_f64.argtypes = [vp, vp, i64, vp, vp, i64, vp]
        L.orc_distort_slerp_f64.restype = None
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


class C:
    @staticmethod
    def distort_slerp_f64(pts, ts, sample_ts, seg):
        """Distortion: every world point (N, 4) at its int64 ns time into the sensor frame of Mode C's pose there."""
        pts, ts, sample_ts, seg = _c(pts, np.float64), _c(ts, np.int64), _c(sample_ts, np.int64), _c(seg, np.float64)
        out = np.empty_like(pts)
        lib().orc_distort_slerp_f64(_p(pts), _p(ts), len(pts), _p(sample_ts), _p(seg), len(sample_ts), _p(out))
        return out


def distort_slerp_scipy(pts, ts, sample_ts, sample_quat_xyzw, sample_pos):
    """Independent distortion: R(t)^-1 (W - x(t)), with R / x from slerp_pose_scipy at each point's time."""
    pts = np.asarray(pts, np.float64)
    out = pts.copy()
    if len(pts):
        Rt, x = slerp_pose_scipy(sample_ts, sample_quat_xyzw, sample_pos, ts)
        out[:, :3] = Rt.inv().apply(pts[:, :3] - x)
    return out
