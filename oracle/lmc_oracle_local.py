"""CPU oracle of the pose at a time and of sensor-frame deskew -- TEST INFRASTRUCTURE ONLY, like lmc_oracle.py, whose Mode C
it extends.  Only tests/ and the profiles may import it, as the checker; the product package never does.

* ``C.*``  -- ctypes bindings of oracle/lmc_oracle_local.c, the explicit-op-order definition.
* ``slerp_pose_scipy`` / ``slerp_deskew_local_scipy`` -- an independent restatement with SciPy ``Slerp`` + ``np.interp``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
from scipy.spatial.transform import Rotation, Slerp

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "lmc_oracle_local.c")
_LIB_PATH = os.path.join(_HERE, "_build", "liblmc_oracle_local.so")
# the flags of oracle/Makefile (explicit FMAs, no contraction)
_CFLAGS = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-mfma", "-Wall", "-Wextra"]


def build(force: bool = False) -> str:
    """Compile oracle/lmc_oracle_local.c (gcc, no external deps) into oracle/_build/."""
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
        L.orc_slerp_pose_at.argtypes = [vp, vp, i64, vp, i64, vp]
        L.orc_slerp_pose_at.restype = None
        L.orc_deskew_slerp_local_f64.argtypes = [vp, vp, vp, i64, vp, vp, i64, vp, vp]
        L.orc_deskew_slerp_local_f64.restype = None
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


class C:
    @staticmethod
    def slerp_pose_at(sample_ts, seg, query_ts):
        """Mode C's pose at each query time (int64 ns) -> (n, 12) rows [R row-major | pos], Mode A's pose_Rt layout."""
        sample_ts, seg, query_ts = _c(sample_ts, np.int64), _c(seg, np.float64), _c(query_ts, np.int64)
        out = np.empty((len(query_ts), 12), np.float64)
        lib().orc_slerp_pose_at(_p(sample_ts), _p(seg), len(sample_ts), _p(query_ts), len(query_ts), _p(out))
        return out

    @staticmethod
    def deskew_slerp_local_f64(pts, ts, frame_off, sample_ts, seg, ref_pose):
        """Sensor-frame deskew: every point of frame f in the frame of ref_pose[f] ((F, 12), Mode A's layout)."""
        pts, ts = _c(pts, np.float64), _c(ts, np.int64)
        frame_off, sample_ts, seg, ref_pose = _c(frame_off, np.int64), _c(sample_ts, np.int64), _c(seg, np.float64), _c(ref_pose, np.float64)
        out = np.empty_like(pts)
        lib().orc_deskew_slerp_local_f64(_p(pts), _p(ts), _p(frame_off), len(frame_off) - 1, _p(sample_ts), _p(seg),
                                         len(sample_ts), _p(ref_pose), _p(out))
        return out


def slerp_pose_scipy(sample_ts, sample_quat_xyzw, sample_pos, query_ts):
    """Independent pose at a time: scipy Slerp for the rotation, np.interp for the position, both clamped to the
    sample span.  Returns (Rotation, (n, 3) positions)."""
    sample_ts = np.asarray(sample_ts, np.int64)
    t0 = sample_ts[0]
    tc = (np.clip(np.asarray(query_ts, np.int64), sample_ts[0], sample_ts[-1]) - t0).astype(np.float64)
    rot = Rotation.from_quat(sample_quat_xyzw)
    if len(sample_ts) == 1:
        return Rotation.from_quat(np.repeat(rot.as_quat().reshape(1, 4), len(tc), axis=0)), np.repeat(np.asarray(sample_pos, np.float64).reshape(1, 3), len(tc), axis=0)
    Rt = Slerp((sample_ts - t0).astype(np.float64), rot)(tc)
    pos = np.stack([np.interp(tc, (sample_ts - t0).astype(np.float64), np.asarray(sample_pos)[:, c]) for c in range(3)], axis=1)
    return Rt, pos


def slerp_deskew_local_scipy(pts, ts, frame_off, sample_ts, sample_quat_xyzw, sample_pos, ref_ts):
    """Independent sensor-frame deskew: R_ref^-1 (R(t) p + x(t) - x_ref), with R / x from slerp_pose_scipy at each point's
    time and at its frame's reference time ref_ts[f]."""
    pts = np.asarray(pts, np.float64)
    fidx = np.repeat(np.arange(len(frame_off) - 1), np.diff(np.asarray(frame_off, np.int64)))
    Rt, x = slerp_pose_scipy(sample_ts, sample_quat_xyzw, sample_pos, ts)
    Rr, xr = slerp_pose_scipy(sample_ts, sample_quat_xyzw, sample_pos, np.asarray(ref_ts, np.int64))
    out = pts.copy()
    if len(pts):
        out[:, :3] = Rr[fidx].inv().apply(Rt.apply(pts[:, :3]) + (x - xr[fidx]))
    return out