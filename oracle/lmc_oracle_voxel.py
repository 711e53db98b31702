"""Voxel-grid map of an (N,4) cloud [x y z intensity]: the definition lmc_voxel_index_* / lmc_voxel_reduce_* reproduce bit
for bit (include/lmc_b200.h), restated in vectorised NumPy.  Test infrastructure only: the package never imports it.

Per point and axis c, in IEEE f64 (f32 points widened exactly):
    u_c = (p_c - o_c) / L_c ;  k_c = floor(u_c) in [-2^20, 2^20) ;  q_c = min(trunc((u_c - k_c) 2^32), 2^32 - 1)
    q_I = rint(I 2^24) for |I| < 256   (round half to even)
A non-finite value drops the point with FLAG_NAN; otherwise a key out of range or |I| >= 256 drops it with FLAG_OVERFLOW.
Per voxel (n points, exact int64 sums S_c, S_I):
    centroid_c = o_c + (k_c + (f64(S_c) / n) 2^-32) L_c ;  intensity = (f64(S_I) / n) 2^-24
every operation rounded to nearest; the f32 layout rounds the f64 result once.  Voxels are ranked by their first point."""
from __future__ import annotations

import numpy as np

FLAG_NAN, FLAG_OVERFLOW = 1, 2
KEY_LIM = 1 << 20


def grid3(v, name):
    """A leaf or origin as three f64 values (a scalar is broadcast)."""
    a = np.broadcast_to(np.asarray(v, np.float64), (3,)).copy()
    if not np.isfinite(a).all():
        raise ValueError(f"{name} must be finite")
    return a


def point_keys(pts, leaf, origin=(0.0, 0.0, 0.0)):
    """Per point: (keep bool[N], k int64[N,3], q int64[N,3], q_I int64[N], flags).  k, q, q_I are 0 for a dropped point."""
    p = np.asarray(pts).reshape(-1, 4).astype(np.float64)
    L, o = grid3(leaf, "leaf"), grid3(origin, "origin")
    finite = np.isfinite(p).all(axis=1)
    with np.errstate(all="ignore"):
        u = (p[:, :3] - o) / L
        k = np.floor(u)
        inrange = ((k >= -KEY_LIM) & (k < KEY_LIM)).all(axis=1) & (np.abs(p[:, 3]) < 256.0)
        keep = finite & inrange
        q = np.minimum(np.trunc((u - k) * 2.0 ** 32), 2.0 ** 32 - 1)
        qi = np.rint(p[:, 3] * 2.0 ** 24)
    flags = (FLAG_NAN if (~finite).any() else 0) | (FLAG_OVERFLOW if (finite & ~inrange).any() else 0)
    k = np.where(keep[:, None], k, 0).astype(np.int64)
    q = np.where(keep[:, None], q, 0).astype(np.int64)
    qi = np.where(keep, qi, 0).astype(np.int64)
    return keep, k, q, qi, flags


def pack_keys(k):
    """The 63-bit key of lmc_voxel.cu: 21 bits per axis, k_c + 2^20."""
    kk = (np.asarray(k, np.int64) + KEY_LIM).astype(np.uint64)
    return (kk[:, 0] | (kk[:, 1] << np.uint64(21)) | (kk[:, 2] << np.uint64(42))).astype(np.int64)


def centroids(k_vox, S, SI, n, leaf, origin, f32):
    """(V,4) centroids from the voxel keys (V,3), the int64 sums (V,3), (V) and the counts (V)."""
    L, o = grid3(leaf, "leaf"), grid3(origin, "origin")
    nf = np.asarray(n, np.int64).astype(np.float64)
    out = np.empty((len(nf), 4), np.float64)
    out[:, :3] = o + (np.asarray(k_vox, np.int64).astype(np.float64) + (np.asarray(S, np.int64).astype(np.float64) / nf[:, None]) * 2.0 ** -32) * L
    out[:, 3] = (np.asarray(SI, np.int64).astype(np.float64) / nf) * 2.0 ** -24
    return out.astype(np.float32) if f32 else out


def voxel_downsample(pts, leaf, origin=(0.0, 0.0, 0.0)):
    """Returns (centroids (V,4) in the input's dtype, counts int32[V], point_voxel int32[N], flags)."""
    pts = np.asarray(pts)
    f32 = pts.dtype == np.float32
    keep, k, q, qi, flags = point_keys(pts, leaf, origin)
    n = len(keep)
    pv = np.full(n, -1, np.int32)
    idx = np.flatnonzero(keep)
    if len(idx) == 0:
        return np.zeros((0, 4), np.float32 if f32 else np.float64), np.zeros(0, np.int32), pv, flags
    _, first, inv = np.unique(pack_keys(k[idx]), return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")                  # voxels by their first point
    rank_of = np.empty(len(first), np.int64)
    rank_of[order] = np.arange(len(first))
    r = rank_of[inv.reshape(-1)]
    pv[idx] = r
    s = np.argsort(r, kind="stable")
    starts = np.flatnonzero(np.r_[True, r[s][1:] != r[s][:-1]])
    S = np.add.reduceat(q[idx][s], starts, axis=0)
    SI = np.add.reduceat(qi[idx][s], starts)
    cnt = np.diff(np.r_[starts, len(s)])
    k_vox = k[idx][s][starts]
    return centroids(k_vox, S, SI, cnt, leaf, origin, f32), cnt.astype(np.int32), pv, flags
