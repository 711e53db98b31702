"""Prior point map, fixed-radius nearest neighbour and per-frame point-to-point Gauss-Newton registration: the definition
lmc_map_build / lmc_map_nearest_* / lmc_register_frames_* follow (include/lmc_b200.h), restated in NumPy.  Test
infrastructure only: the package never imports it.

Map: the voxel map's grid and keys (lmc_oracle_voxel.point_keys), rows sorted stably by voxel rank, CSR offsets.
Nearest of a query w: its cell k and the 27 cells k + {-1,0,1}^3 (each axis inside the key range); per candidate m
    d = w - m ;  d2 = (dx dx + dy dy) + dz dz     (every operation rounded to nearest: NumPy computes the device's bits)
accepted when d2 <= r2 = max_dist^2; the minimum over (d2, original index).  No match: index -1, d2 = +inf.
Register: per frame and iteration, a = R p with a_c = (R_c0 p0 + R_c1 p1) + R_c2 p2, w = a + t; over the inliers
r = w - q the 17 sums; H = [[n I, -[Sa]x], [[Sa]x, S|a|^2 I - S aa^T]], g = [Sr; S a x r]; [tau; phi] = -H^-1 g by
Cholesky; t += tau, R = Exp(phi) R.  n < 6 or a pivot <= 1e-12 trace(H): degenerate, pose kept.  |tau| <= tol_t and
|phi| <= tol_r: converged.  The sums here are NumPy's, not the device's order: poses agree to rounding, correspondences
of a given pose exactly."""
from __future__ import annotations

import numpy as np

from . import lmc_oracle_voxel as ov

CONVERGED, DEGENERATE = 1, 2


def build_map(pts, leaf, origin=(0.0, 0.0, 0.0)):
    """Returns dict(pts (M,4) f64 sorted by voxel, index int64[M], vox_off int64[V+1], keys int64[V] packed key by rank,
    leaf, origin).  ValueError / OverflowError for a point the voxel map drops."""
    p = np.asarray(pts).reshape(-1, 4)
    _, cnt, pv, flags = ov.voxel_downsample(p, leaf, origin)
    if flags & ov.FLAG_NAN:
        raise ValueError("map point with a NaN / inf value")
    if flags & ov.FLAG_OVERFLOW:
        raise OverflowError("map point outside the key or intensity range")
    order = np.argsort(pv, kind="stable").astype(np.int64)
    sp = p[order].astype(np.float64)
    off = np.zeros(len(cnt) + 1, np.int64)
    np.cumsum(cnt, out=off[1:])
    keys = ov.pack_keys(ov.point_keys(sp[off[:-1]], leaf, origin)[1]) if len(cnt) else np.zeros(0, np.int64)
    return dict(pts=sp, index=order, vox_off=off, keys=keys, leaf=ov.grid3(leaf, "leaf"), origin=ov.grid3(origin, "origin"))


def nearest(q, M, max_dist):
    """(index int64[N], d2 f64[N], flags) of every query row (N,3+) against map M (build_map)."""
    w = np.asarray(q)[:, :3].astype(np.float64)
    n = len(w)
    r2 = float(max_dist) * float(max_dist)
    finite = np.isfinite(w).all(axis=1)
    flags = ov.FLAG_NAN if (~finite).any() else 0
    w4 = np.zeros((n, 4))
    w4[:, :3] = w
    keep, k, _, _, _ = ov.point_keys(w4, M["leaf"], M["origin"])
    best_i = np.full(n, -1, np.int64)
    best_d = np.full(n, np.inf)
    qi = np.flatnonzero(keep)
    if len(qi) == 0 or len(M["keys"]) == 0:
        return best_i, best_d, flags
    sk = np.argsort(M["keys"])
    skeys = M["keys"][sk]
    cq, cj = [], []
    for dz in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                kk = k[qi] + np.array([dx, dy, dz])
                ok = ((kk >= -ov.KEY_LIM) & (kk < ov.KEY_LIM)).all(axis=1)
                key = ov.pack_keys(np.where(ok[:, None], kk, 0))
                pos = np.minimum(np.searchsorted(skeys, key), len(skeys) - 1)
                hit = ok & (skeys[pos] == key)
                r = sk[pos[hit]]
                a, b = M["vox_off"][r], M["vox_off"][r + 1]
                cnt = b - a
                cq.append(np.repeat(qi[hit], cnt))
                cj.append(np.repeat(a - (np.cumsum(cnt) - cnt), cnt) + np.arange(cnt.sum()))
    cq, cj = np.concatenate(cq), np.concatenate(cj)
    d = w[cq] - M["pts"][cj, :3]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    acc = d2 <= r2
    cq, cj, d2 = cq[acc], cj[acc], d2[acc]
    idx = M["index"][cj]
    o = np.lexsort((idx, d2, cq))
    first = o[np.r_[True, cq[o][1:] != cq[o][:-1]]] if len(o) else o
    best_i[cq[first]] = idx[first]
    best_d[cq[first]] = d2[first]
    return best_i, best_d, flags


def _skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def _exp(phi):
    th2 = float(phi @ phi)
    th = np.sqrt(th2)
    A = 1.0 - th2 / 6.0 if th < 1e-8 else np.sin(th) / th
    B = 0.5 - th2 / 24.0 if th < 1e-8 else (1.0 - np.cos(th)) / th2
    K = _skew(phi)
    return np.eye(3) + A * K + B * (K @ K)


def transform(p, pose):
    """a = R p and w = a + t of sensor points p (m,3+) under one (12,) pose row, with the device's rounding."""
    p = np.asarray(p)[:, :3].astype(np.float64)
    R, t = pose[:9].reshape(3, 3), pose[9:12]
    a = np.empty((len(p), 3))
    for r in range(3):
        a[:, r] = (R[r, 0] * p[:, 0] + R[r, 1] * p[:, 1]) + R[r, 2] * p[:, 2]
    return a, a + t


def register_frames(pts, frame_off, pose_Rt, M, max_dist, iters=30, tol_t=1e-9, tol_r=1e-12):
    """Returns (pose (F,12), inliers int32[F], rms_m f64[F], iterations int32[F], flags int32[F])."""
    pts = np.asarray(pts)
    off = np.asarray(frame_off, np.int64)
    pose = np.array(pose_Rt, np.float64).reshape(-1, 12)
    F = len(off) - 1
    inl, rms = np.zeros(F, np.int32), np.full(F, np.nan)
    its, fl = np.zeros(F, np.int32), np.zeros(F, np.int32)
    for f in range(F):
        p = pts[off[f]:off[f + 1]]
        for _ in range(iters):
            its[f] += 1
            a, w = transform(p, pose[f])
            j, _, _ = nearest(w, M, max_dist)
            ok = j >= 0
            n = int(ok.sum())
            inl[f] = n
            if n == 0:
                rms[f] = np.nan
                fl[f] = DEGENERATE
                break
            pos = np.empty(len(M["index"]), np.int64)
            pos[M["index"]] = np.arange(len(M["index"]))
            a = a[ok]
            r = w[ok] - M["pts"][pos[j[ok]], :3]
            rms[f] = np.sqrt(np.sum(r * r) / n)
            if n < 6:
                fl[f] = DEGENERATE
                break
            sa, A = a.sum(0), a.T @ a
            H = np.zeros((6, 6))
            H[:3, :3] = n * np.eye(3)
            H[:3, 3:] = -_skew(sa)
            H[3:, :3] = _skew(sa)
            H[3:, 3:] = np.trace(A) * np.eye(3) - A
            g = np.r_[r.sum(0), np.cross(a, r).sum(0)]
            L = np.zeros((6, 6))
            bad = False
            for jj in range(6):
                dd = H[jj, jj] - L[jj, :jj] @ L[jj, :jj]
                if not dd > 1e-12 * np.trace(H):
                    bad = True
                    break
                L[jj, jj] = np.sqrt(dd)
                L[jj + 1:, jj] = (H[jj + 1:, jj] - L[jj + 1:, :jj] @ L[jj, :jj]) / L[jj, jj]
            if bad:
                fl[f] = DEGENERATE
                break
            y = np.zeros(6)
            for i in range(6):
                y[i] = (-g[i] - L[i, :i] @ y[:i]) / L[i, i]
            x = np.zeros(6)
            for i in range(5, -1, -1):
                x[i] = (y[i] - L[i + 1:, i] @ x[i + 1:]) / L[i, i]
            R = _exp(x[3:]) @ pose[f, :9].reshape(3, 3)
            pose[f, :9] = R.reshape(9)
            pose[f, 9:12] += x[:3]
            if np.linalg.norm(x[:3]) <= tol_t and np.linalg.norm(x[3:]) <= tol_r:
                fl[f] = CONVERGED
                break
    return pose, inl, rms, its, fl
