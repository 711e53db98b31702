"""Map normals and point-to-plane registration: the definition lmc_map_normals / lmc_register_frames_plane_* follow
(include/lmc_b200.h), restated in NumPy on top of lmc_oracle_register (map, nearest, transform, update).  Test
infrastructure only: the package never imports it.

Normals of map row p: every map row m of the 27 cells around p with d2 <= r2 = radius^2 (the row itself included), in
the device's visit order (cells in dz, dy, dx order, rows in sorted order inside a cell); d = m - p; sequential sums
S d and S dd^T; mu = S d / n, C = S dd^T / n - mu mu^T; cyclic Jacobi (pairs (0,1), (0,2), (1,2), a rotation skipped
where its entry is exactly 0, until a sweep leaves every off-diagonal at 0, at most JACOBI_SWEEPS); eigenvalues sorted
ascending (ties in index order) and clamped at 0; (unit eigenvector of l_min with its largest-magnitude component
positive, (l_mid - l_min) / l_max), or (NaN, NaN, NaN, 0) for fewer than min_neighbours rows or l_max = 0.  Every
operation is an IEEE-rounded + - x / sqrt, so NumPy computes the device's bits.
Plane registration: register_frames with e = (nx rx + ny ry) + nz rz along the nearest map row's normal, inliers only
where that row's planarity >= min_planarity, J = [n; a x n], H = S J J^T, g = S J e.  The sums here are NumPy's, not
the device's order: poses agree to rounding, correspondences of a given pose exactly."""
from __future__ import annotations

import numpy as np

from . import lmc_oracle_voxel as ov
from .lmc_oracle_register import CONVERGED, DEGENERATE, _exp, nearest, transform

__all__ = ["CONVERGED", "DEGENERATE", "JACOBI_SWEEPS", "jacobi3", "normals", "register_frames_plane"]


JACOBI_SWEEPS = 32


def _ball_candidates(w, M):
    """(cq, cj): every (query row, sorted map row) pair of the 27 cells around each query, in the device's visit order
    (cells in dz, dy, dx order, rows in sorted order inside a cell) once stably sorted by cq."""
    n = len(w)
    w4 = np.zeros((n, 4))
    w4[:, :3] = w
    keep, k, _, _, _ = ov.point_keys(w4, M["leaf"], M["origin"])
    qi = np.flatnonzero(keep)
    sk = np.argsort(M["keys"])
    skeys = M["keys"][sk]
    cq, cj = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
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
    o = np.argsort(cq, kind="stable")
    return cq[o], cj[o]


def _jacobi_rotate(a, V, p, q, act):
    """One rotation of the pair (p, q) on the rows where act and a[:, p, q] != 0 (a (K,3,3) symmetric, V (K,3,3))."""
    apq = a[:, p, q]
    m = act & (apq != 0.0)
    r = 3 - p - q
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        th = (a[:, q, q] - a[:, p, p]) / (2.0 * apq)
        t = 1.0 / (np.abs(th) + np.sqrt(th * th + 1.0))
        t = np.where(th < 0.0, -t, t)
        c = 1.0 / np.sqrt(t * t + 1.0)
        s = t * c
        app, aqq = a[:, p, p] - t * apq, a[:, q, q] + t * apq
        arp, arq = a[:, r, p], a[:, r, q]
        nrp, nrq = c * arp - s * arq, s * arp + c * arq
        vp, vq = V[:, :, p], V[:, :, q]
        nvp, nvq = c[:, None] * vp - s[:, None] * vq, s[:, None] * vp + c[:, None] * vq
    a[:, p, p] = np.where(m, app, a[:, p, p])
    a[:, q, q] = np.where(m, aqq, a[:, q, q])
    a[:, p, q] = a[:, q, p] = np.where(m, 0.0, apq)
    a[:, r, p] = a[:, p, r] = np.where(m, nrp, arp)
    a[:, r, q] = a[:, q, r] = np.where(m, nrq, arq)
    V[:, :, p] = np.where(m[:, None], nvp, vp)
    V[:, :, q] = np.where(m[:, None], nvq, vq)


def jacobi3(C):
    """Cyclic Jacobi of symmetric (K,3,3) matrices: pairs (0,1), (0,2), (1,2), a rotation skipped where its entry is
    exactly 0, until a sweep leaves every off-diagonal at 0 (at most JACOBI_SWEEPS).  Returns (diagonal (K,3), V (K,3,3)
    with the eigenvectors in its columns)."""
    a = np.array(C, np.float64, copy=True)
    V = np.broadcast_to(np.eye(3), a.shape).copy()
    for _ in range(JACOBI_SWEEPS):
        act = (a[:, 0, 1] != 0.0) | (a[:, 0, 2] != 0.0) | (a[:, 1, 2] != 0.0)
        if not act.any():
            break
        for p, q in ((0, 1), (0, 2), (1, 2)):
            _jacobi_rotate(a, V, p, q, act)
    return np.stack([a[:, 0, 0], a[:, 1, 1], a[:, 2, 2]], 1), V


def normals(M, radius, min_neighbours=5):
    """Normals of map M (build_map) in its sorted row order: (normals (M,4) f64 (nx, ny, nz, planarity),
    neighbours int32[M]) -- lmc_map_normals' definition (include/lmc_b200.h), bit for bit."""
    P = M["pts"][:, :3]
    m = len(P)
    r2 = float(radius) * float(radius)
    out = np.zeros((m, 4))
    out[:, :3] = np.nan
    if m == 0:
        return out, np.zeros(0, np.int32)
    cq, cj = _ball_candidates(P, M)
    d = P[cj] - P[cq]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    acc = d2 <= r2
    cq, d = cq[acc], d[acc]
    cnt = np.bincount(cq, minlength=m)
    K = int(cnt.max())
    col = np.arange(len(cq)) - np.repeat(np.cumsum(cnt) - cnt, cnt)        # position inside the row's list
    D = np.zeros((m, K, 3))
    D[cq, col] = d
    valid = np.arange(K)[None, :] < cnt[:, None]
    sd, sdd = np.zeros((m, 3)), np.zeros((m, 6))
    pairs = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))
    for k in range(K):                                                     # sequential per row, in visit order
        dk, vk = D[:, k], valid[:, k]
        sd = np.where(vk[:, None], sd + dk, sd)
        prod = np.stack([dk[:, u] * dk[:, v] for u, v in pairs], 1)
        sdd = np.where(vk[:, None], sdd + prod, sdd)
    ok = cnt >= int(min_neighbours)
    dn = cnt[ok].astype(np.float64)[:, None]
    mu = sd[ok] / dn
    cov = sdd[ok] / dn - np.stack([mu[:, u] * mu[:, v] for u, v in pairs], 1)
    C = np.empty((len(cov), 3, 3))
    for j, (u, v) in enumerate(pairs):
        C[:, u, v] = C[:, v, u] = cov[:, j]
    lam, V = jacobi3(C)
    ix = np.argsort(lam, axis=1, kind="stable")
    ls = np.take_along_axis(lam, ix, 1)
    ls = np.where(ls > 0.0, ls, 0.0)                                       # (negatives and -0 to +0)
    nv = np.take_along_axis(V, ix[:, None, :1], 2)[:, :, 0]
    nr = np.sqrt((nv[:, 0] * nv[:, 0] + nv[:, 1] * nv[:, 1]) + nv[:, 2] * nv[:, 2])
    big = np.argmax(np.abs(nv), axis=1)                                    # (the first maximum on a tie)
    sg = np.where(nv[np.arange(len(nv)), big] < 0.0, -1.0, 1.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        row = np.c_[sg[:, None] * (nv / nr[:, None]), (ls[:, 1] - ls[:, 0]) / ls[:, 2]]
    good = ls[:, 2] != 0.0
    row[~good] = [np.nan, np.nan, np.nan, 0.0]
    out[ok] = row
    return out, cnt.astype(np.int32)


def register_frames_plane(pts, frame_off, pose_Rt, M, N, max_dist, min_planarity, iters=30, tol_t=1e-9, tol_r=1e-12):
    """Point-to-plane registration against map M with its normals N (normals()): register_frames with the residual
    e = (nx rx + ny ry) + nz rz along the nearest map row's normal, an inlier only where that row's planarity >=
    min_planarity, J = [n; a x n], H = S J J^T, g = S J e.  rms_m is the rms plane distance.
    Returns (pose (F,12), inliers int32[F], rms_m f64[F], iterations int32[F], flags int32[F])."""
    pts = np.asarray(pts)
    off = np.asarray(frame_off, np.int64)
    pose = np.array(pose_Rt, np.float64).reshape(-1, 12)
    F = len(off) - 1
    inl, rms = np.zeros(F, np.int32), np.full(F, np.nan)
    its, fl = np.zeros(F, np.int32), np.zeros(F, np.int32)
    pos = np.empty(len(M["index"]), np.int64)
    pos[M["index"]] = np.arange(len(M["index"]))
    for f in range(F):
        p = pts[off[f]:off[f + 1]]
        for _ in range(iters):
            its[f] += 1
            a, w = transform(p, pose[f])
            j, _, _ = nearest(w, M, max_dist)
            row = pos[np.maximum(j, 0)]
            ok = (j >= 0) & (N[row, 3] >= min_planarity)
            n = int(ok.sum())
            inl[f] = n
            if n == 0:
                rms[f] = np.nan
                fl[f] = DEGENERATE
                break
            a, nrm = a[ok], N[row[ok], :3]
            r = w[ok] - M["pts"][row[ok], :3]
            e = (nrm[:, 0] * r[:, 0] + nrm[:, 1] * r[:, 1]) + nrm[:, 2] * r[:, 2]
            rms[f] = np.sqrt(np.sum(e * e) / n)
            if n < 6:
                fl[f] = DEGENERATE
                break
            J = np.c_[nrm, np.cross(a, nrm)]
            H, g = J.T @ J, J.T @ e
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
