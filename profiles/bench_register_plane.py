"""Map normals and point-to-plane against point-to-point registration on one GPU (lmc_register.cu).

Workload: a planar map of --map-points f64 points on 4 x 4 m patches laid on a 10 m grid over 400 x 400 m (ground,
walls facing x and y, and panels tilted about two axes, mixed so that every 5 x 5 block of patches holds all five);
--frames frames of --ppf float4 sensor-frame points, each frame sampling the 25 patches of one 5 x 5 block at points
drawn independently of the map's samples, expressed in the frame of a true pose; each frame starts 3 cm / 0.01 rad off
that pose.  Leaf 1 m, normal radius 1 m, gate 1 m.  Timed with CUDA events (median of --reps after a warm-up):
  normals         ops.estimate_normals over every map row
  iteration       ops.register_frames with tol 0 at iters = 1 and --iters, the difference over iters - 1: one
                  iteration, for the plane metric (k_reg_accum_plane + k_reg_solve_plane) and the point metric
                  (k_reg_accum + k_reg_solve) on the same frames
  call            ops.register_frames with the default tolerances and 30 iterations, both metrics
plus converged counts and the median / max position and rotation error of both metrics.  The card's name, power limit
and SM clock are read in the same run."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from livox_motion_compensation_sim_b200 import ops  # noqa: E402
from profiles.bench_register import card, ev_ms, rot  # noqa: E402


def span(n):
    n = np.asarray(n, np.float64) / np.linalg.norm(n)
    u = np.cross(n, [0.0, 0.0, 1.0])
    u /= np.linalg.norm(u)
    return u, np.cross(n, u)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map-points", type=int, default=4_000_000)
    ap.add_argument("--frames", type=int, default=10_000)
    ap.add_argument("--ppf", type=int, default=10_000)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_register_plane needs a CUDA device")
    dev = torch.device("cuda:0")
    crd = card()
    f64 = dict(device=dev, dtype=torch.float64)
    g = torch.Generator(device=dev).manual_seed(2)
    ex, ey, ez = np.eye(3)
    kinds = [(ex, ey), (ey, ez), (ex, ez), span([1.0, -2.0, 3.0]), span([-3.0, 1.0, 2.0])]
    G = 40                                                                   # patches per axis, 10 m apart
    ii, jj = np.meshgrid(np.arange(G), np.arange(G), indexing="ij")
    kind = ((2 * ii + jj) % 5).reshape(-1)
    ctr = np.c_[10.0 * ii.reshape(-1) - 195.0, 10.0 * jj.reshape(-1) - 195.0, np.where(kind == 0, 0.0, 10.0)]
    U = torch.tensor(np.array([kinds[k][0] for k in kind]), **f64)
    V = torch.tensor(np.array([kinds[k][1] for k in kind]), **f64)
    C = torch.tensor(ctr, **f64)
    P = G * G
    per = a.map_points // P
    M = per * P

    def on_patch(pid):
        s = (torch.rand((len(pid), 2), generator=g, **f64) - 0.5) * 4.0
        return C[pid] + s[:, :1] * U[pid] + s[:, 1:] * V[pid]

    mp = torch.empty((M, 4), **f64)
    mp[:, :3] = on_patch(torch.arange(P, device=dev).repeat_interleave(per))
    mp[:, 3] = 0.5
    leaf, radius, gate = 1.0, 1.0, 1.0
    pm = ops.build_point_map(mp, leaf, (0.25, 0.25, 0.25))
    normals_ms, normals_reps = ev_ms(lambda: ops.estimate_normals(pm, radius), a.reps)
    normals, nb = ops.estimate_normals(pm, radius)
    valid = int(torch.isfinite(normals[:, 0]).sum().item())

    F, ppf = a.frames, a.ppf
    N = F * ppf
    bi = torch.randint(0, G - 4, (F,), generator=g, device=dev)
    bj = torch.randint(0, G - 4, (F,), generator=g, device=dev)
    fidx = torch.arange(F, device=dev).repeat_interleave(ppf)
    slot = torch.arange(N, device=dev) % 25                                 # the block's 25 patches, round robin
    pid = (bi[fidx] + slot // 5) * G + bj[fidx] + slot % 5
    world = on_patch(pid)
    del pid, slot
    t_true = torch.stack([10.0 * bi.double() - 175.0, 10.0 * bj.double() - 175.0, torch.full((F,), 2.0, **f64)], 1)
    t_true += (torch.rand((F, 3), generator=g, **f64) - 0.5) * torch.tensor([6.0, 6.0, 1.0], **f64)
    R_true = rot(torch.randn((F, 3), generator=g, **f64) * 0.3)
    pts = torch.empty((N, 4), dtype=torch.float32, device=dev)
    for s in range(0, N, 1 << 24):
        e = min(N, s + (1 << 24))
        pts[s:e, :3] = torch.einsum('nji,nj->ni', R_true[fidx[s:e]], world[s:e] - t_true[fidx[s:e]]).float()
    pts[:, 3] = 0.5
    del fidx, world
    off = torch.arange(0, N + 1, ppf, dtype=torch.int64, device=dev)
    dR = rot(torch.nn.functional.normalize(torch.randn((F, 3), generator=g, **f64), dim=1) * 0.01)
    init = torch.empty((F, 12), **f64)
    init[:, :9] = (dR @ R_true).reshape(F, 9)
    init[:, 9:] = t_true + 0.03 * torch.nn.functional.normalize(torch.randn((F, 3), generator=g, **f64), dim=1)

    plane = dict(normals=normals)
    res = {}
    for name, kw in (("plane", plane), ("point", {})):
        it1, _ = ev_ms(lambda: ops.register_frames(pts, off, init, pm, gate, iters=1, tol_t=0.0, tol_r=0.0, **kw), a.reps)
        itk, itk_reps = ev_ms(lambda: ops.register_frames(pts, off, init, pm, gate, iters=a.iters, tol_t=0.0, tol_r=0.0, **kw), a.reps)
        full, full_reps = ev_ms(lambda: ops.register_frames(pts, off, init, pm, gate, iters=30, **kw), a.reps)
        pose, st = ops.register_frames(pts, off, init, pm, gate, iters=30, **kw)
        terr = torch.linalg.vector_norm(pose[:, 9:] - t_true, dim=1)
        Rd = pose[:, :9].reshape(F, 3, 3) @ R_true.transpose(1, 2)
        rerr = torch.asin((torch.linalg.vector_norm(torch.stack([Rd[:, 2, 1] - Rd[:, 1, 2], Rd[:, 0, 2] - Rd[:, 2, 0],
                                                                 Rd[:, 1, 0] - Rd[:, 0, 1]], 1), dim=1) / 2.0).clamp(max=1.0))
        res[name] = {
            "iters1_ms": it1, f"iters{a.iters}_ms": itk, f"iters{a.iters}_ms_reps": itk_reps,
            "ms_per_iteration": (itk - it1) / (a.iters - 1), "gpoints_s_per_iteration": N / ((itk - it1) / (a.iters - 1)) / 1e6,
            "call_30_default_tol_ms": full, "call_30_default_tol_ms_reps": full_reps,
            "converged": int(st.converged.sum().item()), "degenerate": int(st.degenerate.sum().item()),
            "iterations_median": float(st.iterations.double().median().item()), "iterations_max": int(st.iterations.max().item()),
            "position_error_m": {"median": float(terr.median().item()), "max": float(terr.max().item())},
            "rotation_error_rad": {"median": float(rerr.median().item()), "max": float(rerr.max().item())},
        }
    line = {
        "card": crd,
        "workload": (f"planar map {M} f64 points on {P} 4x4 m patches over 400x400 m, leaf 1 m, normal radius 1 m, gate 1 m; "
                     f"{F} frames x {ppf} float4 points = {N} queries, scan samples independent of the map's"),
        "map_points": M, "n_voxels": pm.n_voxels, "queries": N, "frames": F,
        "estimate_normals_ms": normals_ms, "estimate_normals_ms_reps": normals_reps, "normals_valid_rows": valid,
        "normals_neighbours_median": float(nb.double().median().item()),
        "plane": res["plane"], "point": res["point"],
    }
    text = json.dumps(line, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
