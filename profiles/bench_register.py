"""Point-map build, fixed-radius nearest-neighbour queries and per-frame pose refinement on one GPU (lmc_register.cu).

Workload: a prior map of --map-points points spread over a 400 x 400 x 40 m block (about one point per 1.6 m^3, so a
1 m cell holds a few points, the density of the C3 environment's map at a 1 m leaf), and --frames frames of
--ppf float4 sensor-frame points each, drawn from the map rows plus 2 cm of noise and expressed in the frame of a
true pose; each frame starts 3 cm / 0.01 rad off that pose.  Gate 1 m on a 1 m leaf.  Timed with CUDA events
(median of --reps after a warm-up):
  build           ops.build_point_map (voxel index + reduce, stable sort, k_map_insert)
  map_nearest     ops.map_nearest over every sensor point taken as a world query (queries per second)
  register        ops.register_frames with tol 0 (every frame runs every iteration) at iters = 1 and --iters; the
                  difference over iters - 1 is the time of one iteration (k_reg_accum + k_reg_solve)
The algorithmic bytes per query: 16 B point in + 16 B out (index, d2) for map_nearest; 16 B point in for an
iteration; the map rows each query reads (27 lookups and the candidates' 32 B rows) come from L2 for a map of this
size.  The card's name, power limit and SM clock are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from livox_motion_compensation_sim_b200 import ops  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def ev_ms(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), ts


def rot(v):
    """(F,3) rotation vectors -> (F,3,3) matrices (Rodrigues, f64)."""
    th = torch.linalg.vector_norm(v, dim=1).clamp_min(1e-300)[:, None, None]
    k = v / th[:, :, 0]
    K = torch.zeros((v.shape[0], 3, 3), dtype=v.dtype, device=v.device)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -k[:, 2], k[:, 1], -k[:, 0]
    K = K - K.transpose(1, 2)
    I = torch.eye(3, dtype=v.dtype, device=v.device).expand_as(K)
    return I + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


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
        raise SystemExit("bench_register needs a CUDA device")
    dev = torch.device("cuda:0")
    crd = card()
    g = torch.Generator(device=dev).manual_seed(1)
    M, F, ppf = a.map_points, a.frames, a.ppf
    N = F * ppf
    mp = torch.empty((M, 4), dtype=torch.float64, device=dev)
    mp[:, :3] = (torch.rand((M, 3), generator=g, device=dev, dtype=torch.float64) - 0.5) * torch.tensor([400.0, 400.0, 40.0], device=dev, dtype=torch.float64)
    mp[:, 3] = 0.5
    leaf, origin = 1.0, (0.0, 0.0, 0.0)
    build_ms, build_reps = ev_ms(lambda: ops.build_point_map(mp, leaf, origin), a.reps)
    pm = ops.build_point_map(mp, leaf, origin)

    # frames: true pose (R_f, t_f); sensor points p = R_f^T (m + noise - t_f), as float4
    t_true = (torch.rand((F, 3), generator=g, device=dev, dtype=torch.float64) - 0.5) * torch.tensor([300.0, 300.0, 10.0], device=dev, dtype=torch.float64)
    R_true = rot(torch.randn((F, 3), generator=g, device=dev, dtype=torch.float64) * 0.5)
    rows = torch.randint(0, M, (N,), generator=g, device=dev)
    fidx = torch.arange(F, device=dev).repeat_interleave(ppf)
    world = mp[rows, :3] + 0.02 * torch.randn((N, 3), generator=g, device=dev, dtype=torch.float64)
    del rows
    pts = torch.empty((N, 4), dtype=torch.float32, device=dev)
    for s in range(0, N, 1 << 24):                                          # (chunked: the (n,3,3) gather is large)
        e = min(N, s + (1 << 24))
        pts[s:e, :3] = torch.einsum('nji,nj->ni', R_true[fidx[s:e]], world[s:e] - t_true[fidx[s:e]]).float()
    pts[:, 3] = 0.5
    del fidx
    off = torch.arange(0, N + 1, ppf, dtype=torch.int64, device=dev)
    dR = rot(torch.nn.functional.normalize(torch.randn((F, 3), generator=g, device=dev, dtype=torch.float64), dim=1) * 0.01)
    init = torch.empty((F, 12), dtype=torch.float64, device=dev)
    init[:, :9] = (dR @ R_true).reshape(F, 9)
    init[:, 9:] = t_true + 0.03 * torch.nn.functional.normalize(torch.randn((F, 3), generator=g, device=dev, dtype=torch.float64), dim=1)

    wq = world.float()
    wq = torch.cat([wq, torch.full((N, 1), 0.5, device=dev)], 1).contiguous()
    del world
    nn_ms, nn_reps = ev_ms(lambda: ops.map_nearest(wq, pm, 1.0), a.reps)
    idx, d2, st = ops.map_nearest(wq, pm, 1.0)
    matched = int((idx >= 0).sum().item())
    del wq, idx, d2

    reg1_ms, _ = ev_ms(lambda: ops.register_frames(pts, off, init, pm, 1.0, iters=1, tol_t=0.0, tol_r=0.0), a.reps)
    regk_ms, regk_reps = ev_ms(lambda: ops.register_frames(pts, off, init, pm, 1.0, iters=a.iters, tol_t=0.0, tol_r=0.0), a.reps)
    full_ms, _ = ev_ms(lambda: ops.register_frames(pts, off, init, pm, 1.0, iters=30), a.reps)
    pose, rs = ops.register_frames(pts, off, init, pm, 1.0, iters=30)
    terr = torch.linalg.vector_norm(pose[:, 9:] - t_true, dim=1)
    per_iter = (regk_ms - reg1_ms) / (a.iters - 1)
    line = {
        "card": crd,
        "workload": f"map {M} f64 points over 400x400x40 m, leaf 1 m, gate 1 m; {F} frames x {ppf} float4 points = {N} queries",
        "map_points": M, "n_voxels": pm.n_voxels, "queries": N, "frames": F,
        "build_point_map_ms": build_ms, "build_point_map_ms_reps": build_reps,
        "map_nearest_ms": nn_ms, "map_nearest_ms_reps": nn_reps, "map_nearest_gqueries_s": N / nn_ms / 1e6,
        "map_nearest_matched": matched, "map_nearest_algorithmic_bytes": N * 32,
        "map_nearest_algorithmic_tb_s": N * 32 / nn_ms / 1e9,
        "register_iters1_ms": reg1_ms, f"register_iters{a.iters}_ms": regk_ms, f"register_iters{a.iters}_ms_reps": regk_reps,
        "register_ms_per_iteration": per_iter, "register_gpoints_s_per_iteration": N / per_iter / 1e6,
        "register_iteration_algorithmic_bytes": N * 16 + F * (12 * 8 * 2),
        "register_frames_30_default_tol_ms": full_ms,
        "register_30_converged": int(rs.converged.sum().item()), "register_30_degenerate": int(rs.degenerate.sum().item()),
        "register_30_iterations_max": int(rs.iterations.max().item()),
        "register_30_position_error_m": {"median": float(terr.median().item()), "max": float(terr.max().item())},
    }
    text = json.dumps(line, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
