"""Voxel-grid map of the M-1H aligned cloud (bench.py's stream: 36 000 frames x 10 000 points, float4, deskewed by Mode C),
at leaves 0.1 / 0.5 / 2.0 m on the grid anchored at the first pose sample.

    python profiles/bench_voxel.py [--iters 5] [--out FILE] [--frames F --ppf P]

Per leaf:
  call      ops.voxel_downsample: both C calls and the host read of V, CUDA events, median of --iters
  index / reduce   the two C calls alone, CUDA events
  kernels   per-kernel device time from torch.profiler (CUDA activities), one profiled call in its own pass
  torch     the plain-torch composition (keys in f64, torch.unique(return_inverse, return_counts) + index_add_), CUDA events
Points per second, V, and the algorithmic bytes of each pass (computed from N, V and the table size).  Context: the NumPy
oracle's host rate on a 1e7-point sample.  The card's name, power limit and SM clock are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from livox_motion_compensation_sim_b200 import _capi as C, ops, synth  # noqa: E402
from oracle import lmc_oracle_voxel as ov  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def pass_bytes(N, V, cap):
    """Bytes each pass needs at minimum (float4 input, no point_voxel)."""
    return {"memset_table": 12 * cap,
            "k_voxel_insert": N * (16 + 4 + 8 + 4),          # point, slot out, key CAS / read, first-index atomicMin
            "k_voxel_count": N * (4 + 4),                    # slot, first index
            "k_voxel_rank": N * (4 + 4) + V * (4 + 8 + 8),   # + rank, key read, key by rank
            "memset_acc": 40 * V,
            "k_voxel_accum": N * (16 + 4 + 4 + 40),          # point, slot, rank, five u64 reductions
            "k_voxel_finalize": V * (40 + 8 + 16 + 4)}


def torch_composition(pts, leaf, origin):
    o = torch.tensor(origin, dtype=torch.float64, device=pts.device)
    k = torch.floor((pts[:, :3].double() - o) / leaf).long() + (1 << 20)
    key = k[:, 0] | (k[:, 1] << 21) | (k[:, 2] << 42)
    del k
    uniq, inv, cnt = torch.unique(key, return_inverse=True, return_counts=True)
    s = torch.zeros((uniq.shape[0], 4), dtype=torch.float64, device=pts.device).index_add_(0, inv, pts.double())
    return s / cnt[:, None], cnt


def ev_ms(fn, iters, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--frames", type=int, default=bench.N_FRAMES)
    ap.add_argument("--ppf", type=int, default=bench.PTS_PER_FRAME)
    ap.add_argument("--leaves", default="0.1,0.5,2.0")
    ap.add_argument("--no-torch", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    crd = card()
    st = synth.make_stream(a.frames, a.ppf, bench.SEED, device=dev, dtype=torch.float32)
    N = st.n_points
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)   # noqa: E731
    pts, _ = ops.deskew_slerp(st.pts, st.ts_off, d(st.frame_off), d(st.frame_start), d(st.sample_ts), d(st.seg))
    st.pts = None
    origin = tuple(float(v) for v in st.seg[0, 9:12])
    lib = C.lib()
    ws = torch.empty(int(lib.lmc_voxel_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    cap = 64
    while cap < 2 * N:
        cap *= 2
    nv = torch.empty(1, dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = lambda: torch.cuda.current_stream().cuda_stream          # noqa: E731
    res = {}
    for leaf in [float(x) for x in a.leaves.split(",")]:
        L3, O3 = (C.ctypes.c_double * 3)(leaf, leaf, leaf), (C.ctypes.c_double * 3)(*origin)
        call_ms, call_reps = ev_ms(lambda: ops.voxel_downsample(pts, leaf, origin), a.iters)
        cent, cnt, _, stt = ops.voxel_downsample(pts, leaf, origin)
        V = cnt.shape[0]
        out = torch.empty((V, 4), dtype=torch.float32, device=dev)
        counts = torch.empty(V, dtype=torch.int32, device=dev)
        idx_ms, _ = ev_ms(lambda: C.check(lib.lmc_voxel_index_f32(pts.data_ptr(), N, L3, O3, ws.data_ptr(), nv.data_ptr(),
                                                                  status.data_ptr(), stream())), a.iters)
        red_ms, _ = ev_ms(lambda: C.check(lib.lmc_voxel_reduce_f32(pts.data_ptr(), N, L3, O3, ws.data_ptr(), V, out.data_ptr(),
                                                                   counts.data_ptr(), None, stream())), a.iters)
        assert out.cpu().numpy().tobytes() == cent.cpu().numpy().tobytes()
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ops.voxel_downsample(pts, leaf, origin)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if "voxel" in ev.key or "scan" in ev.key or "Memset" in ev.key or "Memcpy" in ev.key:
                kern[ev.key] = round(getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3, 4)   # ms
        pb = pass_bytes(N, V, cap)
        r = {"V": V, "status": int(stt.item()), "call_ms": call_ms, "call_ms_reps": call_reps, "index_ms": idx_ms, "reduce_ms": red_ms,
             "gpts_s": N / (call_ms * 1e-3) / 1e9, "kernel_ms": kern, "pass_bytes": pb,
             "pass_bytes_total": sum(pb.values()), "algorithmic_tb_s": sum(pb.values()) / (call_ms * 1e-3) / 1e12}
        del cent, cnt, out, counts
        if not a.no_torch:
            try:
                t_ms, _ = ev_ms(lambda: torch_composition(pts, leaf, origin), max(1, a.iters // 2))
                r["torch_unique_ms"] = t_ms
                r["torch_unique_gpts_s"] = N / (t_ms * 1e-3) / 1e9
            except torch.OutOfMemoryError as e:
                r["torch_unique_ms"] = f"out of memory: {str(e)[:120]}"
            torch.cuda.empty_cache()
        res[str(leaf)] = r
        print(json.dumps({leaf: {k: v for k, v in r.items() if k not in ("kernel_ms", "pass_bytes", "call_ms_reps")}}), flush=True)
    sub = pts[:10_000_000].cpu().numpy()
    t0 = time.perf_counter()
    ov.voxel_downsample(sub, 0.5, origin)
    host_s = time.perf_counter() - t0
    line = {"card": crd, "workload": bench.workload_name(a.frames, a.ppf) + ", aligned by deskew_slerp (float4)",
            "n_points": N, "table_slots": cap, "workspace_bytes": ws.numel(), "origin": origin, "iters": a.iters,
            "numpy_oracle_1e7_pts": {"s": host_s, "mpts_s": 1e7 / host_s / 1e6}, "results": res}
    text = json.dumps(line, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
