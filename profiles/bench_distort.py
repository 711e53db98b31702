"""Distortion on the M-1H stream (bench.py's workload: 36 000 frames x 10 000 points, float4 + u32 offsets, 200 Hz pose
table of f64 rows, inputs >> L2), against Mode C and sensor-frame deskew on the same stream.

    python profiles/bench_distort.py [--reps 3] [--iters 20] [--out FILE] [--ab-lib OTHER/liblmc_b200.so]

Timed with CUDA events, each variant warmed up, the variants alternated --reps times; the median over the reps is reported:
  VD    distort_slerp, raw cloud only                                36 B/pt (16 in + 4 ts + 16 out)
  V4    deskew_slerp (Mode C), aligned cloud only                    36 B/pt
  V4L   deskew_slerp_local, aligned cloud only                       36 B/pt
Gpts/s, TB/s of the bytes each variant moves, and the fraction of bench.measured_peak() for them.
--ab-lib: a second build of the same ABI (e.g. the parent commit's) whose V4 / V5 / V4L kernels are timed alternately with
this tree's, through the same raw C calls.  The card's name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from livox_motion_compensation_sim_b200 import _capi as C, ops, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or q.stderr.strip()


def load_other(path):
    L = ctypes.CDLL(os.path.abspath(path))
    for name in ("lmc_deskew_slerp_f32", "lmc_deskew_slerp_local_f32", "lmc_last_error"):
        args, res = C._SIGNATURES[name]
        getattr(L, name).argtypes, getattr(L, name).restype = args, res
    return L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=bench.N_FRAMES)
    ap.add_argument("--ppf", type=int, default=bench.PTS_PER_FRAME)
    ap.add_argument("--out", default=None)
    ap.add_argument("--ab-lib", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    st = synth.make_stream(a.frames, a.ppf, bench.SEED, device=dev, dtype=torch.float32)
    N = st.n_points
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)   # noqa: E731
    off, fs, sts, seg = d(st.frame_off), d(st.frame_start), d(st.sample_ts), d(st.seg)
    pts, ts = st.pts, st.ts_off
    ref_ts = st.frame_start + (np.diff(st.frame_off) - 1) * 10_000       # sensor-frame deskew: the frame's end
    ref = ops.slerp_pose_at(sts, seg, d(ref_ts))
    out = torch.empty_like(pts)
    lvx = ops.ExportBuffers(lvx14=torch.empty((N, 14), dtype=torch.uint8, device=dev), status=torch.zeros(1, dtype=torch.int32, device=dev))

    runs = {
        "VD": (36, lambda: ops.distort_slerp(pts, ts, off, fs, sts, seg, out=out)),
        "V4": (36, lambda: ops.deskew_slerp(pts, ts, off, fs, sts, seg, out=out)),
        "V4L": (36, lambda: ops.deskew_slerp_local(pts, ts, off, fs, sts, seg, ref, out=out)),
    }
    if a.ab_lib:
        # V4 / V5 / V4L of this tree and of the other build, through the same raw calls
        libs = {"this": C.lib(), "other": load_other(a.ab_lib)}
        ex = C.LmcExport()
        ex.lvx14, ex.lvx_mode, ex.status = lvx.lvx14.data_ptr(), C.LVX_TYPE2_OF_INPUT, lvx.status.data_ptr()
        for k in range(3):
            ex.las_scale[k] = 0.01
        F = st.n_frames
        stream = lambda: torch.cuda.current_stream().cuda_stream        # noqa: E731

        def raw(L, with_lvx):
            def fn():
                C.check(L.lmc_deskew_slerp_f32(pts.data_ptr(), ts.data_ptr(), off.data_ptr(), fs.data_ptr(), sts.data_ptr(), seg.data_ptr(),
                                               len(st.sample_ts), None, out.data_ptr(), N, F, 0, N,
                                               ctypes.byref(ex) if with_lvx else None, stream()))
            return fn

        def raw_local(L):
            def fn():
                C.check(L.lmc_deskew_slerp_local_f32(pts.data_ptr(), ts.data_ptr(), off.data_ptr(), fs.data_ptr(), sts.data_ptr(),
                                                     seg.data_ptr(), len(st.sample_ts), ref.data_ptr(), out.data_ptr(), N, F, 0, N,
                                                     None, stream()))
            return fn
        for who, L in libs.items():
            runs[f"V4[{who}]"] = (36, raw(L, False))
            runs[f"V5[{who}]"] = (50, raw(L, True))
            runs[f"V4L[{who}]"] = (36, raw_local(L))

    def time_ms(fn):
        for _ in range(a.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.iters

    samples = {k: [] for k in runs}
    for _ in range(a.reps):
        for k, (_, fn) in runs.items():
            samples[k].append(time_ms(fn))
    peak_gbs, peak_src = bench.measured_peak()
    res = {}
    for k, (bpp, _) in runs.items():
        ms = float(np.median(samples[k]))
        tbs = N * bpp / (ms * 1e-3) / 1e12
        res[k] = {"ms": ms, "ms_reps": samples[k], "gpts_s": N / (ms * 1e-3) / 1e9, "bytes_per_pt": bpp, "tb_s": tbs,
                  "frac_of_peak": tbs * 1e3 / peak_gbs}
    line = {"card": card(), "workload": bench.workload_name(a.frames, a.ppf), "n_points": N, "iters": a.iters, "reps": a.reps,
            "peak_gbs": peak_gbs, "peak_source": peak_src, "ab_lib": a.ab_lib, "results": res}
    text = json.dumps(line, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
