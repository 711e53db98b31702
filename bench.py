#!/usr/bin/env python
"""
bench.py -- compensated points/s of the motion-compensation hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--variant V5] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[3], SURVEY.md 8d "M-1H"): a synthetic 1 h Mid-70 stream, 36 000
frames x 10 000 points = 3.6e8 points, figure-eight trajectory sampled at 200 Hz (720 001 pose
samples) with GPS/IMU noise.  One "step" = one pass of the fused kernel over the whole stream:
per-point binary search of the timestamp + SLERP/lerp pose interpolation + f64 rigid transform +
LVX int32-mm quantisation (variant V5, 50 algorithmic bytes per point).

At N > 1 every rank processes its own 1 h frame range of an N-hour stream (frame-sharded, weak
scaling, no data-path collective); the merged-cloud all-gather is timed separately and reported
under "merge".  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

METRIC = "compensated points/sec"
UNIT = "points/s"
N_FRAMES, PTS_PER_FRAME, SEED = 36_000, 10_000, 4242

# algorithmic bytes per point (SURVEY.md 8d table; pose/sample tables and frame_off excluded)
VARIANTS = {
    #        mode      f64    ts   lvx    las   B/pt
    "V0": ("rigid", True, None, False, False, 64),
    "V1": ("rigid", False, None, False, False, 32),
    "V2": ("rigid", False, None, True, False, 46),
    "V3": ("rigid", False, None, False, True, 46),
    "V4": ("slerp", False, "u32", False, False, 36),
    "V5": ("slerp", False, "u32", True, False, 50),
    "V5las": ("slerp", False, "u32", False, True, 50),
    "V4b": ("gyro", False, "u32", False, False, 36),
    # the second simulator's fused product: gyro deskew + LVX2 records of the COMPENSATED points (CS:1435-1536 + 365-374)
    "V5b": ("gyro", False, "u32", "lvx2", False, 50),
    # the reference-native types end to end: f64 (N,4) rows, int64 ns timestamps (CS:125), f64 rows out + LVX records
    "V6": ("slerp", True, "i64", True, False, 86),
}


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel (ncu --set full, profiles/)
NCU_TRAFFIC = {("V5", N_FRAMES, PTS_PER_FRAME): 18.100e9, ("V1", N_FRAMES, PTS_PER_FRAME): 11.489e9, ("V2", N_FRAMES, PTS_PER_FRAME): 16.518e9, ("V4b", N_FRAMES, PTS_PER_FRAME): 12.948e9}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", default="V5", choices=sorted(VARIANTS))
    ap.add_argument("--frames", type=int, default=N_FRAMES)
    ap.add_argument("--ppf", type=int, default=PTS_PER_FRAME)
    ap.add_argument("--path", default="auto", choices=["auto", "direct", "tma"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-frames", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0's stream; rows at "
                         "fixed seeded positions when the whole would exceed DUMP_BYTES)")
    return ap.parse_args()


DUMP_BYTES = 60 << 20            # --dump-outputs writes at most this much (plus .npy headers)


def dump_outputs(out_dir, out, into):
    """The headline step's results as a caller of the operator receives them, in float32 / float64: out.npy = the aligned
    rows, lvx.npy = the LVX records decoded to [x_mm, y_mm, z_mm, reflectivity, tag], las.npy = [X, Y, Z, intensity],
    status.npy = the flag word.  Row i of each file is point idx[i] of the stream, idx = the sorted seeded sample below."""
    import torch
    n = out.shape[0]
    row_bytes = 4 * out.element_size() + (40 if into.lvx14 is not None else 0) + (32 if into.las_x is not None else 0)
    k = min(n, DUMP_BYTES // row_bytes)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    idx_d = torch.from_numpy(idx).to(out.device)
    take = lambda t: t.index_select(0, idx_d).cpu().numpy()          # noqa: E731
    arrays = {"out": take(out), "status": into.status.cpu().numpy().astype(np.float64)}
    if into.lvx14 is not None:
        rec = take(into.lvx14)
        arrays["lvx"] = np.column_stack([rec[:, :12].copy().view("<i4"), rec[:, 12:14]]).astype(np.float64)
    if into.las_x is not None:
        intensity = take(into.las_intensity.view(torch.int16)).view(np.uint16)       # index_select has no uint16 kernel
        arrays["las"] = np.column_stack([take(into.las_x), take(into.las_y), take(into.las_z), intensity]).astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------
# clocks during the timed region (NVML; same fields as the recipe's nvidia-smi line)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int, period: float = 0.02):
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self.period, self._stop, self._t = period, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                    # noqa: BLE001
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:                 # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:                     # noqa: BLE001
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        if self._t is not None:
            self._stop.set()
            self._t.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": getattr(self, "err", "no samples")}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max": max(self.power) if self.power else None}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:                          # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU path on this box's host cores
#   kind "reference": the UNMODIFIED reference staged under oracle/_ref (oracle/make_ref.py), stock code path,
#                     one forked worker per host core (oracle/ref_arm.py)
#   kind "port":      the vectorised NumPy/SciPy port on a thread pool (oracle/cpu_baseline.py) -- reported beside it as the
#                     "fair CPU" figure, and the fallback when oracle/_ref was never staged
# ----------------------------------------------------------------------------------------------
def workload_name(F, P):
    return f"M-1H synthetic 1 h Mid-70 stream: {F} frames x {P} pts = {F * P} points, 200 Hz pose samples ({F * 20 + 1}), seed {SEED}"


def sharding_pcd_header(n):
    from livox_motion_compensation_sim_b200.simulator import LiDARMotionSimulator
    return LiDARMotionSimulator._pcd_header(int(n))


def cpu_port_run(steps, warmup, frames, ppf):
    from oracle import cpu_baseline as cb
    threads = cb.default_threads()
    sample = cb.make_sample(frames, ppf)
    for _ in range(warmup):
        cb.run_port(sample, threads)
    times = [cb.run_port(sample, threads) for _ in range(steps)]
    t = float(np.mean(times))
    return dict(value=sample['n_points'] / t, seconds_per_step=t, cores=threads, n_points=sample['n_points'], kind="port",
                sample=f"{frames} frames x {ppf} pts of the M-1H stream per step (f64 (n,4), NumPy/SciPy port of LMC:802-832 + vstack + LVX mm quantise, {threads} threads)")


def cpu_reference_run(steps, warmup, frames, ppf):
    """The stock reference when oracle/_ref is staged, else the port.  Always returns the port's rate too."""
    from oracle import make_ref
    if make_ref.available():
        from oracle import ref_arm
        r = ref_arm.run(steps, warmup, frames, ppf)
        r["kind"] = "reference"
        port = cpu_port_run(min(steps, 3), 1, frames, ppf)
        r["fair_port"] = {"points_per_s": port["value"], "cores": port["cores"], "what": port["sample"]}
        return r
    r = cpu_port_run(steps, warmup, frames, ppf)
    r["note"] = "oracle/_ref is not staged on this box (python oracle/make_ref.py in the build container): the port stands in"
    return r


def cpu_baseline_block(r):
    b = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
    for k in ("stage_a_points_per_s", "stage_b_points_per_s", "fair_port", "note"):
        if k in r:
            b[k] = r[k]
    return b


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    r = cpu_reference_run(steps, warmup, args.cpu_frames, args.ppf)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": r["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.frames, args.ppf),
                   "variant": "the reference's CPU path for the hot path: hold-next pose per frame + transform_pointcloud + vstack + LVX int32-mm records "
                              "(Mode A + LVX = the GPU arm's config.like_for_like variant V2; the reference has no per-point pose interpolation)",
                   "sample_per_step": r["sample"]},
        "cpu_baseline": cpu_baseline_block(r),
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------
def main_b200(args):
    import torch
    import torch.distributed as dist
    from livox_motion_compensation_sim_b200 import _build, _capi as C, ops, synth
    from livox_motion_compensation_sim_b200.pipeline import HostStream, StreamingAligner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from livox_motion_compensation_sim_b200.pipeline import bind_host_to_gpu
    orig_affinity = os.sched_getaffinity(0)
    numa_cpus = None if args.no_numa_bind else bind_host_to_gpu(local)      # pinned e2e buffers on the GPU's own socket
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep NCCL's version banner off stdout (ONE JSON line)
        dist.init_process_group("nccl", device_id=dev)
    if not os.path.exists(_build.LIB_PATH):
        if rank == 0:
            _build.build_library()
        if world > 1:
            dist.barrier()
    if args.path != "auto":
        C.set_path(C.PATH_DIRECT if args.path == "direct" else C.PATH_TMA)

    F, P = args.frames, args.ppf
    # rank r owns hour r of an N-hour stream: same shape, different seed
    st = synth.make_stream(F, P, SEED + 17 * rank, device=dev, dtype=torch.float32)
    N = st.n_points
    n_samples = len(st.sample_ts)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)   # noqa: E731
    off_d, fs_d, sts_d, seg_d = d(st.frame_off), d(st.frame_start), d(st.sample_ts), d(st.seg)
    gyro_d = d(np.random.default_rng(3).normal(0, 0.2, (len(st.sample_ts), 3)))
    # Mode A pose table through the device lookup kernel (a1)
    pose_d, _ = ops.pose_lookup_hold_next(d(st.gps_t), d(st.gps_Rt), d(st.frame_t))
    pts64 = None

    def make_step(variant):
        nonlocal pts64
        mode, f64, ts, lvx, las, bpp = VARIANTS[variant]
        pts = st.pts
        if f64:
            if pts64 is None:
                pts64 = st.pts.to(torch.float64)
            pts = pts64
        ts_d = st.ts_off
        if ts == "i64":                               # absolute int64 ns per point
            ts_d = fs_d.repeat_interleave(off_d[1:] - off_d[:-1]) + st.ts_off.to(torch.int64)
        out = torch.empty_like(pts)
        into = ops.ExportBuffers(status=torch.zeros(1, dtype=torch.int32, device=dev))
        if lvx:
            into.lvx14 = torch.empty((N, 14), dtype=torch.uint8, device=dev)
        if las:
            into.las_x, into.las_y, into.las_z = (torch.empty(N, dtype=torch.int32, device=dev) for _ in range(3))
            into.las_intensity = torch.empty(N, dtype=torch.uint16, device=dev)
        spec = ops.ExportSpec(lvx=bool(lvx), lvx_mode=C.LVX2_OF_OUTPUT if lvx == "lvx2" else C.LVX_TYPE2_OF_INPUT, las=las,
                              las_scale=(0.001,) * 3, into=into) if (lvx or las) else None
        if mode == "rigid":
            fn = lambda: ops.align_rigid(pts, off_d, pose_d, out=out, export=spec)                       # noqa: E731
        elif mode == "slerp":
            fn = lambda: ops.deskew_slerp(pts, ts_d, off_d, fs_d, sts_d, seg_d, out=out, export=spec)  # noqa: E731
        else:
            fn = lambda: ops.deskew_gyro(pts, ts_d, off_d, fs_d, sts_d, gyro_d, out=out, export=spec)  # noqa: E731
        return fn, bpp, (out, into)

    def timed(fn, steps, warmup, sampler=None):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        for i in range(steps):
            fn()
            evs[i + 1].record()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        if world > 1:
            dist.barrier()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        total_ms = evs[0].elapsed_time(evs[steps])
        if world > 1:
            t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms, per, clocks

    # ---- headline: resident inputs, CUDA events, max over ranks ------------------------------------
    fn, bpp, keep = make_step(args.variant)
    sampler = ClockSampler(local)
    total_ms, per, clocks = timed(fn, args.steps, max(args.warmup, 3), sampler)
    ms_per_step = total_ms / args.steps
    value = world * N / (ms_per_step * 1e-3)
    kern_ms = float(np.mean(per))                     # one fused kernel per step on this stream
    peak, peak_src = measured_peak()
    achieved = N * bpp / (kern_ms * 1e-3) / 1e9
    flags = keep[1].flags()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *keep)
    del keep, fn

    # ---- other variants (short runs; context for the roofline) ---------------------------------------
    sweep = {}
    if not args.no_sweep:
        for v in VARIANTS:
            if v == args.variant:
                continue
            try:
                f2, b2, k2 = make_step(v)
                tms, _, _ = timed(f2, 10, 3)
                sweep[v] = {"points_per_s": world * N / (tms / 10 * 1e-3), "GBps_per_gpu": N * b2 / (tms / 10 * 1e-3) / 1e9,
                            "frac": N * b2 / (tms / 10 * 1e-3) / 1e9 / peak, "bytes_per_point": b2}
                del f2, k2
            except Exception as e:                # noqa: BLE001
                sweep[v] = {"error": repr(e)}
            torch.cuda.empty_cache()
    pts64 = None
    torch.cuda.empty_cache()

    # ---- M-SWEEP (BASELINE configs[4]): fused transform + LVX / LAS int32 quantise, 10 k .. 1 M points per frame,
    #      1e8 points each (same resident points, re-framed) -----------------------------------------------------
    m_sweep = None
    if rank == 0 and not args.no_sweep:
        try:
            m_sweep = {}
            n2 = min(N, 100_000_000)
            lvx_b = torch.empty((n2, 14), dtype=torch.uint8, device=dev)
            las_b = [torch.empty(n2, dtype=torch.int32, device=dev) for _ in range(3)] + [torch.empty(n2, dtype=torch.uint16, device=dev)]
            out_b = torch.empty((n2, 4), dtype=torch.float32, device=dev)
            for ppf in (10_000, 31_600, 96_000, 100_000, 316_000, 1_000_000):
                Fs = (n2 + ppf - 1) // ppf
                offs = np.minimum(np.arange(Fs + 1, dtype=np.int64) * ppf, n2)
                offs_d, pose_s = d(offs), pose_d[:Fs].contiguous()
                res = {}
                for tag, spec in (("lvx", ops.ExportSpec(lvx=True, into=ops.ExportBuffers(lvx14=lvx_b))),
                                  ("las", ops.ExportSpec(las=True, las_scale=(0.001,) * 3,
                                                         into=ops.ExportBuffers(las_x=las_b[0], las_y=las_b[1], las_z=las_b[2], las_intensity=las_b[3])))):
                    fn_s = lambda: ops.align_rigid(st.pts[:n2], offs_d, pose_s, out=out_b, export=spec)      # noqa: E731
                    for _ in range(3):
                        fn_s()
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(10):
                        fn_s()
                    e1.record(); torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1) / 10
                    res[tag] = {"points_per_s": n2 / (ms * 1e-3), "frac": n2 * 46 / (ms * 1e-3) / 1e9 / peak}
                m_sweep[str(ppf)] = res
            del lvx_b, las_b, out_b
        except Exception as e:                    # noqa: BLE001
            m_sweep = {"error": repr(e)}
        torch.cuda.empty_cache()

    # ---- the reference's own preset shape (BASELINE configs[1]: urban_complex, 1200 frames x ~1.6 k pts,
    #      f64 (n,4) host arrays) through the drop-in API: host list in -> host arrays out ------------------
    presets = None
    if rank == 0 and not args.no_sweep:
        try:
            from livox_motion_compensation_sim_b200 import LiDARMotionSimulator
            rngp = np.random.default_rng(42)
            cnt = rngp.integers(911, 2576, 1200)
            frames_h = [np.column_stack([rngp.uniform(-60, 60, (c, 3)), rngp.uniform(0.1, 0.9, c)]) for c in cnt]
            posp, eulp = rngp.uniform(-30, 30, (1200, 3)), rngp.normal(0, 0.3, (1200, 3))
            simp = LiDARMotionSimulator({'device': f'cuda:{local}', 'pinned_results': True})
            for _ in range(3):                                          # steady state: pinned result blocks cached
                simp.align_frames(frames_h, posp, eulp)
            t0 = time.perf_counter()
            for _ in range(5):
                merged_p, _, _ = simp.align_frames(frames_h, posp, eulp)
            t_api = (time.perf_counter() - t0) / 5
            from oracle import lmc_oracle as _orc                       # CPU port of the same loop, for context only
            t0 = time.perf_counter()
            want_p = _orc.align_frames_np(frames_h, posp, eulp)
            t_np = time.perf_counter() - t0
            presets = {"urban_complex_shape": {"frames": 1200, "points": int(cnt.sum()),
                                               "b200_api_ms": t_api * 1e3, "numpy_port_ms": t_np * 1e3,
                                               "bit_exact": bool(merged_p.tobytes() == want_p.tobytes()),
                                               "what": "LiDARMotionSimulator.align_frames(list of f64 (n,4)) incl. flatten, pose table, H2D, kernel, D2H vs the reference's per-frame loop + vstack"}}
            # the reference's WHOLE frame loop for configs[1] wording (figure-eight, complex, 60 s, 10 fps): pose
            # lookup + scan of every frame + noise replay + alignment, from the golden inputs of that run
            gp = os.path.join(ROOT, "tests", "golden", "scan_C2a.npz")
            if os.path.exists(gp):
                import hashlib
                g = dict(np.load(gp))
                cfgp = json.loads(g['config_json'].tobytes().decode())

                class _Src:
                    trajectory = {'time': g['traj_time'], 'position_gps': g['traj_position_gps'], 'orientation_imu': g['traj_orientation_imu'],
                                  'velocity': np.zeros_like(g['traj_position_gps'])}
                    environment = g['environment']
                simr = LiDARMotionSimulator(dict(cfgp, device=f'cuda:{local}', pinned_results=True))
                best = 1e9
                for _ in range(3):
                    np.random.set_state(('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached'])))
                    t0 = time.perf_counter()
                    resr = simr.run_simulation(_Src)
                    best = min(best, time.perf_counter() - t0)
                al = np.vstack(resr['aligned_pointclouds'])
                np.random.set_state(('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached'])))
                t0 = time.perf_counter()
                tms = np.linspace(0, cfgp['duration'], int(cfgp['duration'] * cfgp['lidar_fps']))
                ix = _orc.pose_lookup_hold_next_np(g['traj_time'], tms)
                fr_c = _orc.scan_frames(g['environment'], g['traj_position_gps'][ix], g['traj_orientation_imu'][ix], cfgp)
                _orc.align_frames_np(fr_c, g['traj_position_gps'][ix], g['traj_orientation_imu'][ix], merge=False)
                cpu_loop_ms = (time.perf_counter() - t0) * 1e3
                man = json.load(open(os.path.join(ROOT, "tests", "golden", "MANIFEST.json")))['lmc']['C2a']
                presets["urban_complex_60s_whole_loop"] = {
                    "frames": len(resr['raw_scans']), "points": int(len(al)), "b200_run_simulation_ms": best * 1e3,
                    "aligned_sha256_matches_reference": hashlib.sha256(al.tobytes()).hexdigest() == man['aligned_sha256'],
                    "cpu_port_ms": cpu_loop_ms,
                    "what": "LiDARMotionSimulator.run_simulation with the device scanner (LMC:778-858 loop: lookup + scan_environment + transform), host noise replay, results as host arrays; cpu_port_ms = the oracle's C scanner + NumPy transform port of the same loop, 1 thread"}
                # the run's hot-path outputs (LMC:860-930): 2 x 600 per-frame PCDs + 2 merged PCDs + LAS + LVX, text formatted
                # / quantised / laid out on the device (one formatting pass per cloud family), files written to local disk
                import shutil
                import tempfile
                tmpd = tempfile.mkdtemp(prefix="lmc_save_")
                try:
                    save_t = []
                    for rep in range(3):                                # first call pays `import pandas` and the pinned blocks
                        t0 = time.perf_counter()
                        simr.save_results(resr, os.path.join(tmpd, f"r{rep}"))
                        save_t.append((time.perf_counter() - t0) * 1e3)
                    one = os.path.join(tmpd, "r2")
                    n_files = sum(len(fs) for _, _, fs in os.walk(one))
                    n_bytes = sum(os.path.getsize(os.path.join(dp, f)) for dp, _, fs in os.walk(one) for f in fs)
                    presets["urban_complex_60s_save_results"] = {
                        "files": n_files, "bytes": n_bytes, "b200_save_results_ms": min(save_t[1:]), "first_call_ms": save_t[0],
                        "what": "LiDARMotionSimulator.save_results of that run: per-frame + merged PCD ('%.6f' text of 4 x 976 720 points), "
                                "LAS, LVX v1.1, CSVs; the reference's per-point Python writers format 0.26-0.8 Mpts/s (PCD) and 0.04 Mpts/s (LVX)"}
                finally:
                    shutil.rmtree(tmpd, ignore_errors=True)
            # configs[2] wording: parking_detailed (circular, medium, 30 s at 20 fps) with the per-point deskew
            # (pose_interpolation='slerp'): lookup + scan of every frame + per-point SLERP alignment
            gp3 = os.path.join(ROOT, "tests", "golden", "scan_C3.npz")
            if os.path.exists(gp3):
                g3 = dict(np.load(gp3))
                cfg3 = json.loads(g3['config_json'].tobytes().decode())

                class _Src3:
                    trajectory = {'time': g3['traj_time'], 'position_gps': g3['traj_position_gps'], 'orientation_imu': g3['traj_orientation_imu'],
                                  'velocity': np.zeros_like(g3['traj_position_gps'])}
                    environment = g3['environment']
                sim3 = LiDARMotionSimulator(dict(cfg3, device=f'cuda:{local}', pose_interpolation='slerp', pinned_results=True))
                best3 = 1e9
                for _ in range(3):
                    np.random.set_state(('MT19937', g3['rng_keys'], int(g3['rng_pos']), int(g3['rng_has_gauss']), float(g3['rng_cached'])))
                    t0 = time.perf_counter()
                    res3 = sim3.run_simulation(_Src3)
                    best3 = min(best3, time.perf_counter() - t0)
                presets["parking_detailed_30s_per_point_deskew"] = {
                    "frames": len(res3['raw_scans']), "points": int(sum(len(a) for a in res3['aligned_pointclouds'])),
                    "b200_run_simulation_ms": best3 * 1e3,
                    "what": "LiDARMotionSimulator({'pose_interpolation': 'slerp'}).run_simulation: device scanner + per-point bracket search / SLERP / lerp over the trajectory samples (parity vs the SciPy oracle in tests)"}
        except Exception as e:                    # noqa: BLE001
            presets = {"error": repr(e)}

    # ---- downstream writers fed from device buffers (SURVEY 8f N1 / N2), bounded sample ---------------
    writers = None
    if rank == 0 and not args.no_sweep:
        try:
            from livox_motion_compensation_sim_b200.lvx import frame_layout
            fw = min(F, 3600)
            nw = int(st.frame_off[fw])
            _, fpos = frame_layout(st.frame_off[:fw + 1])
            fpos_d, offw, ftw, idw = d(fpos), d(st.frame_off[:fw + 1]), d(st.frame_t[:fw]), d(np.arange(fw, dtype=np.int64))
            raw = st.pts[:nw]

            def t_ms(fn, reps=5):
                fn(); torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn()
                e1.record(); torch.cuda.synchronize()
                return e0.elapsed_time(e1) / reps
            lvx_ms = t_ms(lambda: ops.build_lvx_v11(raw, offw, fpos_d, ftw, idw, P, size=int(fpos[-1])))
            lvx_bytes = int(fpos[-1])
            pcd_ms = t_ms(lambda: ops.pcd_ascii_body(raw))
            pcd_bytes = int(ops.pcd_ascii_body(raw)[0].numel())
            from livox_motion_compensation_sim_b200 import _capi as _C
            tsw = d((st.frame_t[:fw] * 1e9).astype(np.int64))
            pre2 = bytes(88)
            cs_ms = t_ms(lambda: ops.build_lvx_cs(raw, None, offw, tsw, pre2, _C.LVXCS_LVX2, P))
            cs_bytes = 88 + 45 * fw + 14 * nw
            las_ms = t_ms(lambda: ops.build_las_pf3(raw, scale=(0.001,) * 3, offset=(0.0,) * 3))
            las_bytes = _C.LAS_HEADER_BYTES + _C.LAS_RECORD_BYTES * nw
            rows5 = torch.cat([raw.double(), torch.arange(nw, device=raw.device, dtype=torch.float64).unsqueeze(1) * 1000.0], dim=1).contiguous()
            rows5[:, 3] = torch.floor(rows5[:, 3] * 255.0)
            txt_ms = t_ms(lambda: ops.text_rows(rows5, (0, 1, 2, 3, 4), (6, 6, 6, 0, 0), " "), reps=3)
            txt_bytes = int(ops.text_rows(rows5, (0, 1, 2, 3, 4), (6, 6, 6, 0, 0), " ")[0].numel())
            del rows5
            writers = {"sample_points": nw,
                       "cs_pcd_text": {"points_per_s": nw / (txt_ms * 1e-3), "GBps": (2 * nw * 40 + txt_bytes) / (txt_ms * 1e-3) / 1e9, "text_bytes": txt_bytes,
                                       "what": "'%.6f %.6f %.6f %.0f %.0f\\n' rows of the (N,5) f64 export array (CS:1663-1664), size + write passes"},
                       "lvx2_file": {"points_per_s": nw / (cs_ms * 1e-3), "GBps": (nw * 16 + cs_bytes) / (cs_ms * 1e-3) / 1e9,
                                     "file_bytes": cs_bytes, "what": "float4 [x y z intensity] -> complete LVX2 file image (CS:269-374) on the device"},
                       "las_pf3_file": {"points_per_s": nw / (las_ms * 1e-3), "GBps": (nw * 16 + las_bytes) / (las_ms * 1e-3) / 1e9,
                                        "file_bytes": las_bytes, "what": "float4 -> LAS 1.2 PF3 file image with header min/max (LMC:950-963), parity unpinned"},
                       "lvx_v11_file": {"points_per_s": nw / (lvx_ms * 1e-3), "GBps": (nw * 16 + lvx_bytes) / (lvx_ms * 1e-3) / 1e9,
                                        "file_bytes": lvx_bytes, "what": "raw float4 -> complete LVX v1.1 file image (LMC:58-272) on the device"},
                       "pcd_ascii": {"points_per_s": nw / (pcd_ms * 1e-3), "GBps": (2 * nw * 16 + pcd_bytes) / (pcd_ms * 1e-3) / 1e9,
                                     "text_bytes": pcd_bytes, "what": "'%.6f %.6f %.6f %.6f\\n' per point (LMC:946-947), size + write passes"}}
            del raw
        except Exception as e:                    # noqa: BLE001
            writers = {"error": repr(e)}
        torch.cuda.empty_cache()

    # ---- end to end: pinned host buffers in, pinned host buffers out ---------------------------------
    e2e = None
    e2e_mode_a = None
    if not args.no_e2e:
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:                          # noqa: BLE001
            avail = 64 << 30
        bytes_per_pt_host = 16 + 4 + 16 + 14
        budget = min(avail // (3 * max(world, 1)), N * bytes_per_pt_host)
        fe = max(1, min(F, int(budget // (bytes_per_pt_host * P))))
        ne = fe * P
        hs = HostStream(pts=torch.empty((ne, 4), dtype=torch.float32).pin_memory(),
                        ts_off=torch.empty(ne, dtype=torch.uint32).pin_memory(),
                        out=torch.empty((ne, 4), dtype=torch.float32).pin_memory(),
                        lvx14=torch.empty((ne, 14), dtype=torch.uint8).pin_memory(),
                        frame_off=st.frame_off[:fe + 1], frame_start=st.frame_start[:fe])
        hs.pts.copy_(st.pts[:ne]); hs.ts_off.copy_(st.ts_off[:ne])
        torch.cuda.synchronize()
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()   # noqa: E731
        pose_h = (pin(st.sample_quat), pin(st.sample_pos), pin(st.sample_ts))       # the pose stream travels with the points
        sa = StreamingAligner(dev, hs.frame_off, hs.frame_start, mode="slerp", lvx=True, pose_samples=pose_h)
        sa.run(hs); torch.cuda.synchronize()          # warm-up
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(args.e2e_steps):
            sa.run(hs)
        e1.record(); torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / args.e2e_steps
        ems = e0.elapsed_time(e1) / args.e2e_steps
        if world > 1:
            t = torch.tensor([ems], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        # spot check: the pipelined host result equals the resident-data result
        chk = ops.deskew_slerp(st.pts[:P], st.ts_off[:P], d(st.frame_off[:2]), fs_d[:1].contiguous(), sa.sample_ts, sa.seg)[0]
        assert torch.equal(chk.cpu(), hs.out[:P]), "e2e pipeline result differs from the resident-data result"
        e2e = {"value": world * ne / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": sa.h2d_bytes, "d2h_bytes_per_step": sa.d2h_bytes,
               "ms_per_step": ems, "wall_ms_per_step": wall * 1e3, "points_per_step_per_gpu": ne, "kernel_launches_per_step": sa.launches,
               "what": "StreamingAligner.run: pinned host float4 + u32 ts + the 200 Hz pose samples (quat, pos, ts) -> H2D, pose-segment table built on the device, chunked fused Mode C + LVX kernel, D2H of float4 + 14-B records, 3 streams",
               "h2d_GBps": sa.h2d_bytes / (ems * 1e-3) / 1e9, "d2h_GBps": sa.d2h_bytes / (ems * 1e-3) / 1e9,
               "host_cpus_bound": None if numa_cpus is None else len(numa_cpus)}
        # the same host buffers through the reference's own transform (Mode A + LVX records = variant V2): the like-for-like
        # partner of the reference arm, which has no per-point pose interpolation
        try:
            sa2 = StreamingAligner(dev, hs.frame_off, hs.frame_start, mode="rigid", lvx=True, pose_Rt=pose_d[:fe].contiguous())
            sa2.run(hs); torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0.record()
            for _ in range(args.e2e_steps):
                sa2.run(hs)
            e1.record(); torch.cuda.synchronize()
            ems2 = e0.elapsed_time(e1) / args.e2e_steps
            if world > 1:
                t = torch.tensor([ems2], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ems2 = float(t.item())
            e2e_mode_a = {"value": world * ne / (ems2 * 1e-3), "ms_per_step": ems2, "h2d_bytes_per_step": sa2.h2d_bytes, "d2h_bytes_per_step": sa2.d2h_bytes}
            del sa2
        except Exception as e:                     # noqa: BLE001
            e2e_mode_a = {"error": repr(e)}
        # the step's own copies without its kernels: the SAME pinned buffers, byte counts and chunking, H2D on one stream || D2H on
        # another, nothing between them (the 1 GiB-buffer ceiling below can overstate what 18 GB of pinned traffic per rank sustains)
        try:
            cur = torch.cuda.current_stream(dev)
            cuts = sa.cuts

            def raw_step():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(cur)
                sa.s_in.wait_event(e0); sa.s_out.wait_event(e0)
                for ci, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
                    p0, p1 = int(hs.frame_off[a]), int(hs.frame_off[b])
                    m, sl = p1 - p0, ci % sa.nbuf
                    with torch.cuda.stream(sa.s_in):
                        sa.d_pts[sl][:m].copy_(hs.pts[p0:p1], non_blocking=True)
                        sa.d_ts[sl][:m].copy_(hs.ts_off[p0:p1], non_blocking=True)
                    with torch.cuda.stream(sa.s_out):
                        hs.out[p0:p1].copy_(sa.d_out[sl][:m], non_blocking=True)
                        hs.lvx14[p0:p1].copy_(sa.d_lvx[sl][:m], non_blocking=True)
                cur.wait_stream(sa.s_in); cur.wait_stream(sa.s_out)
                e1.record(cur)
                torch.cuda.synchronize()
                return e0.elapsed_time(e1)
            best = None
            for _ in range(3):                               # first pass = warm-up, counted only if fastest
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                ms_raw = raw_step()
                if world > 1:
                    t = torch.tensor([ms_raw], dtype=torch.float64, device=dev)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    ms_raw = float(t.item())
                best = ms_raw if best is None else min(best, ms_raw)
            e2e["copy_ceiling_step_buffers"] = {
                "ms": best, "points_per_s": world * ne / (best * 1e-3), "h2d_GBps_per_gpu": ne * 20 / (best * 1e-3) / 1e9,
                "d2h_GBps_per_gpu": ne * 30 / (best * 1e-3) / 1e9,
                "what": "the step's own cudaMemcpyAsync calls (same pinned buffers, 20 B in + 30 B out per point, same chunks) with no kernels and no "
                        "dependencies between the two copy streams, every rank at once, max over ranks"}
            e2e["frac_of_step_buffer_copy_ceiling"] = e2e["value"] / e2e["copy_ceiling_step_buffers"]["points_per_s"]
        except Exception as e:                     # noqa: BLE001
            e2e["copy_ceiling_step_buffers_error"] = repr(e)
        del hs, sa
        torch.cuda.empty_cache()
        # raw copy ceiling of this box for the step's byte mix (profiles/pcie_ceiling.py: cudaMemcpyAsync only, every rank at once)
        try:
            sys.path.insert(0, os.path.join(ROOT, "profiles"))
            import pcie_ceiling
            ceil = pcie_ceiling.measure(dev, world, total=1 << 30, reps=2)
            e2e["copy_ceiling_points_per_s"] = ceil["e2e_points_per_s_ceiling_per_gpu"] * world
            e2e["frac_of_copy_ceiling"] = e2e["value"] / e2e["copy_ceiling_points_per_s"]
            e2e["copy_ceiling"] = {"duplex_h2d_GBps_per_gpu": ceil["duplex_h2d_GBps_per_gpu"], "duplex_d2h_GBps_per_gpu": ceil["duplex_d2h_GBps_per_gpu"],
                                   "h2d_alone_GBps_per_gpu": ceil["h2d_GBps_per_gpu"], "d2h_alone_GBps_per_gpu": ceil["d2h_GBps_per_gpu"],
                                   "what": "pinned cudaMemcpyAsync H2D || D2H in the step's 20:30 byte ratio, all ranks concurrently, no kernels (max over ranks)"}
        except Exception as e:                     # noqa: BLE001
            e2e["copy_ceiling_error"] = repr(e)
    # ---- merged cloud (BASELINE configs[3] literally): ONE 1 h stream, frame-sharded over the N ranks, the merged aligned
    #      cloud + LVX records assembled on every rank (np.vstack of LMC:886-899, as an all-gather).  Strong scaling.  Every
    #      method's merged buffers are compared byte for byte, on every rank, with the single-launch result of the whole
    #      stream computed on that rank; any difference fails the run.
    merge = None
    if world > 1:
        from livox_motion_compensation_sim_b200 import sharding
        del st
        torch.cuda.empty_cache()
        sm_st = synth.make_stream(F, P, SEED, device=dev, dtype=torch.float32)          # the SAME stream on every rank
        Nm = sm_st.n_points
        offm, fsm = d(sm_st.frame_off), d(sm_st.frame_start)
        stsm, segm = d(sm_st.sample_ts), d(sm_st.seg)                                    # ITS pose table (the ranks' own streams differ)
        fcuts, pcuts = sharding.shard_ranges(sm_st.frame_off, world)
        pb, pe = int(pcuts[rank]), int(pcuts[rank + 1])
        symm = sharding.SymmetricMerged(Nm, dev, lvx=True)
        po, pl = symm.peer_ptrs()
        mo, ml = symm.mc_ptrs()
        whole, wbuf = ops.deskew_slerp(sm_st.pts, sm_st.ts_off, offm, fsm, stsm, segm, export=ops.ExportSpec(lvx=True))   # 1-GPU result
        own = lambda: ops.ExportBuffers(lvx14=symm.lvx14)                                # noqa: E731

        def run_shard_only():
            ops.deskew_slerp(sm_st.pts, sm_st.ts_off, offm, fsm, stsm, segm, out=symm.out,
                             export=ops.ExportSpec(lvx=True, into=own()), p_range=(pb, pe))

        def run_nccl():
            run_shard_only()
            sharding.all_gather_merged([symm.out, symm.lvx14], pcuts)

        def run_fused():
            ops.deskew_slerp(sm_st.pts, sm_st.ts_off, offm, fsm, stsm, segm, out=symm.out,
                             export=ops.ExportSpec(lvx=True, into=own(), peer_out=po, peer_lvx14=pl), p_range=(pb, pe))
            symm.barrier()

        def run_mc():
            ops.deskew_slerp(sm_st.pts, sm_st.ts_off, offm, fsm, stsm, segm, out=symm.out,
                             export=ops.ExportSpec(lvx=True, into=own(), peer_out=po, peer_lvx14=pl, mc_out=mo, mc_lvx14=ml), p_range=(pb, pe))
            symm.barrier()

        def identical(fn):
            """zero the merged buffers everywhere, run once, compare with the single-launch result on every rank"""
            symm.out.zero_(); symm.lvx14.zero_()
            symm.barrier()
            fn()
            torch.cuda.synchronize()
            ok = torch.equal(symm.out, whole) and torch.equal(symm.lvx14, wbuf.lvx14)
            t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            return bool(t.item())

        def t_max_ms(fn, reps=5):
            for _ in range(2):
                fn()
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record(); torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            return float(t.item())

        recv = (Nm - (pe - pb)) * 30
        recv_t = torch.tensor([recv], dtype=torch.int64, device=dev)
        dist.all_reduce(recv_t, op=dist.ReduceOp.MAX)
        recv = int(recv_t.item())
        shard_ms = t_max_ms(run_shard_only)
        methods = {}
        for name, fn, what in (
                ("nccl_allgather", run_nccl, "shard kernel, then NCCL all-gather(v) of the aligned cloud + records"),
                ("fused_peer_store", run_fused, "ONE kernel: the epilogue also stores every result into each peer's symmetric-memory copy (st.global over NVLink), then a stream-ordered cross-rank barrier"),
                ("fused_multicast", run_mc if mo else None, "ONE kernel: every result of a full tile leaves as one multimem.st to the NVSwitch multicast mapping (replicated by the switch into all copies), then the barrier")):
            if fn is None:
                methods[name] = {"unavailable": "the symmetric buffers have no multicast mapping on this box"}
                continue
            try:
                ok = identical(fn)
                ms = t_max_ms(fn)
                methods[name] = {"ms": ms, "points_per_s": Nm / (ms * 1e-3), "ingress_GBps_per_rank": recv / (ms * 1e-3) / 1e9,
                                 "byte_identical": ok, "what": what}
            except Exception as e:                 # noqa: BLE001
                methods[name] = {"error": repr(e)}
        timed_ok = {k: v for k, v in methods.items() if "ms" in v}
        if not timed_ok:
            raise SystemExit(f"merged-cloud assembly failed on every path: {methods}")
        bad = [k for k, v in timed_ok.items() if not v["byte_identical"]]
        if bad:
            raise SystemExit(f"merged cloud differs from the single-launch result: {bad}")
        best = min(timed_ok, key=lambda k: timed_ok[k]["ms"])
        merge = {"what": f"ONE 1 h stream ({Nm} pts) frame-sharded over {world} ranks; aligned float4 cloud + 14-B LVX records merged on EVERY rank (np.vstack of LMC:886-899 as an all-gather); strong scaling",
                 "points": Nm, "bytes_received_per_rank": recv,
                 "shard_ms": shard_ms, "shard_points_per_s": Nm / (shard_ms * 1e-3),
                 "nccl_ms": methods["nccl_allgather"].get("ms"), "fused_ms": methods["fused_peer_store"].get("ms"),
                 "multicast_ms": methods["fused_multicast"].get("ms"),
                 "best": best, "best_ms": timed_ok[best]["ms"], "merged_points_per_s": Nm / (timed_ok[best]["ms"] * 1e-3),
                 "ingress_GBps": timed_ok[best]["ingress_GBps_per_rank"],
                 "byte_identical": all(v["byte_identical"] for v in timed_ok.values()), "methods": methods}
        # ---- replication-free file production: every rank turns ITS frames into ITS byte range of the LVX / LAS / PCD files
        #      (closed-form or prefix-summed offsets; only 6 + W integers cross ranks) -- the path that scales with N.
        try:
            from livox_motion_compensation_sim_b200.lvx import frame_layout
            fa, fb = int(fcuts[rank]), int(fcuts[rank + 1])
            ids_np = np.arange(F, dtype=np.int64)
            _, fpos_np = frame_layout(sm_st.frame_off)
            las_kw = dict(scale=(0.001,) * 3, year=2026, day_of_year=1)

            def files_sharded():
                run_shard_only()
                a = sharding.lvx_v11_shard(sm_st.pts, sm_st.frame_off, sm_st.frame_t, ids_np, fa, fb)
                b = sharding.las_pf3_shard(symm.out, pb, pe, rank, **las_kw)
                c = sharding.pcd_ascii_shard(symm.out[pb:pe], Nm, rank)
                return a, b, c

            def files_one_gpu():
                ops.deskew_slerp(sm_st.pts, sm_st.ts_off, offm, fsm, stsm, segm, out=whole, export=ops.ExportSpec(lvx=True, into=ops.ExportBuffers(lvx14=wbuf.lvx14)))
                a = ops.build_lvx_v11(sm_st.pts, offm, d(fpos_np), d(sm_st.frame_t), d(ids_np), P)
                b = ops.build_las_pf3(whole, **las_kw)
                c = ops.pcd_ascii_body(whole)
                return a, b, c
            (lv_s, lv_pos, _), (la_s, la_pos, _), (tx_s, tx_pos, tx_hdr, _) = files_sharded()
            (lv_w, _), (la_w, _), (tx_w, _) = files_one_gpu()
            torch.cuda.synchronize()
            hdr_len = len(sharding_pcd_header(Nm))
            same = (torch.equal(lv_s, lv_w[lv_pos:lv_pos + lv_s.numel()]) and torch.equal(la_s, la_w[la_pos:la_pos + la_s.numel()])
                    and torch.equal(tx_s, tx_w[tx_pos - hdr_len:tx_pos - hdr_len + tx_s.numel()]))
            t = torch.tensor([1 if same else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            file_bytes = int(lv_w.numel() + la_w.numel() + tx_w.numel() + hdr_len)
            del lv_s, la_s, tx_s, lv_w, la_w, tx_w
            torch.cuda.empty_cache()
            if not bool(t.item()):
                raise SystemExit("sharded file ranges differ from the single-GPU file images")
            one_ms = t_max_ms(lambda: (torch.cuda.synchronize(), files_one_gpu()), reps=2)
            shard_files_ms = t_max_ms(lambda: (torch.cuda.synchronize(), files_sharded()), reps=2)
            sharded_files = {"what": "aligned cloud + LVX v1.1 file image (raw points) + LAS 1.2 PF3 file image + ASCII PCD text of the merged cloud, every rank building only ITS byte range "
                                     "(shard kernel + k_lvx_v11 + k_las_* + k_pcd_*; all-reduce of 6 extremes, all-gather of W text sizes); one_gpu_ms = the same kernels over the whole stream on one GPU",
                             "file_bytes": file_bytes, "ms": shard_files_ms, "one_gpu_ms": one_ms, "speedup_vs_one_gpu": one_ms / shard_files_ms,
                             "points_per_s": Nm / (shard_files_ms * 1e-3), "byte_identical": True}
        except SystemExit:
            raise
        except Exception as e:                     # noqa: BLE001
            sharded_files = {"error": repr(e)}
        merge["sharded_files"] = sharded_files
        del symm, sm_st, whole, wbuf
        torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, N = 1 only): the reference's own code on the host cores + the integer parity check ----------
    cpu = None
    int_mism = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, orig_affinity)             # the CPU baseline gets every host core back
        r = cpu_reference_run(3, 1, args.cpu_frames, P)
        cpu = cpu_baseline_block(r)
        try:
            from oracle import cpu_baseline as cb
            cpu["c_port_mode_c_1thread_points_per_s"] = cb.run_c_port_mode_c()
            cpu["writers_port_points_per_s"] = cb.run_writers_port()
        except Exception as e:                     # noqa: BLE001
            cpu["c_port_error"] = repr(e)
        # integer export buffers of the first 48 frames against the oracle (bit-exact is the bar: every count must be 0)
        try:
            from oracle import lmc_oracle as orc
            fc = min(F, 48)
            nc = int(st.frame_off[fc])
            offc, fsc = d(st.frame_off[:fc + 1]), fs_d[:fc].contiguous()
            p64 = st.pts[:nc].cpu().numpy().astype(np.float64)
            ts64 = st.frame_start[np.repeat(np.arange(fc), np.diff(st.frame_off[:fc + 1]))] + st.ts_off[:nc].cpu().numpy().astype(np.int64)
            spec = ops.ExportSpec(lvx=True, las=True, las_scale=(0.001,) * 3)
            o_c, b_c = ops.deskew_slerp(st.pts[:nc].contiguous(), st.ts_off[:nc].contiguous(), offc, fsc, sts_d, seg_d, export=spec)
            want = orc.C.deskew_slerp_f64(p64, ts64, st.frame_off[:fc + 1], st.sample_ts, st.seg)
            X, Y, Z, I, _ = orc.C.quantize_las(want, [0.001] * 3, [0.0] * 3, 0)
            int_mism = {"points": nc,
                        "lvx_records_mode_c": int((b_c.lvx14.cpu().numpy() != orc.C.quantize_lvx_type2(p64)[0]).any(axis=1).sum()),
                        "las_xyz_mode_c": int((b_c.las_x.cpu().numpy() != X).sum() + (b_c.las_y.cpu().numpy() != Y).sum() + (b_c.las_z.cpu().numpy() != Z).sum()),
                        "las_intensity_mode_c": int((b_c.las_intensity.cpu().numpy() != I).sum()),
                        "float_max_abs_err_m": float(np.abs(o_c.cpu().numpy().astype(np.float64) - want).max())}
            pose_c = st.gps_Rt[orc.pose_lookup_hold_next_np(st.gps_t, st.frame_t[:fc])]
            o_a, b_a = ops.align_rigid(d(p64), offc, d(pose_c), export=ops.ExportSpec(lvx=True, las=True, las_scale=(0.001,) * 3))
            want_a = orc.C.align_rigid_f64(p64, st.frame_off[:fc + 1], pose_c)
            Xa, Ya, Za, Ia, _ = orc.C.quantize_las(want_a, [0.001] * 3, [0.0] * 3, 0)
            int_mism["f64_rows_mode_a"] = int((o_a.cpu().numpy() != want_a).any(axis=1).sum())
            int_mism["lvx_records_mode_a"] = int((b_a.lvx14.cpu().numpy() != orc.C.quantize_lvx_type2(p64)[0]).any(axis=1).sum())
            int_mism["las_xyz_mode_a"] = int((b_a.las_x.cpu().numpy() != Xa).sum() + (b_a.las_y.cpu().numpy() != Ya).sum() + (b_a.las_z.cpu().numpy() != Za).sum())
        except Exception as e:                     # noqa: BLE001
            int_mism = {"error": repr(e)}

    if rank == 0:
        mode, f64, ts, lvx, las, _ = VARIANTS[args.variant]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(F, P), "per_gpu": f"every rank owns one such stream (rank r = hour r of an N-hour recording, seed {SEED} + 17 r)",
                       "variant": f"{args.variant}: mode={mode} io={'f64' if f64 else 'f32 float4'} ts={ts} lvx={lvx} las={las}, f64 arithmetic",
                       "bytes_per_point": bpp, "kernel_path": {0: "direct", 1: "auto (persistent TMA pipeline at this size)", 2: "tma"}[C.get_path()],
                       "l2": f"inputs {N * (16 + 4) / 1e9:.1f} GB >> 126 MB L2: no flush needed", "parallelism": f"frame-sharded x{world}",
                       "status_flags": flags},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": NCU_TRAFFIC.get((args.variant, F, P)), "traffic_source": f"profiles/{'r02' if args.variant in ('V5', 'V4b') else 'r01'}_ncu_{args.variant.lower()}_summary.md (dram__bytes_read + dram__bytes_write of one launch, ncu --set full)" if (args.variant, F, P) in NCU_TRAFFIC else None, "peak_source": peak_src, "kernel_ms": kern_ms,
                         "algorithmic_bytes_per_launch": N * bpp, "frac_of_nominal_8TBps": achieved / 8000.0},
            "clocks": clocks, "gpu_launches": args.steps, "e2e": e2e, "cpu_baseline": cpu,
        }
        if int_mism is not None:
            line["config"]["int_mismatches"] = int_mism
        if sweep.get("V2") or e2e_mode_a:
            line["config"]["like_for_like"] = {
                "variant": "V2: Mode A (the reference's hold-next frame pose, LMC:802-832) + LVX records -- the transform the reference arm runs",
                "value": (sweep.get("V2") or {}).get("points_per_s"), "roofline_frac": (sweep.get("V2") or {}).get("frac"), "e2e": e2e_mode_a}
        if merge:
            line["config"]["merge"] = merge
            line["roofline"]["nvlink"] = {"bound": "nvlink ingress", "bytes_received_per_rank": merge["bytes_received_per_rank"], "ms": merge["best_ms"],
                                          "achieved": merge["ingress_GBps"], "peak": 900.0, "unit": "GB/s", "frac": merge["ingress_GBps"] / 900.0,
                                          "method": merge["best"], "peak_source": "NVLink 5 nominal 900 GB/s per direction per GPU (B200_PROFILING.md); measured raw all-gather ceiling of this pool: profiles/r02_nvlink_ceiling_n*.json"}
        if sweep:
            line["variants"] = sweep
        if writers:
            line["writers"] = writers
        if presets:
            line["presets"] = presets
        if m_sweep:
            line["m_sweep"] = m_sweep
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


class _QuietStdout:
    """Everything but the final JSON line goes to stderr -- including C-level writes to fd 1 such as
    the 'NCCL version ...' banner printed at communicator creation -- so stdout carries ONE line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


_real_print = print


def print(*a, **k):                       # noqa: A001  (the JSON line is printed while fd 1 is diverted: send it to the saved fd)
    if _QUIET is not None:
        sys.stdout.flush()
        os.write(_QUIET.saved, (" ".join(str(x) for x in a) + "\n").encode())
    else:
        _real_print(*a, **k)


_QUIET = None

if __name__ == "__main__":
    a = parse()
    with _QuietStdout() as _QUIET:
        if a.impl == "reference":
            main_reference(a)
        else:
            main_b200(a)
