"""CPU-only tests: host logic of the product package, the C-ABI surface (load + exported symbols,
no compute calls), the LVX container layout against the reference's file bytes, and the
frame-sharded merge over gloo with world_size 2."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from livox_motion_compensation_sim_b200 import _build, _capi, frames as FR
from livox_motion_compensation_sim_b200.lvx import build_lvx_v11_file, frame_layout, FILE_HEADER
from oracle import lmc_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    return _build.build_library()


def test_capi_exports_every_declared_symbol(built_lib):
    header = open(os.path.join(ROOT, "include", "lmc_b200.h")).read()
    declared = set(re.findall(r"\b(lmc_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(built_lib)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/lmc_b200.h but not exported"
    assert declared == set(_capi.EXPORTED_SYMBOLS)
    assert _capi.lib().lmc_version() == 100


def test_capi_struct_layout_matches_header():
    # struct lmc_export: pointer/int interleaving -> check ctypes offsets against the C layout rules
    E = _capi.LmcExport
    assert E.lvx14.offset == 0 and E.lvx_mode.offset == 8 and E.tag.offset == 16
    assert E.las_x.offset == 24 and E.las_intensity.offset == 48 and E.las_intensity_mode.offset == 56
    assert E.las_scale.offset == 64 and E.las_offset.offset == 88 and E.status.offset == 112
    assert E.n_peers.offset == 120 and E.peer_out.offset == 128 and E.peer_lvx14.offset == 184
    assert E.mc_out.offset == 240 and E.mc_lvx14.offset == 248
    assert ctypes.sizeof(E) == 256


def test_capi_fails_loudly_without_gpu(built_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = _capi.lib()
    rc = L.lmc_device_query(None, None, None)
    assert rc == _capi.ERR_CUDA
    with pytest.raises(_capi.LmcError):
        _capi.check(rc)
    from livox_motion_compensation_sim_b200 import ops
    with pytest.raises(TypeError):                      # CPU tensors are refused: no CPU fallback
        ops.align_rigid(torch.zeros((4, 4), dtype=torch.float64), torch.tensor([0, 4]), torch.zeros((1, 12), dtype=torch.float64))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "livox_motion_compensation_sim_b200")
    for dp, _, fn in os.walk(pkg):
        for f in fn:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "lmc_oracle" not in src or f.endswith((".cu", ".cuh")), f


def test_config_contract():
    import torch  # noqa: F401
    from livox_motion_compensation_sim_b200.simulator import LiDARMotionSimulator
    sim = LiDARMotionSimulator({'duration': 12.0, 'some_unknown_key': 1})
    assert sim.config['duration'] == 12.0 and sim.config['some_unknown_key'] == 1
    ref_defaults = {'duration': 60.0, 'lidar_fps': 10, 'imu_rate': 100, 'gps_rate': 5, 'random_seed': 42, 'max_speed': 15.0,
                    'max_angular_vel': 0.5, 'trajectory_type': 'figure_eight', 'fov_horizontal': 70.0, 'fov_vertical': 77.2,
                    'range_max': 90.0, 'range_min': 0.05, 'points_per_frame': 96000, 'angular_resolution': 0.28,
                    'gps_noise_std': 0.03, 'imu_accel_noise': 0.1, 'imu_gyro_noise': 0.01, 'lidar_range_noise': 0.02,
                    'environment_complexity': 'medium', 'ground_height': 0.0, 'obstacle_density': 0.1}
    d = LiDARMotionSimulator().config
    for k, v in ref_defaults.items():
        assert d[k] == v
    for bad, msg in [({'duration': 'x'}, "Configuration 'duration' must be numeric"), ({'lidar_fps': 0}, "LiDAR frame rate must be positive"),
                     ({'duration': -1}, "Simulation duration must be positive"), ({'max_speed': -1}, "Maximum speed cannot be negative"),
                     ({'range_max': 1, 'range_min': 2}, "Maximum range must be greater than minimum range")]:
        with pytest.raises(ValueError, match=re.escape(msg)):
            LiDARMotionSimulator(bad)
    with pytest.raises(NotImplementedError):
        sim.run_simulation()


def test_frame_times_and_flatten():
    t = FR.lidar_frame_times(60.0, 10)
    assert len(t) == 600 and t[-1] == 60.0 and abs(t[1] - 60.0 / 599) < 1e-15        # linspace WITH endpoint (LMC:792)
    frames = [np.zeros((0, 4)), np.ones((3, 4)), np.array([]).reshape(0, 4), 2 * np.ones((1, 4))]
    flat, off = FR.flatten_frames(frames)
    assert off.tolist() == [0, 0, 3, 3, 4] and flat.shape == (4, 4)
    assert np.array_equal(flat, np.vstack(frames))
    back = FR.split_frames(flat, off)
    assert [len(b) for b in back] == [0, 3, 0, 1]


def test_host_gather_and_copy(built_lib):
    """lmc_host_gather / lmc_host_copy (host-only helpers of the C ABI): the threaded pack of a frame list equals
    np.vstack for ragged, empty, read-only and mixed-dtype lists, at every thread count."""
    rng = np.random.default_rng(5)
    cnt = rng.integers(0, 3000, 700)
    cnt[[0, 5, 699]] = 0
    frames = [rng.uniform(-90, 90, (c, 4)) for c in cnt]
    frames[7] = np.array([]).reshape(0, 4)
    frames[9].flags.writeable = False
    want = np.vstack(frames)
    flat = np.full_like(want, np.nan)
    FR.flatten_frames_into(frames, flat)
    assert flat.tobytes() == want.tobytes()
    mixed = list(frames)
    mixed[3] = mixed[3].astype(np.float32)                      # NumPy route (dtype conversion)
    mixed[4] = np.asfortranarray(mixed[4])
    flat[:] = np.nan
    FR.flatten_frames_into(mixed, flat)
    assert np.allclose(flat, want, rtol=1e-6)
    with pytest.raises(ValueError):
        FR.flatten_frames_into(frames[:-2], flat)
    L = _capi.lib()
    ptrs = np.array([FR._addr(a) for a in frames], np.uintp)
    boff = np.zeros(len(frames) + 1, np.int64)
    np.cumsum([a.nbytes for a in frames], out=boff[1:])
    for th in (1, 2, 3, 7, 64, 1000, 0, -3):
        dst = np.zeros(want.nbytes + 64, np.uint8)
        assert L.lmc_host_gather(ptrs.ctypes.data, boff.ctypes.data, len(frames), dst.ctypes.data, th) == 0
        assert dst[:want.nbytes].tobytes() == want.tobytes() and not dst[want.nbytes:].any()
        dst2 = np.zeros(want.nbytes + 64, np.uint8)
        assert L.lmc_host_copy(dst2.ctypes.data, want.ctypes.data, want.nbytes, th) == 0
        assert dst2[:want.nbytes].tobytes() == want.tobytes() and not dst2[want.nbytes:].any()
    assert L.lmc_host_gather(None, None, 0, None, 4) == 0 and L.lmc_host_copy(None, None, 0, 4) == 0
    bad = boff.copy(); bad[3] = bad[4] + 8
    assert L.lmc_host_gather(ptrs.ctypes.data, bad.ctypes.data, len(frames), flat.ctypes.data, 2) == _capi.ERR_INVALID
    assert L.lmc_host_copy(None, want.ctypes.data, 8, 1) == _capi.ERR_INVALID


def test_host_gather_property(built_lib):
    """Property test of lmc_host_gather: any list of byte runs (empty ones included), any thread count, any destination
    offset -> the concatenation, and not one byte outside it."""
    from hypothesis import given, settings, strategies as st
    L = _capi.lib()

    @settings(max_examples=60, deadline=None)
    @given(sizes=st.lists(st.integers(0, 3_000_000), min_size=0, max_size=40), threads=st.integers(-2, 70),
           lead=st.integers(0, 100), seed=st.integers(0, 2 ** 31))
    def check(sizes, threads, lead, seed):
        rng = np.random.default_rng(seed)
        srcs = [rng.integers(0, 256, n, dtype=np.uint8) for n in sizes]
        want = np.concatenate(srcs) if srcs else np.zeros(0, np.uint8)
        ptrs = np.array([FR._addr(a) for a in srcs], np.uintp)
        boff = np.full(len(srcs) + 1, lead, np.int64)
        if srcs:
            boff[1:] += np.cumsum(sizes)
        dst = np.full(lead + len(want) + 64, 0xEE, np.uint8)
        assert L.lmc_host_gather(ptrs.ctypes.data, boff.ctypes.data, len(srcs), dst.ctypes.data, threads) == 0
        assert dst[lead:lead + len(want)].tobytes() == want.tobytes()
        assert (dst[:lead] == 0xEE).all() and (dst[lead + len(want):] == 0xEE).all()
    check()


def test_legacy_normal_replays_numpy_global_stream(built_lib):
    """lmc_host_legacy_normal == np.random.normal on the seeded global generator (the stream scan_environment
    consumes at LMC:767): identical bits for even / odd / zero sizes, a cached second half carried across calls,
    block boundaries of the 624-word state, NumPy draws interleaved with ours, and the generator left behind."""
    for seed in (42, 7, 2024):
        for sizes in ([7, 8, 1, 0, 50_001, 5, 2], [2, 2, 623, 1, 20_000], [1] * 9 + [0, 3, 1234]):
            np.random.seed(seed); np.random.uniform(size=seed % 5)
            want = [np.random.normal(0, 0.02, n) for n in sizes]
            tail_w = (np.random.normal(0, 1, 5), np.random.random(3), np.random.randint(0, 1 << 30, 4))
            np.random.seed(seed); np.random.uniform(size=seed % 5)
            got = [FR.legacy_normal(0.02, n) for n in sizes]
            tail_g = (np.random.normal(0, 1, 5), np.random.random(3), np.random.randint(0, 1 << 30, 4))
            assert all(a.tobytes() == b.tobytes() for a, b in zip(want, got))
            assert all(a.tobytes() == b.tobytes() for a, b in zip(tail_w, tail_g))
    np.random.seed(9)
    a = (np.random.normal(0, 0.5, 3), np.random.normal(0, 0.5, (4, 3)), np.random.normal(0, 0.5, 2))
    np.random.seed(9)
    b = (np.random.normal(0, 0.5, 3), FR.legacy_normal(0.5, 12).reshape(4, 3), np.random.normal(0, 0.5, 2))
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    # from the generator state the reference run itself was in right before its frame loop (golden scan_C3.npz)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scan_C3.npz"))
    state = ('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached']))
    np.random.set_state(state); w = np.random.normal(0, 0.02, (100_003, 3)); w2 = np.random.normal(0, 0.02, 7)
    np.random.set_state(state); v = FR.legacy_normal(0.02, 300_009).reshape(-1, 3); v2 = np.random.normal(0, 0.02, 7)
    assert w.tobytes() == v.tobytes() and w2.tobytes() == v2.tobytes()
    out = np.empty(10)
    assert FR.legacy_normal(1.0, 10, out=out) is out
    with pytest.raises(ValueError):
        FR.legacy_normal(-1.0, 4)
    with pytest.raises(ValueError):
        FR.legacy_normal(1.0, 4, out=np.empty(5))
    L = _capi.lib()
    assert L.lmc_host_legacy_normal(None, None, None, None, 0.0, 1.0, 4, out.ctypes.data, 1) == _capi.ERR_INVALID


def test_one_markstein_correction_is_ieee_division(tmp_path):
    """The Mode B kernel forms alpha = a / b (CS:1503; integers a < b < 2^50) as a * RN(1/b) plus ONE Markstein
    correction; oracle/check_div.c compares that sequence with the IEEE division (fma() is exact in libm)."""
    exe = tmp_path / "check_div"
    src = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "check_div.c")
    subprocess.run(["gcc", "-O2", "-o", str(exe), src, "-lm"], check=True)
    r = subprocess.run([str(exe), "3000000"], capture_output=True, text=True, timeout=300)
    n, bad = (int(x) for x in r.stdout.split())
    assert r.returncode == 0 and n > 2e7 and bad == 0


def test_pose_table_is_scipy_exact(golden):
    g = golden("lmc_edge.npz")
    assert np.array_equal(FR.pose_table(g['pose_position'], g['pose_euler']), orc.pose_table_np(g['pose_position'], g['pose_euler']))
    rng = np.random.default_rng(0)
    from scipy.spatial.transform import Rotation
    q = Rotation.from_euler('xyz', rng.normal(0, 1, (50, 3))).as_quat()
    pos = rng.normal(0, 10, (50, 3))
    ts = np.cumsum(rng.integers(1, 9_000_000, 50)).astype(np.int64)
    assert np.array_equal(FR.slerp_segment_table(q, pos, ts), orc.slerp_segment_table(q, pos, ts))


def test_partition_frames_balances_points():
    rng = np.random.default_rng(1)
    counts = rng.integers(0, 3000, 1000); counts[::7] = 0
    off = np.concatenate([[0], np.cumsum(counts)])
    for W in (1, 2, 3, 8):
        cuts = FR.partition_frames(off, W)
        assert cuts[0] == 0 and cuts[-1] == 1000 and np.all(np.diff(cuts) >= 0) and len(cuts) == W + 1
        per = np.diff(off[cuts])
        assert per.sum() == off[-1] and per.max() - per.min() <= 2 * 3000
    off = np.arange(36001) * 10000
    assert np.array_equal(np.diff(FR.partition_frames(off, 8)), np.full(8, 4500))


def test_lvx_container_bytes_equal_reference_file(golden):
    g = golden("lvx_file.npz")
    rec, flags = orc.C.quantize_lvx_type2(g['raw'])          # records from the (pinned) oracle: no GPU needed here
    assert flags == 0
    data = build_lvx_v11_file(rec, g['frame_off'], g['timestamps'], np.arange(len(g['frame_off']) - 1))
    assert np.array_equal(data, g['file_bytes'])
    pk, pos = frame_layout(g['frame_off'])
    assert pos[0] == FILE_HEADER == 88 and pk.tolist() == [0, 1, 1, 1, 2, 3, 0, 1]
    with pytest.raises(ValueError):
        build_lvx_v11_file(np.zeros((0, 14), np.uint8), np.array([0]), np.array([]), np.array([]))


GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["LMC_ROOT"])
import numpy as np, torch, torch.distributed as dist
from livox_motion_compensation_sim_b200 import frames as FR
from livox_motion_compensation_sim_b200.sharding import shard_ranges, all_gather_merged
from oracle import lmc_oracle as orc
dist.init_process_group("gloo")
rank, W = dist.get_rank(), dist.get_world_size()
for case in ("ragged", "equal"):
    rng = np.random.default_rng(7)
    F = 64
    counts = rng.integers(0, 500, F) if case == "ragged" else np.full(F, 128)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    N = int(off[-1])
    pts = np.column_stack([rng.uniform(-90, 90, (N, 3)), rng.uniform(0, 1, N)])
    pose = orc.pose_table_np(rng.uniform(-30, 30, (F, 3)), rng.normal(0, 0.5, (F, 3)))
    whole = orc.C.align_rigid_f64(pts, off, pose)
    rec_whole, _ = orc.C.quantize_lvx_type2(pts)
    fcuts, pcuts = shard_ranges(off, W)
    a, b = int(fcuts[rank]), int(fcuts[rank + 1])
    # this rank computes only its frame range (the CPU oracle stands in for the kernel: host-logic test)
    merged = torch.zeros((N, 4), dtype=torch.float64)
    lvx = torch.zeros((N, 14), dtype=torch.uint8)
    u16 = torch.zeros(N, dtype=torch.uint16)
    sl = slice(int(pcuts[rank]), int(pcuts[rank + 1]))
    loc_off = off[a:b + 1] - off[a]
    merged[sl] = torch.from_numpy(orc.C.align_rigid_f64(pts[sl], loc_off, pose[a:b]))
    lvx[sl] = torch.from_numpy(rec_whole[sl])
    u16[sl] = torch.from_numpy((np.arange(N)[sl] % 65536).astype(np.uint16))
    all_gather_merged([merged, lvx, u16, None], pcuts)
    assert merged.numpy().tobytes() == whole.tobytes(), case          # == np.vstack order, no permutation
    assert np.array_equal(lvx.numpy(), rec_whole), case
    assert np.array_equal(u16.numpy(), (np.arange(N) % 65536).astype(np.uint16)), case
dist.destroy_process_group()
print("OK", rank)
'''


def test_frame_sharded_merge_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, LMC_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29617", str(script)],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("OK") == 2


GLOO_FILES_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["LMC_ROOT"])
import numpy as np, torch, torch.distributed as dist
from livox_motion_compensation_sim_b200 import sharding
from livox_motion_compensation_sim_b200.lvx import build_lvx_v11_file, frame_layout
from oracle import lmc_oracle as orc
dist.init_process_group("gloo")
rank, W = dist.get_rank(), dist.get_world_size()
out_dir = os.environ["LMC_OUT"]
rng = np.random.default_rng(11)
F = 37
counts = rng.integers(0, 300, F); counts[5] = 0
off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
N = int(off[-1])
pts = np.column_stack([rng.uniform(-90, 90, (N, 3)), rng.uniform(0, 1, N)])
ts, ids = np.arange(F) * 0.1, np.arange(F, dtype=np.int64)
fcuts, pcuts = sharding.shard_ranges(off, W)
a, b = int(fcuts[rank]), int(fcuts[rank + 1])
# LVX v1.1: closed-form offsets, no exchange.  (Host-logic test: the CPU restatement stands in for the kernel; each rank cuts
# ITS byte range out of the image and writes it at ITS offset.)
whole = build_lvx_v11_file(orc.C.quantize_lvx_type2(pts)[0], off, ts, ids)
_, fpos = frame_layout(off)
pos0 = 0 if a == 0 else int(fpos[a])
mine = whole[pos0:int(fpos[b])]
path = os.path.join(out_dir, "sharded.lvx")
assert sharding.pwrite_range(path, pos0, mine) == len(mine)
# variable-length text: sizes all-gathered, offsets by prefix sum, rank 0 owns the header
lines = ["%.6f %.6f %.6f %.6f\n" % tuple(r) for r in pts]
text_mine = "".join(lines[int(pcuts[rank]):int(pcuts[rank + 1])]).encode()
header = b"# header of %d points\n" % N
sizes = sharding.all_gather_sizes(len(text_mine), torch.device("cpu"))
offs = sharding.file_offsets(sizes, len(header))
tpath = os.path.join(out_dir, "sharded.pcd")
if rank == 0:
    sharding.pwrite_range(tpath, 0, header)
sharding.pwrite_range(tpath, int(offs[rank]) + (len(header) if rank == 0 else 0), text_mine)
dist.barrier()
if rank == 0:
    assert open(path, "rb").read() == whole.tobytes()
    assert open(tpath, "rb").read() == header + "".join(lines).encode()
    assert int(offs[-1]) == len(header) + sum(len(l) for l in lines)
dist.destroy_process_group()
print("OK", rank)
'''


def test_sharded_file_writers_gloo_world2(tmp_path):
    """SURVEY 8e, replication-free file production: every rank pwrite()s its own byte range (closed-form LVX offsets;
    all-gathered text sizes) and the result is the single-writer file."""
    script = tmp_path / "worker_files.py"
    script.write_text(GLOO_FILES_WORKER)
    env = dict(os.environ, LMC_ROOT=ROOT, MASTER_ADDR="127.0.0.1", LMC_OUT=str(tmp_path))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29619", str(script)],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("OK") == 2


def test_file_offsets():
    from livox_motion_compensation_sim_b200.sharding import file_offsets
    assert file_offsets([10, 0, 5], 7).tolist() == [0, 17, 17, 22]
    assert file_offsets([3], 0).tolist() == [0, 3]


def test_lvx_cs_host_layout_and_errors():
    """Host side of the complete simulator's LVX writer mirror (CS:235-374): prefixes, frame flattening, the
    struct.pack errors the reference raises before any byte is written."""
    import struct
    from livox_motion_compensation_sim_b200 import lvx
    from livox_motion_compensation_sim_b200.compensator import LiDARPoint
    di = lvx.DeviceInfo("SN123", 1, "fw", True, 0.1, 0.2, 0.3, 1.0, 2.0, 3.0)
    p2 = lvx.lvx_cs_prefix("lvx2", di, 7)
    assert len(p2) == 88 and p2[:10] == b"livox_tech" and p2[10:15] == b"2.0.0" and struct.unpack_from('<I', p2, 16)[0] == 0xAC0EA767
    assert struct.unpack_from('<II', p2, 24) == (50, 1) and p2[32:37] == b"SN123" and p2[48] == 1 and p2[49] == 1
    assert struct.unpack_from('<6f', p2, 50) == struct.unpack('<6f', struct.pack('<6f', 0.1, 0.2, 0.3, 1.0, 2.0, 3.0))
    assert lvx.lvx_cs_prefix("lvx3", di, 7) == p2
    p1 = lvx.lvx_cs_prefix("lvx", di, 7)
    assert len(p1) == 60 and p1[:10] == b"livox_file" and struct.unpack_from('<II', p1, 10) == (1, 7) and p1[44] == 1
    with pytest.raises(ValueError):
        lvx.lvx_cs_prefix("lvx9", di, 1)
    with pytest.raises(ValueError):
        lvx.LivoxLVXWriter("lvx9")
    frames = [{'points': [LiDARPoint(1.0, 2.0, 3.0, 7, 0, 0, 2)], 'timestamp': 5}, {'points': [], 'timestamp': 6},
              {'points': np.array([[4.0, 5.0, 6.0, 9.0, 1.0]]), 'timestamp': 7}]
    pts, tag, off, ts = lvx.frames_to_arrays(frames)
    assert off.tolist() == [0, 1, 1, 2] and ts.tolist() == [5, 6, 7] and tag.tolist() == [2, 1]
    assert np.array_equal(pts, [[1, 2, 3, 7], [4, 5, 6, 9]])
    with pytest.raises(struct.error):
        lvx.frames_to_arrays([{'points': [LiDARPoint(0.0, 0.0, 0.0, 1, 0, 0, 256)], 'timestamp': 0}])
    with pytest.raises(struct.error):
        lvx.frames_to_arrays([{'points': [], 'timestamp': -1}])


def test_exporter_merge_frames():
    from livox_motion_compensation_sim_b200 import exporter
    from livox_motion_compensation_sim_b200.compensator import LiDARPoint
    frames = [{'points': [LiDARPoint(1.0, 2.0, 3.0, 7, 11, 0, 2)]}, {'points': []}, {'points': np.arange(10.0).reshape(2, 5)}]
    m = exporter.merge_frames(frames)
    assert m.shape == (3, 5) and m[0].tolist() == [1.0, 2.0, 3.0, 7.0, 11.0] and m[2, 4] == 9.0
    assert exporter.merge_frames([]).shape == (0, 5)
    assert exporter.PCD_HEADER.format(n=3).count("3") == 2 and exporter.CSV_HEADER == "x,y,z,intensity,timestamp\n"


def _text_digit_table(src):
    m = re.search(r"kTextT\[10\]\[20\]\s*=\s*\{(.*?)\n\};", src, re.S)
    rows = re.findall(r"\{([^{}]*)\}", m.group(1))
    return [[float.fromhex(t.strip()) if "x" in t else float(t) for t in r.split(",")] for r in rows]


def test_pcd_digit_count_thresholds_are_exact():
    """csrc/lmc_pcd.cu: the length of '%.6f' is decided by comparing |v| with kDigitT[k-1] = the smallest double >= 10^k - 5e-7
    (the real threshold is never a double, so the comparison is exact).  The four constants are the '%.6f' row of the text
    writer's kTextT (whose exact derivation is checked below); check the boundary doubles against CPython's formatting."""
    import math
    src = open(os.path.join(ROOT, "livox_motion_compensation_sim_b200", "csrc", "lmc_pcd.cu")).read()
    m = re.search(r"kDigitT\[4\]\s*=\s*\{([^}]*)\}", src)
    consts = [float.fromhex(t.strip()) for t in m.group(1).split(",")]
    assert consts == _text_digit_table(src)[6][1:5]
    for k, c in enumerate(consts, start=1):
        below = math.nextafter(c, 0.0)
        assert "%.6f" % c == "1" + "0" * k + ".000000" and "%.6f" % below == "9" * k + ".999999"
        assert len("%.6f" % -c) == k + 9 and len("%.6f" % -below) == k + 8


def test_text_digit_count_table_is_exact():
    """csrc/lmc_pcd.cu: kTextT[d][k] = the smallest double >= 10^k - 0.5 * 10^-d, and the exponent-based choice of k
    (text_nd): re-derive all 190 constants with exact fractions, check the boundary doubles against CPython's formatting,
    and replay text_nd on the host for random magnitudes and every d."""
    import math
    from fractions import Fraction
    src = open(os.path.join(ROOT, "livox_motion_compensation_sim_b200", "csrc", "lmc_pcd.cu")).read()
    T = _text_digit_table(src)
    assert len(T) == 10 and all(len(r) == 20 for r in T)
    for d in range(10):
        for k in range(1, 20):
            thr = Fraction(10) ** k - Fraction(1, 2) / Fraction(10) ** d
            c = T[d][k]
            below = math.nextafter(c, 0.0)
            assert Fraction(below) < thr <= Fraction(c), (d, k)
            assert len(("%%.%df" % d) % c) == k + 1 + (d + 1 if d else 0), (d, k)
            assert len(("%%.%df" % d) % below) == k + (d + 1 if d else 0), (d, k)

    def text_nd(a, d):
        e = (struct.unpack("<Q", struct.pack("<d", a))[0] >> 52 & 0x7ff) - 1023
        k0 = (e * 1233) >> 12 if e > 0 else 0
        return k0 + 1 + (1 if a >= T[d][k0 + 1] else 0)
    import struct
    rng = np.random.default_rng(5)
    vals = np.concatenate([10.0 ** rng.uniform(-12, 19.2, 20000), [0.0, 0.5, 1.5, 2.5, 9.5, 0.95, 0.995, 5e-324, 2.0 ** 63, 2.0 ** 64 - 2048.0],
                           [math.nextafter(10.0 ** k, 0.0) for k in range(1, 20)], [10.0 ** k for k in range(0, 20)]])
    for d in range(10):
        for a in vals[:: (1 if d in (0, 6) else 7)]:
            txt = ("%%.%df" % d) % a
            assert text_nd(float(a), d) == len(txt.split(".")[0]), (a, d, txt)


def test_nvtx_spans_are_off_by_default_and_balanced():
    """_trace: ranges only when enabled (LMC_NVTX=1 / enable()); a raising body still closes its range."""
    from livox_motion_compensation_sim_b200 import _trace
    assert not _trace.enabled() or os.environ.get("LMC_NVTX", "0") not in ("", "0")
    calls = []

    @_trace.traced("t.f")
    def f(x):
        calls.append(_trace.depth())
        if x < 0:
            raise ValueError("neg")
        return x + 1
    was = _trace.enabled()
    try:
        _trace.enable(False)
        assert f(1) == 2 and calls[-1] == 0
        import torch
        pushed = []
        orig = torch.cuda.nvtx.range_push, torch.cuda.nvtx.range_pop
        torch.cuda.nvtx.range_push = lambda name: pushed.append(name)
        torch.cuda.nvtx.range_pop = lambda: pushed.append("pop")
        try:
            _trace.enable(True)
            assert f(2) == 3 and calls[-1] == 1
            with pytest.raises(ValueError):
                f(-1)
            assert _trace.depth() == 0 and pushed == ["t.f", "pop", "t.f", "pop"]
        finally:
            torch.cuda.nvtx.range_push, torch.cuda.nvtx.range_pop = orig
    finally:
        _trace.enable(was)


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver's reference arm) needs no GPU: one bounded step of the reference's own code path
    (oracle/_ref when staged, else the oracle port) -> ONE JSON line with the B200 arm's metric / unit / config.workload."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(root, "BASELINE.json")))
    assert d["impl"] == "reference" and d["steps"] == 1 and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert d["unit"] == "points/s" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["metric"] in base["metric"] or base["metric"] in d["metric"] or "points" in d["metric"]
    assert "360000000 points" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    from oracle import make_ref
    assert cb["kind"] == ("reference" if make_ref.available() else "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_under_torchrun_prints_one_line():
    """The driver launches the reference arm like the B200 arm (torchrun, one rank per GPU): rank 0 alone runs and prints it."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29557", os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
