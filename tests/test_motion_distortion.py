"""Distortion (lmc_distort_slerp_*): world points into the sensor frame of Mode C's pose at each point's own time, and the
simulator's motion-distorted scans built on it (lmc_scan_emit_index, ops.scan_frames(motion=...), 'motion_distortion').

CPU: the C oracle against an independent SciPy restatement (Slerp + np.interp, then R(t)^-1 (W - x(t))) and against Mode C
(deskewing the distorted points gives the world back), the launch plan's routing of the new mode, the library's k_fused /
k_stream instantiations of the mode against the kernels this file's GPU table names, and the simulator's argument checks.
GPU: every new kernel against the oracle on a stream built as test_kernel_variants builds it, the fast and the general route
byte for byte, the refusals, the inverse properties (Mode C and sensor-frame deskew of distorted points), the scanner on a
stationary trajectory, and the C3 golden run with and without motion distortion."""
import ctypes
import json
import os
import re
import shutil
import subprocess
from dataclasses import dataclass
from typing import Optional

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import lmc_oracle as orc                                      # noqa: E402  (checker only)
from oracle import lmc_oracle_distort as odis                             # noqa: E402  (checker only)
from oracle import lmc_oracle_local as orl                                # noqa: E402  (checker only)
from tests.test_launch_plan import (ERR_INVALID, GEN, LVX, LVX2, LVX2_OF_OUTPUT, LVX_TYPE2_OF_INPUT, OK, OUT, SMS,  # noqa: E402
                                    plan, row)  # noqa: F401  (plan is a fixture)
from tests.test_deskew_local import _frames, _random_trajectory        # noqa: E402

DISTORT = 5                                                                # lmc::kSlerpDistort
TOL_M = 1e-4                                                               # Mode C's f32 bar (test_kernel_variants)
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def tile_points_distort(f64):
    return 960 if f64 else 2880                                            # Mode C's tile shape


# ------------------------------------------------------------------------------------------
# CPU: the definition
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,max_angle,seed", [(50, 0.05, 1), (80, 0.6, 2), (2, 0.3, 3), (1, 0.0, 4)],
                         ids=["small-angles", "sincos-tier", "two-samples", "one-sample"])
def test_oracle_vs_scipy_and_mode_c(S, max_angle, seed):
    """Ragged sample spacing (1..9 ms), times before and after the sample span; 1e-9 m against SciPy, and Mode C of the
    distorted points is the world point within 1e-9 m."""
    rng = np.random.default_rng(100 + seed)
    sample_ts, quat, pos = _random_trajectory(rng, S, max_angle)
    W, ts, off, _ = _frames(rng, sample_ts)
    W[:, :3] += pos[0]                                                     # world points around the trajectory
    assert (ts < sample_ts[0]).any() and (ts > sample_ts[-1]).any()
    seg = orc.slerp_segment_table(quat, pos, sample_ts)
    if S > 2:
        assert seg[:-1, 15].max() > (0.5 if max_angle > 0.5 else 0.0)      # the library-sincos tier is reached where asked
    got = odis.C.distort_slerp_f64(W, ts, sample_ts, seg)
    want = odis.distort_slerp_scipy(W, ts, sample_ts, quat, pos)
    assert np.abs(got[:, :3] - want[:, :3]).max(initial=0.0) <= 1e-9
    assert np.array_equal(got[:, 3], W[:, 3])
    back = orc.C.deskew_slerp_f64(got, ts, np.array([0, len(ts)], np.int64), sample_ts, seg)
    assert np.abs(back[:, :3] - W[:, :3]).max(initial=0.0) <= 1e-9


# ------------------------------------------------------------------------------------------
# CPU: routing (csrc/lmc_plan.h, driven like test_launch_plan)
# ------------------------------------------------------------------------------------------
def _case(f64, path, ex, n_tiles, **kw):
    out, lvx14, lvx_mode, las_x, las_int = ex
    tp = tile_points_distort(f64)
    c = dict(f64=f64, mode=DISTORT, path=path, p_begin=tp + 7, p_end=tp + (n_tiles - 1) * tp + 1, ts=1,
             tag=1 if lvx14 and lvx_mode == LVX2_OF_OUTPUT else 0, out=out, lvx14=lvx14, las_x=las_x, las_int=las_int,
             lvx_mode=lvx_mode, n_peers=0, mc=0, hold_idx=0, frame_start=1, n_samp=720_001)
    c.update(kw)
    return c


EXPORTS = {                                                                # one lean kernel: the raw cloud alone
    "out": ((1, 0, 0, 0, 0), OUT),
    "out+lvx2": ((1, 1, LVX2_OF_OUTPUT, 0, 0), GEN),
    "out+lvx": ((1, 1, LVX_TYPE2_OF_INPUT, 0, 0), GEN),
    "out+las": ((1, 0, 0, 1, 1), GEN),
    "lvx2": ((0, 1, LVX2_OF_OUTPUT, 0, 0), GEN),
}


def test_routing(plan):
    rows, want = [], []
    for f64 in (True, False):
        for name, (ex, lean) in EXPORTS.items():
            for path in (0, 1, 2):
                for below in (True, False):
                    n_tiles = 2 * SMS - 1 if below else 2 * SMS             # the size threshold of path 1
                    stream = path == 2 or (path == 1 and not below)
                    rows.append(_case(f64, path, ex, n_tiles))
                    want.append((OK, int(stream), lean if stream else 0, n_tiles))
                    # timestamps / tag bytes the TMA engine cannot read: the direct kernel
                    rows.append(_case(f64, path, ex, n_tiles, ts=2))
                    want.append((OK, 0, 0, n_tiles))
                    if ex[1] and ex[2] == LVX2_OF_OUTPUT:
                        rows.append(_case(f64, path, ex, n_tiles, tag=2))
                        want.append((OK, 0, 0, n_tiles))
                    # lean needs 2 <= n_samp < 2^31 - 1 (and frame_start for f32): otherwise the generic kernel
                    for ns in (1, 2, 2 ** 31 - 1):
                        rows.append(_case(f64, path, ex, n_tiles, n_samp=ns))
                        want.append((OK, int(stream), (lean if ns == 2 else GEN) if stream else 0, n_tiles))
                    rows.append(_case(f64, path, ex, n_tiles, frame_start=0))
                    want.append((OK, int(stream), (lean if f64 else GEN) if stream else 0, n_tiles))
                    # peers and multicast are refused on every path
                    rows.append(_case(f64, path, ex, n_tiles, n_peers=1))
                    want.append((ERR_INVALID, 0, 0, n_tiles))
                    rows.append(_case(f64, path, ex, n_tiles, n_peers=1, mc=1))
                    want.append((ERR_INVALID, 0, 0, n_tiles))
    got = plan([row(c) for c in rows])
    assert len(got) == len(rows)
    for c, w, (rc, stream, ex, grid, tile0, n) in zip(rows, want, got):
        assert (rc, stream, ex if stream else 0) == w[:3], (c, (rc, stream, ex))
        if stream:
            assert (tile0, n, grid) == (tile_points_distort(c["f64"]), w[3], SMS), c


# ------------------------------------------------------------------------------------------
# The GPU table: one row per new kernel
# ------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    f64: bool
    path: int
    kernel: tuple                  # ("distort_fused", f64): k_fused<F64, 5>; ("distort_stream", f64, ex): k_stream<F64, 5, ex>
    out: bool = True
    lvx: Optional[str] = None      # None | "t2" | "lvx2" | "lvx2+tag"
    las: bool = False              # LAS x / y / z + intensity, decimal scales

    @property
    def id(self):
        ex = "+".join(x for x in ("out" if self.out else None, self.lvx, "las" if self.las else None) if x)
        return f"{'f64' if self.f64 else 'f32'}-{ex}-p{self.path}"


TABLE = []
for _f64 in (True, False):
    TABLE += [
        Case(_f64, 0, ("distort_fused", _f64), lvx="lvx2+tag", las=True),
        Case(_f64, 2, ("distort_stream", _f64, OUT)),
        Case(_f64, 2, ("distort_stream", _f64, GEN), lvx="t2", las=True),
        Case(_f64, 2, ("distort_stream", _f64, GEN), lvx="lvx2"),
        Case(_f64, 2, ("distort_stream", _f64, GEN), out=False, lvx="lvx2+tag"),
    ]


def test_table_routes_to_its_kernels(plan):
    rows = []
    for c in TABLE:
        ex = (int(c.out), int(c.lvx is not None), LVX2_OF_OUTPUT if c.lvx and c.lvx.startswith("lvx2") else LVX_TYPE2_OF_INPUT,
              int(c.las), int(c.las))
        rows.append(row(_case(c.f64, c.path, ex, 3 * SMS, tag=int(c.lvx == "lvx2+tag"))))
    for c, (rc, stream, ex, *_) in zip(TABLE, plan(rows)):
        assert rc == OK
        assert (("distort_stream", c.f64, ex) if stream else ("distort_fused", c.f64)) == c.kernel, c.id


def test_table_covers_every_distort_kernel():
    """The library's k_fused / k_stream instantiations of mode 5 are exactly the kernels the GPU table names: a variant
    without a row fails."""
    from livox_motion_compensation_sim_b200 import _build
    path = os.environ.get("LMC_B200_LIB", _build.LIB_PATH)
    if not os.path.exists(path):
        pytest.skip(f"{path} is not built")
    exe = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    text = subprocess.run([exe, "-symbols", path], capture_output=True, text=True, check=True, timeout=300).stdout
    built = {("distort_fused", f == "1") for f in re.findall(rf"k_fusedILb([01])ELi{DISTORT}EE", text)}
    built |= {("distort_stream", f == "1", int(x)) for f, x in re.findall(rf"k_streamILb([01])ELi{DISTORT}ELi(\d+)EE", text)}
    assert built == {c.kernel for c in TABLE}


# ------------------------------------------------------------------------------------------
# CPU: the simulator's argument checks
# ------------------------------------------------------------------------------------------
def test_simulator_refuses_what_it_cannot_distort():
    from livox_motion_compensation_sim_b200 import LiDARMotionSimulator
    sim = LiDARMotionSimulator({'motion_distortion': True})
    assert LiDARMotionSimulator().config['motion_distortion'] is False

    class HostScanner:
        trajectory = {}

        def scan(self, i, t, pose):
            return np.zeros((0, 4))
    with pytest.raises(ValueError, match="motion_distortion"):
        sim.run_simulation(HostScanner())
    with pytest.raises(ValueError, match="env"):
        sim.alignment_error({'raw_scans': [{'points_local': np.zeros((0, 4))}], 'aligned_pointclouds': [np.zeros((0, 4))]})


# ------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------
DEV = "cuda:0"


def _C():
    from livox_motion_compensation_sim_b200 import _capi as C
    return C


def d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@dataclass
class Inputs:
    f64: bool
    n: int
    pts: "torch.Tensor"
    pts64: np.ndarray
    args: tuple                    # device arguments between pts and out: ts, frame_off, frame_start, sample_ts, seg, S
    want: np.ndarray
    tag: "torch.Tensor"
    tag_np: np.ndarray
    block: tuple
    b: int
    e: int
    cuts: tuple


def _make_inputs(f64):
    from livox_motion_compensation_sim_b200 import frames as FR, synth
    from tests.test_kernel_variants import _counts, _edge_values, _sm_count
    tp = tile_points_distort(f64)
    sms = _sm_count()
    rng = np.random.default_rng(5050 + f64)
    edge = _edge_values(f64)
    nb = len(edge)
    n_tiles = sms * (4 + 2) + 4                                   # STAGES + 2 tiles per CTA at least
    N = n_tiles * tp + 1237 + 911 + 2 * tp // 3
    p0 = (int(0.45 * N) // tp) * tp - 45                          # the block straddles a tile boundary
    counts, fb = _counts(rng, N, p0, nb)
    F = len(counts)
    st = synth.make_stream(F, counts, 5050, device=DEV, dtype=torch.float64 if f64 else torch.float32)
    st.pts[p0:p0 + nb] = torch.from_numpy(edge).to(DEV, st.pts.dtype)
    pts64 = st.pts.cpu().numpy().astype(np.float64)
    frame_start = st.frame_start.copy()
    frame_start[fb:fb + 3] += 1000
    fidx = np.repeat(np.arange(F), counts)
    ts64 = frame_start[fidx] + st.ts_off.cpu().numpy().astype(np.int64)
    around = np.concatenate([np.arange(20 * f - 1, 20 * f + 3) for f in range(fb, fb + 3)])
    quat, pos = st.sample_quat.copy(), st.sample_pos.copy()
    quat[around] = [0.0, 0.0, 0.0, 1.0]                           # the edge block's points: the identity transform
    pos[around] = 0.0
    keep = slice(200, len(st.sample_ts) - 200)                    # the stream's first and last second clamp to the end samples
    sample_ts, quat, pos = st.sample_ts[keep], quat[keep], pos[keep]
    seg = FR.slerp_segment_table(quat, pos, sample_ts)
    want = odis.C.distort_slerp_f64(pts64, ts64, sample_ts, seg)
    blk = slice(p0, p0 + nb)
    fin = np.isfinite(pts64[blk, :3]).all(axis=1)
    assert np.array_equal(want[blk][fin], pts64[blk][fin], equal_nan=True), "the edge block's transform is not the identity"
    assert (ts64[1237:-911] < sample_ts[0]).any() and (ts64[1237:-911] > sample_ts[-1]).any()
    ts = d(ts64) if f64 else st.ts_off
    args = (ts, d(st.frame_off), d(frame_start), d(sample_ts), d(seg), len(sample_ts))
    tag_np = rng.integers(0, 256, N).astype(np.uint8)
    b, e = 1237, N - 911
    assert b % tp and e % tp
    cuts = (b, p0 + 71, int(0.7 * N) | 1, e)
    return Inputs(f64, N, st.pts, pts64, args, want, d(tag_np), tag_np, (p0, p0 + nb), b, e, cuts)


@pytest.fixture(scope="module")
def inputs():
    cache = {}

    def get(f64):
        if f64 not in cache:
            cache.clear()
            torch.cuda.empty_cache()
            cache[f64] = _make_inputs(f64)
        return cache[f64]
    return get


LAS_DEC = ((0.001, 0.01, 0.001), (-1.5, 2.0, 1000.0), 1)          # LAS_CFG["dec"] of test_kernel_variants


class Buffers:
    def __init__(self, c: Case, x: Inputs):
        from tests.test_kernel_variants import Guarded
        n, fdt = x.n, torch.float64 if x.f64 else torch.float32
        self.out = Guarded(n, (4,), fdt, -123.0) if c.out else None
        self.lvx = Guarded(n, (14,), torch.uint8, 0xAB) if c.lvx else None
        self.las = [Guarded(n, (), torch.int32, -77) for _ in range(3)] if c.las else None
        self.las_int = Guarded(n, (), torch.int16, 0x5A5A) if c.las else None
        self.status = torch.zeros(1, dtype=torch.int32, device=DEV)

    def local(self):
        return [g for g in [self.out, self.lvx, self.las_int] + (self.las or []) if g is not None]

    def flags(self):
        return int(self.status.item())


def _call(c: Case, x: Inputs, B: Buffers, path, b, e, n_samp=None, peers=None, mc=None):
    C = _C()
    ex = C.LmcExport()
    ex.lvx14 = B.lvx.view.data_ptr() if B.lvx else None
    ex.lvx_mode = LVX2_OF_OUTPUT if c.lvx and c.lvx.startswith("lvx2") else LVX_TYPE2_OF_INPUT
    if c.lvx == "lvx2+tag":
        ex.tag = x.tag.data_ptr()
    for k in range(3):
        ex.las_scale[k], ex.las_offset[k] = (LAS_DEC[0][k], LAS_DEC[1][k]) if c.las else (0.01, 0.0)
    if c.las:
        ex.las_x, ex.las_y, ex.las_z = (g.view.data_ptr() for g in B.las)
        ex.las_intensity = B.las_int.view.data_ptr()
        ex.las_intensity_mode = LAS_DEC[2]
    ex.status = B.status.data_ptr()
    if peers is not None:
        ex.n_peers = 1
        ex.peer_out[0] = peers
    if mc is not None:
        ex.mc_out, ex.mc_lvx14 = mc
    a = [v.data_ptr() if isinstance(v, torch.Tensor) else v for v in x.args]
    if n_samp is not None:
        a[5] = n_samp
    F = x.args[1].shape[0] - 1
    L = C.lib()
    fn = L.lmc_distort_slerp_f64 if x.f64 else L.lmc_distort_slerp_f32
    C.set_path(path)
    try:
        rc = fn(x.pts.data_ptr(), *a, B.out.view.data_ptr() if B.out else None, x.n, F, b, e, ctypes.byref(ex),
                torch.cuda.current_stream().cuda_stream)
    finally:
        C.set_path(C.PATH_AUTO)
    torch.cuda.synchronize()
    return rc


def _device_rows(c: Case, x: Inputs, B: Buffers, b, e):
    """What the LVX2 / LAS quantisers see: the device's own rows (f64), the oracle's (f32, as test_kernel_variants does)."""
    if not c.f64:
        return x.want[b:e]
    if c.out:
        return B.out.view[b:e].cpu().numpy()
    co = Case(**{**c.__dict__, "out": True, "lvx": None, "las": False})
    Bo = Buffers(co, x)
    _C().check(_call(co, x, Bo, c.path, b, e))
    return Bo.out.view[b:e].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("c", TABLE, ids=[c.id for c in TABLE])
def test_distort_kernel_vs_oracle(c: Case, inputs):
    from tests.test_kernel_variants import _all_same, _check_rows
    C = _C()
    x = inputs(c.f64)
    b, e = x.b, x.e
    p0, p1 = x.block
    B = Buffers(c, x)
    C.check(_call(c, x, B, c.path, b, e))
    if c.out:
        got = B.out.view[b:e].cpu().numpy()
        _check_rows(c.f64, 2, got, x.want[b:e])                   # Mode C's bars: 1e-10 m (f64), 1e-4 m (f32)
    rows = _device_rows(c, x, B, b, e)
    want, fl = {}, 0
    if c.lvx == "t2":
        want["lvx"], f = orc.C.quantize_lvx_type2(x.pts64[b:e])
        fl |= f
    elif c.lvx:
        want["lvx"], f = orc.C.quantize_lvx2(rows, x.tag_np[b:e] if c.lvx == "lvx2+tag" else None)
        fl |= f
    if c.las:
        X, Y, Z, I, f = orc.C.quantize_las(rows, LAS_DEC[0], LAS_DEC[1], LAS_DEC[2])
        want["las"], want["las_int"] = (X, Y, Z), I
        fl |= f
    if "lvx" in want:
        got = B.lvx.view[b:e].cpu().numpy()
        bad = np.flatnonzero((got != want["lvx"]).any(axis=1))
        assert bad.size == 0, (b + bad[:5], got[bad[:3]], want["lvx"][bad[:3]])
    if "las" in want:
        for g, w in zip(B.las, want["las"]):
            assert np.array_equal(g.view[b:e].cpu().numpy(), w)
        assert np.array_equal(B.las_int.view[b:e].cpu().numpy().view(np.uint16), want["las_int"])
    assert B.flags() == fl, (B.flags(), fl)
    if c.lvx or c.las:
        assert fl != 0 and b <= p0 and p1 <= e
    for g in B.local():
        assert g.untouched_outside(b, e)
    # the other kernel family: the same bytes, the same status
    B2 = Buffers(c, x)
    C.check(_call(c, x, B2, 2 if c.path == 0 else 0, b, e))
    assert _all_same(B, B2, peers=False) and B2.flags() == B.flags()
    # three odd-cut shards compose to the single launch
    B3 = Buffers(c, x)
    for lo, hi in zip(x.cuts[:-1], x.cuts[1:]):
        C.check(_call(c, x, B3, c.path, lo, hi))
    assert _all_same(B, B3, peers=False) and B3.flags() == B.flags()
    # a range that avoids the edge block reports nothing
    B4 = Buffers(c, x)
    C.check(_call(c, x, B4, c.path, b, p0 - 1))
    assert B4.flags() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [True, False], ids=["f64", "f32"])
def test_refusals_write_nothing(f64, inputs):
    """Peers, multicast and sample tables outside 1 .. 2^31 - 1 rows are bad arguments, on both paths, and nothing is
    written (nor a status bit set)."""
    C = _C()
    x = inputs(f64)
    c = Case(f64, 2, ("distort_stream", f64, GEN), lvx="lvx2+tag")
    peer = torch.empty_like(x.pts)
    mc_out, mc_lvx = torch.empty_like(x.pts), torch.empty((x.n, 14), dtype=torch.uint8, device=DEV)
    for path in (0, 2):
        for kw in (dict(peers=peer.data_ptr()), dict(peers=peer.data_ptr(), mc=(mc_out.data_ptr(), mc_lvx.data_ptr())),
                   dict(n_samp=0), dict(n_samp=2 ** 31)):
            B = Buffers(c, x)
            assert _call(c, x, B, path, x.b, x.e, **kw) == C.ERR_INVALID, kw
            assert B.flags() == 0
            for g in B.local():
                assert g.untouched_outside(0, 0), kw


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [True, False], ids=["f64", "f32"])
def test_fast_and_general_route_same_bytes(f64):
    """One frame of time-ordered points (pairs inside one pose segment: the straight-line route) against the same points
    interleaved with points half the frame away (no pair shares a segment: every point takes the general route), on both
    kernel families: bit-identical rows."""
    from livox_motion_compensation_sim_b200 import ops, synth
    st = synth.make_stream(1, 300_000, 21, device=DEV, dtype=torch.float64 if f64 else torch.float32, point_dt_ns=10_000)
    tb = synth.make_tables(50, 21)                                 # 5 s of pose samples
    n = st.n_points
    fs = np.array([tb['sample_ts'][100] + 777], np.int64)          # the frame spans samples 100 .. 700 (3 s)
    ts_off = st.ts_off.cpu().numpy().astype(np.int64)
    perm = np.empty(2 * n, np.int64)
    perm[0::2] = np.arange(n)
    perm[1::2] = (np.arange(n) + n // 2) % n
    two = lambda a: d(np.asarray(a)[perm])                        # noqa: E731
    sts, seg = d(tb['sample_ts']), d(tb['seg'])
    pts_np = st.pts.cpu().numpy()
    for path in (0, 2):
        _C().set_path(path)
        try:
            if f64:
                a, _ = ops.distort_slerp(st.pts, d(fs[0] + ts_off), d(np.array([0, n])), None, sts, seg)
                g, _ = ops.distort_slerp(two(pts_np), d((fs[0] + ts_off)[perm]), d(np.array([0, 2 * n])), None, sts, seg)
            else:
                a, _ = ops.distort_slerp(st.pts, st.ts_off, d(np.array([0, n])), d(fs), sts, seg)
                g, _ = ops.distort_slerp(two(pts_np), two(st.ts_off.cpu().numpy()), d(np.array([0, 2 * n])), d(fs), sts, seg)
        finally:
            _C().set_path(_C().PATH_AUTO)
        assert a.cpu().numpy().tobytes() == g[0::2].cpu().numpy().tobytes(), path


def _small_stream(quat=None, pos=None, n_frames=60, ppf=3000, seed=11):
    from livox_motion_compensation_sim_b200 import frames as FR, synth
    st = synth.make_stream(n_frames, ppf, seed, device=DEV, dtype=torch.float64)
    quat = st.sample_quat if quat is None else quat
    pos = st.sample_pos if pos is None else pos
    seg = FR.slerp_segment_table(quat, pos, st.sample_ts)
    fidx = np.repeat(np.arange(n_frames), np.diff(st.frame_off))
    ts64 = st.frame_start[fidx] + st.ts_off.cpu().numpy().astype(np.int64)
    return st, seg, ts64


@pytest.mark.gpu
@pytest.mark.parametrize("utm", [False, True], ids=["local", "utm"])
def test_mode_c_inverts_it(utm):
    """deskew_slerp(distort_slerp(W)) is W: within 1e-9 m at local positions; at UTM-scale ones (5e5, 4.4e6, 50 m) within
    4 ulp of the largest world coordinate (2^-30 m there), the rounding of forming W back from its offset."""
    from livox_motion_compensation_sim_b200 import ops, synth
    st0 = synth.make_stream(60, 3000, 11, device=DEV, dtype=torch.float64, with_points=False)
    pos = st0.sample_pos + (np.array([5e5, 4.4e6, 50.0]) if utm else 0.0)
    st, seg, ts64 = _small_stream(pos=pos)
    rng = np.random.default_rng(31)
    pose_i = orl.C.slerp_pose_at(st.sample_ts, seg, ts64)
    W = np.column_stack([pose_i[:, 9:] + rng.uniform(-60, 60, (len(ts64), 3)), rng.uniform(0, 1, len(ts64))])
    args = (d(ts64), d(st.frame_off), None, d(st.sample_ts), d(seg))
    raw, _ = ops.distort_slerp(d(W), *args)
    back, _ = ops.deskew_slerp(raw, *args)
    err = np.abs(back.cpu().numpy()[:, :3] - W[:, :3]).max()
    print(f"Mode C of the distorted points ({'UTM-scale' if utm else 'local'} positions): max |W' - W| = {err:.3e} m")
    assert err <= (4 * 2.0 ** -30 if utm else 1e-9)
    assert np.array_equal(back.cpu().numpy()[:, 3], W[:, 3])
    # the raw points are the oracle's, and local-scale numbers whatever the world position
    want = odis.C.distort_slerp_f64(W, ts64, st.sample_ts, seg)
    assert np.abs(raw.cpu().numpy() - want).max() <= 1e-10
    assert np.abs(raw.cpu().numpy()[:, :3]).max() < 120.0


@pytest.mark.gpu
def test_sensor_frame_deskew_of_distorted_points():
    """deskew_slerp_local(distort_slerp(W), ref) is W seen from the reference pose, R_r^T (W - x_r), within 1e-9 m."""
    from livox_motion_compensation_sim_b200 import ops
    st, seg, ts64 = _small_stream()
    rng = np.random.default_rng(32)
    N = len(ts64)
    pose_i = orl.C.slerp_pose_at(st.sample_ts, seg, ts64)
    W = np.column_stack([pose_i[:, 9:] + rng.uniform(-60, 60, (N, 3)), rng.uniform(0, 1, N)])
    ref_ts = st.frame_start + 100_000_000
    ref = ops.slerp_pose_at(d(st.sample_ts), d(seg), d(ref_ts))
    raw, _ = ops.distort_slerp(d(W), d(ts64), d(st.frame_off), None, d(st.sample_ts), d(seg))
    got, _ = ops.deskew_slerp_local(raw, d(ts64), d(st.frame_off), None, d(st.sample_ts), d(seg), ref)
    r = ref.cpu().numpy()
    fidx = np.repeat(np.arange(st.n_frames), np.diff(st.frame_off))
    want = np.einsum('nji,nj->ni', r[fidx, :9].reshape(N, 3, 3), W[:, :3] - r[fidx, 9:])
    assert np.abs(got.cpu().numpy()[:, :3] - want).max() <= 1e-9
    assert np.abs(raw.cpu().numpy()[:, :3] - want).max() > 0.1               # the raw cloud itself is smeared by the motion


@pytest.mark.gpu
def test_scanner_stationary_trajectory():
    """A trajectory that does not move: index emission + distortion reproduce lmc_scan_emit's raw points within 1e-12 m, the
    frame offsets exactly, and the emitted rows are the environment rows the points came from; the point times follow
    deskew_scans' convention."""
    from scipy.spatial.transform import Rotation
    from livox_motion_compensation_sim_b200 import ops
    rng = np.random.default_rng(33)
    M, F = 80_000, 7
    env = np.column_stack([rng.uniform(-40, 120, M), rng.uniform(-60, 60, M), rng.uniform(-5, 30, M), rng.uniform(0.1, 0.9, M)])
    eul, p = np.array([0.02, -0.05, 0.7]), np.array([3.0, -2.0, 1.5])
    s_ts = np.arange(200, dtype=np.int64) * 5_000_000
    quat = np.tile(Rotation.from_euler('xyz', eul).as_quat(), (len(s_ts), 1))
    seg = ops.build_slerp_table(d(quat), d(np.tile(p, (len(s_ts), 1))), d(s_ts))
    pos, Rm = np.tile(p, (F, 1)), np.tile(Rotation.from_euler('xyz', eul).as_matrix().reshape(9), (F, 1))
    kw = dict(range_max=90.0, range_min=0.05, fov_horizontal=70.0, fov_vertical=77.2, points_per_frame=1500, noise_std=0.0)
    fstart = np.arange(F, dtype=np.int64) * 100_000_000 + 3
    raw0, off0 = ops.scan_frames(d(env), d(pos), d(Rm), **kw)
    raw1, off1, ts1, idx = ops.scan_frames(d(env), d(pos), d(Rm), **kw, motion=(d(s_ts), seg, fstart, 100_000_000),
                                           max_flag_bytes=3 * M)            # frames in chunks of 3
    assert np.array_equal(off0, off1) and off0[-1] > 0 and (np.diff(off0) == 1500).all()
    assert np.abs(raw1.cpu().numpy() - raw0.cpu().numpy()).max() <= 1e-12
    i = idx.cpu().numpy()
    assert np.array_equal(raw0.cpu().numpy()[:, 3], env[i, 3])
    want = np.einsum('ji,nj->ni', Rm[0].reshape(3, 3), env[i, :3] - p)
    assert np.abs(raw0.cpu().numpy()[:, :3] - want).max() <= 1e-12
    fidx = np.repeat(np.arange(F), np.diff(off0))
    m = np.diff(off0)[fidx]
    assert np.array_equal(ts1, fstart[fidx] + ((np.arange(off0[-1]) - off0[fidx]) * 100_000_000) // m)


def _c3_run(golden, **cfg_over):
    from livox_motion_compensation_sim_b200 import LiDARMotionSimulator
    g = golden("scan_C3.npz")
    cfg = json.loads(bytes(g['config_json']).decode())
    vel = np.zeros_like(g['traj_position_gps'])

    class Source:
        trajectory = {'time': g['traj_time'], 'position': g['traj_position_gps'], 'velocity': vel, 'orientation': g['traj_orientation_imu'],
                      'position_gps': g['traj_position_gps'], 'orientation_imu': g['traj_orientation_imu']}
        environment = g['environment']
    sim = LiDARMotionSimulator(dict(cfg, **cfg_over))
    np.random.set_state(('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached'])))
    res = sim.run_simulation(Source)
    return sim, res, np.random.get_state(), g, cfg


def _sha(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.gpu
def test_c3_run_with_motion_distortion(golden):
    """The C3 golden run with 'motion_distortion': the same frames, point sets, environment rows and noise stream as the
    undistorted run (the NumPy RNG ends in the same state), each point observed from the pose at its own time."""
    from scipy.spatial.transform import Rotation
    _, res0, rng0, g, cfg = _c3_run(golden)
    _, res1, rng1, _, _ = _c3_run(golden, motion_distortion=True)
    assert [len(s['points_local']) for s in res0['raw_scans']] == [len(s['points_local']) for s in res1['raw_scans']]
    assert all(np.array_equal(a, b) for a, b in zip(rng0[1:], rng1[1:])) and rng0[0] == rng1[0]
    env = g['environment']
    raw0 = np.vstack([s['points_local'] for s in res0['raw_scans']])
    raw1 = np.vstack([s['points_local'] for s in res1['raw_scans']])
    idx = np.concatenate([s['env_index'] for s in res1['raw_scans']])
    ts = np.concatenate([s['point_times'] for s in res1['raw_scans']])
    assert len(idx) == len(ts) == len(raw1) and raw0.shape == raw1.shape
    # the noise of the undistorted run (its raw points minus the hold-next view of env[idx]) is the noise of the distorted
    # one (its raw points minus the distortion of env[idx]): the same rows, in the same slots, with the same draws
    fidx = np.repeat(np.arange(len(res1['raw_scans'])), [len(s['points_local']) for s in res1['raw_scans']])
    R = Rotation.from_euler('xyz', np.array([s['sensor_pose']['orientation'] for s in res1['raw_scans']])).as_matrix()
    P = np.array([s['sensor_pose']['position'] for s in res1['raw_scans']])
    noise0 = raw0[:, :3] - np.einsum('nji,nj->ni', R[fidx], env[idx, :3] - P[fidx])
    s_ts = np.round(g['traj_time'] * 1e9).astype(np.int64)
    seg = orc.slerp_segment_table(Rotation.from_euler('xyz', g['traj_orientation_imu']).as_quat(), g['traj_position_gps'], s_ts)
    noise1 = raw1[:, :3] - odis.C.distort_slerp_f64(env[idx], ts, s_ts, seg)[:, :3]
    assert np.abs(noise0 - noise1).max() <= 1e-9
    assert np.abs(noise0).max() > 0.01                                          # (the noise is on)
    assert np.array_equal(raw0[:, 3], raw1[:, 3]) and np.array_equal(raw1[:, 3], env[idx, 3])
    # ... and the raw points really moved
    assert np.abs(raw1 - raw0).max() > 0.01


@pytest.mark.gpu
def test_c3_alignment_error(golden):
    """Noise off: Mode C ('slerp') recovers the environment from the distorted scans to 1e-9 m; frame-rigid alignment
    ('hold_next') leaves a residual more than 1000x larger."""
    sim_s, res_s, _, _, _ = _c3_run(golden, motion_distortion=True, lidar_range_noise=0.0, pose_interpolation='slerp')
    sim_h, res_h, _, _, _ = _c3_run(golden, motion_distortion=True, lidar_range_noise=0.0)
    es, eh = sim_s.alignment_error(res_s), sim_h.alignment_error(res_h)
    print(f"C3 with motion distortion, noise off: slerp max {es['max_m']:.3e} m rms {es['rms_m']:.3e} m; "
          f"hold_next max {eh['max_m']:.3e} m rms {eh['rms_m']:.3e} m")
    assert es['max_m'] <= 1e-9
    assert eh['max_m'] > 1000 * max(es['max_m'], 1e-12)
    assert len(es['per_frame_max_m']) == len(res_s['raw_scans']) and max(es['per_frame_max_m']) == es['max_m']


@pytest.mark.gpu
def test_c3_run_motion_distortion_off_is_the_reference(golden, tmp_path):
    """'motion_distortion': False is the default behaviour: the raw and aligned sha256 of the reference run, and every
    output file of save_results as the run without the key writes it."""
    import contextlib
    import hashlib
    import io
    man = json.load(open(os.path.join(GOLDEN, "MANIFEST.json")))['lmc']['C3']
    out = {}
    for name, over in (("absent", {}), ("false", {'motion_distortion': False})):
        sim, res, _, _, _ = _c3_run(golden, **over)
        assert _sha(np.vstack([s['points_local'] for s in res['raw_scans']])) == man['raw_sha256']
        assert _sha(np.vstack(res['aligned_pointclouds'])) == man['aligned_sha256']
        assert all('env_index' not in s and 'point_times' not in s for s in res['raw_scans'])
        with contextlib.redirect_stdout(io.StringIO()):
            dd = sim.save_results(res, str(tmp_path / name))
        files = {}
        for dp, _, fs in os.walk(dd):
            for f in fs:
                files[os.path.relpath(os.path.join(dp, f), dd)] = hashlib.sha256(open(os.path.join(dp, f), 'rb').read()).hexdigest()
        out[name] = files
    assert out["absent"] == out["false"] and len(out["false"]) > 2
