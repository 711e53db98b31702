"""Sensor-frame deskew (lmc_deskew_slerp_local_*) and the pose at a time (lmc_slerp_pose_at).

CPU: the C oracle against an independent SciPy restatement (Slerp + np.interp, then R_ref^-1 (R(t) p + x(t) - x_ref)), the
pose oracle against Slerp and the golden lerp, the launch plan's routing of the new mode, and the library's k_fused /
k_stream instantiations of the mode against the kernels this file's GPU table names.
GPU: every new kernel against the oracle on a stream built as test_kernel_variants builds it (empty and one-point frames,
tiles with 0 / 1 / many boundaries, clamps, an edge-value block), plus the properties that make the output a sensor-frame
cloud: a stationary trajectory changes nothing, align_rigid at the reference pose gives Mode C's world cloud back, raw
points generated from a static world come out as that world seen from the reference pose, and UTM-scale positions cost the
f32 layout nothing."""
import ctypes
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
from oracle import lmc_oracle_local as orl                                # noqa: E402  (checker only)
from tests.test_launch_plan import (ERR_INVALID, GEN, LVX, LVX2, LVX2_OF_OUTPUT, LVX_TYPE2_OF_INPUT, OK, OUT, SMS,  # noqa: E402
                                    plan, row)  # noqa: F401  (plan is a fixture)

LOCAL = 4                                                                  # lmc::kSlerpLocal
TOL_M = 1e-4                                                               # Mode C's f32 bar (test_kernel_variants)


def tile_points_local(f64):
    return 960 if f64 else 1920


# ------------------------------------------------------------------------------------------
# CPU: the definition
# ------------------------------------------------------------------------------------------
def _random_trajectory(rng, S, max_angle):
    """S samples with ragged spacing (1..9 ms), random rotations whose consecutive relative angle reaches max_angle."""
    from scipy.spatial.transform import Rotation
    sample_ts = np.cumsum(rng.integers(1_000_000, 9_000_000, S)).astype(np.int64) + 10 ** 12
    steps = Rotation.from_rotvec(rng.normal(0, 1, (S, 3)) * (max_angle * rng.uniform(0.2, 1.0, (S, 1))) / np.sqrt(3))
    rots = [Rotation.from_rotvec(rng.normal(0, 1, 3))]
    for k in range(1, S):
        rots.append(rots[-1] * steps[k])
    quat = np.array([r.as_quat() for r in rots])
    pos = np.cumsum(rng.normal(0, 0.1, (S, 3)), axis=0) + rng.normal(0, 50, 3)
    return sample_ts, quat, pos


def _frames(rng, sample_ts, n_frames=40):
    """Frames over (and beyond) the sample span; the first and last frames lie entirely outside it."""
    span = max(sample_ts[-1] - sample_ts[0], 50_000_000)
    counts = rng.integers(0, 60, n_frames)
    counts[rng.integers(0, n_frames, 3)] = 1
    off = np.zeros(n_frames + 1, np.int64)
    np.cumsum(counts, out=off[1:])
    fstart = np.sort(rng.integers(sample_ts[0] - span // 5, sample_ts[-1] + span // 5, n_frames)).astype(np.int64)
    fstart[0], fstart[-1] = sample_ts[0] - 50_000_000, sample_ts[-1] + 10_000_000
    ts = np.concatenate([fstart[f] + np.sort(rng.integers(0, 20_000_000, counts[f])) for f in range(n_frames)]).astype(np.int64)
    pts = np.column_stack([rng.uniform(-40, 40, (len(ts), 3)), rng.uniform(0, 1, len(ts))])
    ref_ts = fstart + rng.integers(-30_000_000, 30_000_000, n_frames)
    return pts, ts, off, ref_ts


@pytest.mark.parametrize("S,max_angle,seed", [(50, 0.05, 1), (80, 0.6, 2), (2, 0.3, 3), (1, 0.0, 4)],
                         ids=["small-angles", "sincos-tier", "two-samples", "one-sample"])
def test_oracle_vs_scipy(S, max_angle, seed):
    rng = np.random.default_rng(seed)
    sample_ts, quat, pos = _random_trajectory(rng, S, max_angle)
    pts, ts, off, ref_ts = _frames(rng, sample_ts)
    assert (ts < sample_ts[0]).any() and (ts > sample_ts[-1]).any()
    assert (ref_ts < sample_ts[0]).any() and (ref_ts > sample_ts[-1]).any()
    seg = orc.slerp_segment_table(quat, pos, sample_ts)
    if S > 2:
        assert seg[:-1, 15].max() > (0.5 if max_angle > 0.5 else 0.0)      # the library-sincos tier is reached where asked
    ref = orl.C.slerp_pose_at(sample_ts, seg, ref_ts)
    got = orl.C.deskew_slerp_local_f64(pts, ts, off, sample_ts, seg, ref)
    want = orl.slerp_deskew_local_scipy(pts, ts, off, sample_ts, quat, pos, ref_ts)
    assert np.abs(got[:, :3] - want[:, :3]).max(initial=0.0) <= 1e-9
    assert np.array_equal(got[:, 3], pts[:, 3])


def test_pose_at_vs_scipy_and_golden_lerp(golden):
    rng = np.random.default_rng(7)
    sample_ts, quat, pos = _random_trajectory(rng, 60, 0.6)
    seg = orc.slerp_segment_table(quat, pos, sample_ts)
    q = np.concatenate([rng.integers(sample_ts[0] - 10 ** 8, sample_ts[-1] + 10 ** 8, 500), sample_ts]).astype(np.int64)
    got = orl.C.slerp_pose_at(sample_ts, seg, q)
    R, x = orl.slerp_pose_scipy(sample_ts, quat, pos, q)
    assert np.abs(got[:, :9] - R.as_matrix().reshape(-1, 9)).max() <= 1e-12
    assert np.abs(got[:, 9:] - x).max() <= 1e-9
    # position columns: the reference's own np.interp trajectory (identity orientations), to Mode C's lerp bar
    g = golden("modec_lerp.npz")
    S = len(g['sample_ts'])
    seg = orc.slerp_segment_table(np.tile([0.0, 0.0, 0.0, 1.0], (S, 1)), g['sample_pos'], g['sample_ts'])
    got = orl.C.slerp_pose_at(g['sample_ts'], seg, g['ts'])
    assert np.abs(got[:, 9:] - g['ref_position']).max() <= 1e-9
    assert np.array_equal(got[:, :9], np.tile(np.eye(3).reshape(9), (len(g['ts']), 1)))
    # align_rigid with the rows is Mode A at the interpolated pose: one point per query is Mode C at that time
    pts = np.column_stack([rng.uniform(-30, 30, (len(q), 3)), np.zeros(len(q))])
    seg = orc.slerp_segment_table(quat, pos, sample_ts)
    rows = orl.C.slerp_pose_at(sample_ts, seg, q)
    a = np.concatenate([orc.C.align_rigid_f64(np.repeat(p[None], 2, 0), np.array([0, 2], np.int64), r[None])[:1] for p, r in zip(pts, rows)])
    c = orc.C.deskew_slerp_f64(pts, q, np.array([0, len(q)], np.int64), sample_ts, seg)
    assert np.abs(a - c).max() <= 1e-12


# ------------------------------------------------------------------------------------------
# CPU: routing (csrc/lmc_plan.h, driven like test_launch_plan)
# ------------------------------------------------------------------------------------------
def _case(f64, path, ex, n_tiles, **kw):
    out, lvx14, lvx_mode, las_x, las_int = ex
    tp = tile_points_local(f64)
    c = dict(f64=f64, mode=LOCAL, path=path, p_begin=tp + 7, p_end=tp + (n_tiles - 1) * tp + 1, ts=1,
             tag=1 if lvx14 and lvx_mode == LVX2_OF_OUTPUT else 0, out=out, lvx14=lvx14, las_x=las_x, las_int=las_int,
             lvx_mode=lvx_mode, n_peers=0, mc=0, hold_idx=0, frame_start=1, n_samp=720_001)
    c.update(kw)
    return c


EXPORTS = {
    "out": ((1, 0, 0, 0, 0), OUT),
    "out+lvx2": ((1, 1, LVX2_OF_OUTPUT, 0, 0), OUT | LVX | LVX2),
    "out+lvx": ((1, 1, LVX_TYPE2_OF_INPUT, 0, 0), GEN),
    "out+las": ((1, 0, 0, 1, 1), GEN),
    "lvx2": ((0, 1, LVX2_OF_OUTPUT, 0, 0), GEN),
    "out+lvx2+las": ((1, 1, LVX2_OF_OUTPUT, 1, 1), GEN),
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
                    rows.append(_case(f64, path, ex, n_tiles, n_samp=1))
                    want.append((OK, int(stream), GEN if stream else 0, n_tiles))
                    rows.append(_case(f64, path, ex, n_tiles, frame_start=0))
                    want.append((OK, int(stream), (lean if f64 else GEN) if stream else 0, n_tiles))
                    # no merged cloud of sensor-frame points: peers and multicast are refused on every path
                    rows.append(_case(f64, path, ex, n_tiles, n_peers=1))
                    want.append((ERR_INVALID, 0, 0, n_tiles))
                    rows.append(_case(f64, path, ex, n_tiles, n_peers=1, mc=1))
                    want.append((ERR_INVALID, 0, 0, n_tiles))
    got = plan([row(c) for c in rows])
    assert len(got) == len(rows)
    for c, w, (rc, stream, ex, grid, tile0, n) in zip(rows, want, got):
        assert (rc, stream, ex if stream else 0) == w[:3], (c, (rc, stream, ex))
        if stream:
            assert (tile0, n, grid) == (tile_points_local(c["f64"]), w[3], SMS), c


# ------------------------------------------------------------------------------------------
# The GPU table: one row per new kernel
# ------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    f64: bool
    path: int
    kernel: tuple                  # ("local_fused", f64): k_fused<F64, 4>; ("local_stream", f64, ex): k_stream<F64, 4, ex>
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
        Case(_f64, 0, ("local_fused", _f64), lvx="lvx2+tag", las=True),
        Case(_f64, 2, ("local_stream", _f64, OUT)),
        Case(_f64, 2, ("local_stream", _f64, OUT | LVX | LVX2), lvx="lvx2+tag"),
        Case(_f64, 2, ("local_stream", _f64, OUT | LVX | LVX2), lvx="lvx2"),
        Case(_f64, 2, ("local_stream", _f64, GEN), lvx="t2", las=True),
        Case(_f64, 2, ("local_stream", _f64, GEN), out=False, lvx="lvx2+tag"),
    ]


def test_table_routes_to_its_kernels(plan):
    rows = []
    for c in TABLE:
        ex = (int(c.out), int(c.lvx is not None), LVX2_OF_OUTPUT if c.lvx and c.lvx.startswith("lvx2") else LVX_TYPE2_OF_INPUT,
              int(c.las), int(c.las))
        rows.append(row(_case(c.f64, c.path, ex, 3 * SMS, tag=int(c.lvx == "lvx2+tag"))))
    for c, (rc, stream, ex, *_) in zip(TABLE, plan(rows)):
        assert rc == OK
        assert (("local_stream", c.f64, ex) if stream else ("local_fused", c.f64)) == c.kernel, c.id


def test_table_covers_every_local_kernel():
    """The library's k_fused / k_stream instantiations of mode 4 are exactly the kernels the GPU table names: a variant
    without a row fails."""
    from livox_motion_compensation_sim_b200 import _build
    path = os.environ.get("LMC_B200_LIB", _build.LIB_PATH)
    if not os.path.exists(path):
        pytest.skip(f"{path} is not built")
    exe = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    text = subprocess.run([exe, "-symbols", path], capture_output=True, text=True, check=True, timeout=300).stdout
    built = {("local_fused", f == "1") for f in re.findall(rf"k_fusedILb([01])ELi{LOCAL}EE", text)}
    built |= {("local_stream", f == "1", int(x)) for f, x in re.findall(rf"k_streamILb([01])ELi{LOCAL}ELi(\d+)EE", text)}
    assert built == {c.kernel for c in TABLE}


# ------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------
DEV = "cuda:0"


def _C():
    from livox_motion_compensation_sim_b200 import _capi as C
    return C


@dataclass
class Inputs:
    f64: bool
    n: int
    pts: "torch.Tensor"
    pts64: np.ndarray
    args: tuple                    # device arguments between pts and out: ts, frame_off, frame_start, sample_ts, seg, S, ref_pose
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
    tp = tile_points_local(f64)
    sms = _sm_count()
    rng = np.random.default_rng(4040 + f64)
    edge = _edge_values(f64)
    nb = len(edge)
    n_tiles = sms * (4 + 2) + 4                                   # STAGES + 2 tiles per CTA at least
    N = n_tiles * tp + 1237 + 911 + 2 * tp // 3
    p0 = (int(0.45 * N) // tp) * tp - 45                          # the block straddles a tile boundary
    counts, fb = _counts(rng, N, p0, nb)
    F = len(counts)
    st = synth.make_stream(F, counts, 4040, device=DEV, dtype=torch.float64 if f64 else torch.float32)
    st.pts[p0:p0 + nb] = torch.from_numpy(edge).to(DEV, st.pts.dtype)
    pts64 = st.pts.cpu().numpy().astype(np.float64)
    frame_start = st.frame_start.copy()
    frame_start[fb:fb + 3] += 1000
    fidx = np.repeat(np.arange(F), counts)
    ts64 = frame_start[fidx] + st.ts_off.cpu().numpy().astype(np.int64)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    around = np.concatenate([np.arange(20 * f - 1, 20 * f + 3) for f in range(fb, fb + 3)])
    quat, pos = st.sample_quat.copy(), st.sample_pos.copy()
    quat[around] = [0.0, 0.0, 0.0, 1.0]
    pos[around] = 0.0
    keep = slice(200, len(st.sample_ts) - 200)                    # the stream's first and last second clamp to the end samples
    sample_ts, quat, pos = st.sample_ts[keep], quat[keep], pos[keep]
    seg = FR.slerp_segment_table(quat, pos, sample_ts)
    # reference pose: the pose at the frame's last point (frame start for an empty frame); identity for the edge block
    ref_ts = frame_start.copy()
    full = np.flatnonzero(counts > 0)
    ref_ts[full] = ts64[st.frame_off[full + 1] - 1]
    ref = orl.C.slerp_pose_at(sample_ts, seg, ref_ts)
    ref[fb:fb + 3] = [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]
    want = orl.C.deskew_slerp_local_f64(pts64, ts64, st.frame_off, sample_ts, seg, ref)
    blk = slice(p0, p0 + nb)
    fin = np.isfinite(pts64[blk, :3]).all(axis=1)
    assert np.array_equal(want[blk][fin], pts64[blk][fin], equal_nan=True), "the edge block's transform is not the identity"
    assert (ts64[1237:-911] < sample_ts[0]).any() and (ts64[1237:-911] > sample_ts[-1]).any()
    ts = d(ts64) if f64 else st.ts_off
    args = (ts, d(st.frame_off), d(frame_start), d(sample_ts), d(seg), len(sample_ts), d(ref))
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


def _call(c: Case, x: Inputs, B: Buffers, path, b, e, ref_pose=True, n_samp=None, peers=None, mc=None):
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
    if not ref_pose:
        a[6] = None
    if n_samp is not None:
        a[5] = n_samp
    F = x.args[1].shape[0] - 1
    L = C.lib()
    fn = L.lmc_deskew_slerp_local_f64 if x.f64 else L.lmc_deskew_slerp_local_f32
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
def test_local_kernel_vs_oracle(c: Case, inputs):
    from tests.test_kernel_variants import _all_same, _check_rows, _same   # noqa: F401
    C = _C()
    x = inputs(c.f64)
    b, e = x.b, x.e
    p0, p1 = x.block
    B = Buffers(c, x)
    C.check(_call(c, x, B, c.path, b, e))
    if c.out:
        got = B.out.view[b:e].cpu().numpy()
        _check_rows(c.f64, 2, got, x.want[b:e])                   # Mode C's bars: 1e-10 m (f64), 1e-4 m / 4 roundings (f32)
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
    """Peers, multicast, a NULL reference pose and an empty sample table are bad arguments, on both paths, and nothing is
    written (nor a status bit set)."""
    C = _C()
    x = inputs(f64)
    c = Case(f64, 2, ("local_stream", f64, OUT | LVX | LVX2), lvx="lvx2+tag")
    peer = torch.empty_like(x.pts)
    mc_out, mc_lvx = torch.empty_like(x.pts), torch.empty((x.n, 14), dtype=torch.uint8, device=DEV)
    for path in (0, 2):
        for kw in (dict(peers=peer.data_ptr()), dict(peers=peer.data_ptr(), mc=(mc_out.data_ptr(), mc_lvx.data_ptr())),
                   dict(ref_pose=False), dict(n_samp=0), dict(n_samp=2 ** 31)):
            B = Buffers(c, x)
            assert _call(c, x, B, path, x.b, x.e, **kw) == C.ERR_INVALID, kw
            assert B.flags() == 0
            for g in B.local():
                assert g.untouched_outside(0, 0), kw


@pytest.mark.gpu
def test_pose_at_device_vs_oracle():
    """Positions bit-identical (the same FMA); rotation entries within 1e-14 (device sin / cos polynomials vs libm)."""
    from livox_motion_compensation_sim_b200 import ops, synth
    st = synth.make_stream(30, 100, 5, device=DEV, with_points=False)
    rng = np.random.default_rng(5)
    q = np.concatenate([rng.integers(st.sample_ts[0] - 10 ** 8, st.sample_ts[-1] + 10 ** 8, 20000), st.sample_ts]).astype(np.int64)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    got = ops.slerp_pose_at(d(st.sample_ts), d(st.seg), d(q)).cpu().numpy()
    want = orl.C.slerp_pose_at(st.sample_ts, st.seg, q)
    assert np.array_equal(got[:, 9:], want[:, 9:])
    assert np.abs(got[:, :9] - want[:, :9]).max() <= 1e-14
    # one-sample table: every query is that sample's pose
    one = ops.slerp_pose_at(d(st.sample_ts[:1]), d(st.seg[:1]), d(q[:50])).cpu().numpy()
    assert np.array_equal(one, np.tile(orl.C.slerp_pose_at(st.sample_ts[:1], st.seg[:1], q[:1]), (50, 1)))


def _small_stream(f64, quat=None, pos=None, n_frames=60, ppf=3000, seed=11):
    from livox_motion_compensation_sim_b200 import frames as FR, synth
    st = synth.make_stream(n_frames, ppf, seed, device=DEV, dtype=torch.float64 if f64 else torch.float32)
    quat = st.sample_quat if quat is None else quat
    pos = st.sample_pos if pos is None else pos
    seg = FR.slerp_segment_table(quat, pos, st.sample_ts)
    fidx = np.repeat(np.arange(n_frames), np.diff(st.frame_off))
    ts64 = st.frame_start[fidx] + st.ts_off.cpu().numpy().astype(np.int64)
    return st, seg, ts64, quat, pos


def _local(st, seg, ts64, ref_ts, f64, pts=None, **kw):
    from livox_motion_compensation_sim_b200 import ops
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    pts = st.pts if pts is None else pts
    ref = ops.slerp_pose_at(d(st.sample_ts), d(seg), d(np.asarray(ref_ts, np.int64)))
    out, _ = ops.deskew_slerp_local(pts, d(ts64) if f64 else st.ts_off, d(st.frame_off), d(st.frame_start), d(st.sample_ts),
                                    d(seg), ref, **kw)
    return out, ref


@pytest.mark.gpu
def test_stationary_trajectory():
    """Identity orientation and a constant position: the output is the input bit for bit.  A constant arbitrary orientation:
    within 1e-12 m."""
    from scipy.spatial.transform import Rotation
    st, _, _, _, _ = _small_stream(True)
    S = len(st.sample_ts)
    pos = np.tile([1234.5, -77.25, 3.0], (S, 1))
    for quat, exact in ((np.tile([0.0, 0.0, 0.0, 1.0], (S, 1)), True), (np.tile(Rotation.from_rotvec([0.3, -1.1, 2.0]).as_quat(), (S, 1)), False)):
        st, seg, ts64, _, _ = _small_stream(True, quat, pos)
        for path in (0, 2):
            _C().set_path(path)
            try:
                out, _ = _local(st, seg, ts64, st.frame_start, True)
            finally:
                _C().set_path(_C().PATH_AUTO)
            got, pin = out.cpu().numpy(), st.pts.cpu().numpy()
            if exact:
                assert got.tobytes() == pin.tobytes()
            else:
                assert np.abs(got - pin).max() <= 1e-12


@pytest.mark.gpu
def test_round_trip_to_world():
    """align_rigid(local, slerp_pose_at(ref_ts)) is deskew_slerp's world cloud within 1e-9 m (f64)."""
    from livox_motion_compensation_sim_b200 import ops
    st, seg, ts64, _, _ = _small_stream(True)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    ref_ts = st.frame_start + 50_000_000
    local, ref = _local(st, seg, ts64, ref_ts, True)
    world, _ = ops.align_rigid(local, d(st.frame_off), ref)
    want, _ = ops.deskew_slerp(st.pts, d(ts64), d(st.frame_off), d(st.frame_start), d(st.sample_ts), d(seg))
    assert (world - want).abs().max().item() <= 1e-9


@pytest.mark.gpu
def test_it_deskews_a_static_world():
    """Raw points generated as T(t_i)^-1 W from a static world W come out as T_ref^-1 W: the smear of the motion is gone."""
    st, seg, ts64, _, _ = _small_stream(True)
    rng = np.random.default_rng(12)
    N = st.n_points
    pose_i = orl.C.slerp_pose_at(st.sample_ts, seg, ts64)                 # T(t_i) of every point
    W = pose_i[:, 9:] + rng.uniform(-60, 60, (N, 3))                      # world points around the sensor
    R = pose_i[:, :9].reshape(N, 3, 3)
    raw = np.column_stack([np.einsum('nji,nj->ni', R, W - pose_i[:, 9:]), rng.uniform(0, 1, N)])     # R^T (W - x)
    fidx = np.repeat(np.arange(st.n_frames), np.diff(st.frame_off))
    ref_ts = st.frame_start + 100_000_000                                 # the frame's end
    ref = orl.C.slerp_pose_at(st.sample_ts, seg, ref_ts)
    Rr = ref[fidx, :9].reshape(N, 3, 3)
    want = np.einsum('nji,nj->ni', Rr, W - ref[fidx, 9:])
    out, _ = _local(st, seg, ts64, ref_ts, True, pts=torch.from_numpy(raw).to(DEV))
    got = out.cpu().numpy()
    assert np.abs(got[:, :3] - want).max() <= 1e-9
    # ... where the raw cloud itself is smeared by the motion (12 m/s over a 100 ms frame)
    assert np.abs(raw[:, :3] - want).max() > 0.1


@pytest.mark.gpu
def test_utm_scale_positions():
    """Positions of 5e5 / 4.4e6 / 50 m: the f32-layout output stays within the f32 bar of the f64 oracle, while the two-pass
    composition (Mode C world cloud in f32, then align_rigid with the inverse reference pose) rounds the world position to
    the f32 spacing there.  Prints both errors."""
    from livox_motion_compensation_sim_b200 import ops
    st, _, _, quat, pos = _small_stream(False)
    pos = pos + np.array([5e5, 4.4e6, 50.0])
    st, seg, ts64, _, _ = _small_stream(False, quat, pos)
    ref_ts = st.frame_start + 100_000_000
    out, ref = _local(st, seg, ts64, ref_ts, False)
    pts64 = st.pts.cpu().numpy().astype(np.float64)
    want = orl.C.deskew_slerp_local_f64(pts64, ts64, st.frame_off, st.sample_ts, seg, ref.cpu().numpy())
    err_local = np.abs(out.cpu().numpy().astype(np.float64) - want).max()
    assert err_local <= TOL_M
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    world, _ = ops.deskew_slerp(st.pts, st.ts_off, d(st.frame_off), d(st.frame_start), d(st.sample_ts), d(seg))
    r = ref.cpu().numpy()
    Rt = r[:, :9].reshape(-1, 3, 3).transpose(0, 2, 1)
    inv = np.concatenate([Rt.reshape(-1, 9), -np.einsum('fij,fj->fi', Rt, r[:, 9:])], axis=1)
    two, _ = ops.align_rigid(world, d(st.frame_off), d(inv))
    err_two = np.abs(two.cpu().numpy().astype(np.float64) - want).max()
    print(f"UTM-scale positions (5e5, 4.4e6, 50 m), f32 layout: fused local {err_local:.3e} m, "
          f"two-pass deskew_slerp + align_rigid {err_two:.3e} m")
    assert err_two > 100 * err_local


@pytest.mark.gpu
def test_simulator_deskew_scans_local():
    """deskew_scans_local with 'start', 'end' and an array is the ops-level call with those reference times."""
    from scipy.spatial.transform import Rotation
    from livox_motion_compensation_sim_b200 import LiDARMotionSimulator, ops
    rng = np.random.default_rng(13)
    sim = LiDARMotionSimulator()
    F = 12
    t = np.arange(0, 2.0, 0.005)
    traj = {'time': t, 'position_gps': np.column_stack([12 * t, np.sin(t), 0.1 * t]),
            'orientation_imu': np.column_stack([0.01 * t, np.zeros_like(t), 0.5 * t])}
    counts = rng.integers(0, 400, F)
    counts[3] = 0
    counts[5] = 1
    scans = [{'points_local': np.column_stack([rng.uniform(-20, 20, (m, 3)), rng.uniform(0, 1, m)]), 'timestamp': 0.1 * i + 0.05}
             for i, m in enumerate(counts)]
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(sim.device)  # noqa: E731
    off = np.zeros(F + 1, np.int64)
    np.cumsum(counts, out=off[1:])
    fstart = np.round(np.array([s['timestamp'] for s in scans]) * 1e9).astype(np.int64)
    period = int(round(1e9 / float(sim.config['lidar_fps'])))
    ts = np.concatenate([fstart[i] + (np.arange(m, dtype=np.int64) * period) // max(m, 1) for i, m in enumerate(counts)])
    s_ts = np.round(t * 1e9).astype(np.int64)
    quat = Rotation.from_euler('xyz', traj['orientation_imu']).as_quat()
    seg = ops.build_slerp_table(d(quat), d(traj['position_gps']), d(s_ts))
    flat = d(np.concatenate([s['points_local'] for s in scans]))
    end = fstart.copy()
    end[counts > 0] = ts[off[1:][counts > 0] - 1]
    arr = fstart + rng.integers(-10 ** 7, 10 ** 8, F)
    for reference, ref_ts in (('start', fstart), ('end', end), (arr, arr)):
        got = sim.deskew_scans_local(scans, traj, reference=reference)
        ref = ops.slerp_pose_at(d(s_ts), seg, d(ref_ts))
        want, _ = ops.deskew_slerp_local(flat, d(ts), d(off), d(fstart), d(s_ts), seg, ref)
        assert [len(g) for g in got] == list(counts)
        assert np.concatenate(got).tobytes() == want.cpu().numpy().tobytes()
    with pytest.raises(ValueError):
        sim.deskew_scans_local(scans, traj, reference='middle')
