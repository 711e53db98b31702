"""Every point kernel an aligned-cloud call can run -- the 8 direct kernels k_fused<F64, MODE> and the 30 streaming kernels
k_stream<F64, MODE, EX> other than the two multicast ones -- against the oracle, one table row per (layout, mode, export set,
peer set, path).  Each lean streaming variant has its own epilogue in consume_tile (csrc/lmc_tma.cu), so a call routed to it
is only as good as that epilogue: these tests run every one of them.

CPU: each row routes to the kernel it names (plan_point_launch through the driver of test_launch_plan), and the rows name
every such kernel the built library contains.
GPU: per row, a shard [b, e) with mid-tile ends over a stream large enough that every CTA of the persistent grid walks at
least STAGES + 2 tiles.  The stream carries empty and one-point frames, tiles with 0 / 1 / many frame boundaries, a run of
0-3 point frames (the per-point frame search of overflowing tiles) and an edge-value block: frames with an identity
transform, straddling a tile boundary and a shard cut, whose points reach the quantisers unchanged -- LAS exact ties and
near-ties, the int32 ends of the LAS range, the type-2 LVX clip, out-of-range intensities, NaN, +-inf and signed zeros.
Checked: rows, integer exports (exact), the status word, nothing written outside [b, e) or the buffers, the other path,
composing shards, and peer copies (any device pointer is a valid peer, so local buffers stand in for other ranks)."""
import ctypes
import os
import re
import shutil
import subprocess
from dataclasses import dataclass
from typing import Optional

import numpy as np
import pytest

from tests.test_launch_plan import (GEN, GYRO, LAS, LVX, LVX2, LVX2_OF_OUTPUT, LVX_TYPE2_OF_INPUT, MC, OUT, PB, QUANT, RIGID,
                                    SLERP, plan, row, tile_points)  # noqa: F401  (plan is a fixture)

torch = pytest.importorskip("torch")

from livox_motion_compensation_sim_b200 import _build                      # noqa: E402
from livox_motion_compensation_sim_b200 import _capi as C                  # noqa: E402
from oracle import lmc_oracle as orc                                      # noqa: E402  (checker only)

DEV = "cuda:0"
TOL_M = 1e-4
MODE_NAMES = {RIGID: "rigid", GYRO: "gyro", SLERP: "slerp", QUANT: "quant"}

# LAS configurations.  POW2: power-of-two scales and dyadic offsets, so that (v - offset) / scale is exact and a tie in
# the input is a tie for the rounding (round-half-even is decided by the kernel, not by an f64 rounding).  DEC: decimal
# scales with non-zero offsets, whose near-ties take the exact route of q_las.
LAS_CFG = {
    "pow2": ((0.25, 2.0 ** -10, 2.0 ** -10), (0.0, 0.5, -3.25), C.LAS_INTENSITY_UNIT),
    "dec": ((0.001, 0.01, 0.001), (-1.5, 2.0, 1000.0), C.LAS_INTENSITY_RAW),
}


@dataclass(frozen=True)
class Case:
    f64: bool
    mode: int
    path: int                      # lmc_set_path: 0 direct, 2 streaming
    kernel: tuple                  # ("fused", f64, mode) or ("stream", f64, mode, ex)
    out: bool = True
    lvx: Optional[str] = None      # None | "t2" (type-2 of the input) | "lvx2" | "lvx2+tag" (records of the output)
    las: Optional[str] = None      # None | a LAS_CFG key (x / y / z + intensity) | "int:<key>" (intensity only)
    peers: int = 0                 # 0, 1, or 7 with a NULL entry in the middle

    @property
    def id(self):
        ex = "+".join(x for x in ("out" if self.out else None, self.lvx, self.las and "las:" + self.las) if x)
        return f"{'f64' if self.f64 else 'f32'}-{MODE_NAMES[self.mode]}-{ex}-p{self.path}" + (f"-peers{self.peers}" if self.peers else "")


def _fused(f64, mode):
    return ("fused", f64, mode)


def _stream(f64, mode, ex):
    return ("stream", f64, mode, ex)


def _table():
    rows = []
    for f64 in (True, False):
        rigid = lambda **kw: Case(f64=f64, mode=RIGID, **kw)         # noqa: E731
        rows += [
            rigid(path=0, lvx="t2", las="pow2", kernel=_fused(f64, RIGID)),
            rigid(path=2, kernel=_stream(f64, RIGID, OUT)),
            rigid(path=2, lvx="t2", kernel=_stream(f64, RIGID, OUT | LVX)),
            rigid(path=2, las="pow2", kernel=_stream(f64, RIGID, OUT | LAS)),
            rigid(path=2, las="dec", kernel=_stream(f64, RIGID, OUT | LAS)),
            rigid(path=2, lvx="lvx2+tag", kernel=_stream(f64, RIGID, GEN)),      # LVX2 records on Mode A: generic
            rigid(path=2, out=False, lvx="t2", kernel=_stream(f64, RIGID, GEN)),  # records without the aligned cloud
            rigid(path=2, lvx="t2", las="dec", kernel=_stream(f64, RIGID, GEN)),
        ]
        gyro = lambda **kw: Case(f64=f64, mode=GYRO, **kw)           # noqa: E731
        rows += [
            gyro(path=0, lvx="lvx2+tag", las="dec", kernel=_fused(f64, GYRO)),
            gyro(path=0, lvx="t2", kernel=_fused(f64, GYRO)),                      # the direct kernel's type-2 branch of Mode B
            gyro(path=2, kernel=_stream(f64, GYRO, OUT)),
            gyro(path=2, lvx="t2", kernel=_stream(f64, GYRO, OUT | LVX)),
            gyro(path=2, las="pow2", kernel=_stream(f64, GYRO, OUT | LAS)),
            gyro(path=2, lvx="lvx2", kernel=_stream(f64, GYRO, OUT | LVX | LVX2)),
            gyro(path=2, lvx="lvx2+tag", kernel=_stream(f64, GYRO, OUT | LVX | LVX2)),
            gyro(path=2, lvx="t2", las="dec", kernel=_stream(f64, GYRO, GEN)),
            gyro(path=2, las="int:dec", kernel=_stream(f64, GYRO, GEN)),         # LAS intensity alone: generic
        ]
        slerp = lambda **kw: Case(f64=f64, mode=SLERP, **kw)         # noqa: E731
        rows += [
            slerp(path=0, lvx="t2", las="dec", kernel=_fused(f64, SLERP)),
            slerp(path=2, kernel=_stream(f64, SLERP, OUT)),
            slerp(path=2, lvx="t2", kernel=_stream(f64, SLERP, OUT | LVX)),
            slerp(path=2, las="dec", kernel=_stream(f64, SLERP, OUT | LAS)),
            slerp(path=2, las="pow2", kernel=_stream(f64, SLERP, OUT | LAS)),
            slerp(path=2, lvx="lvx2", kernel=_stream(f64, SLERP, GEN)),
            slerp(path=2, out=False, lvx="t2", las="pow2", kernel=_stream(f64, SLERP, GEN)),
        ]
        quant = lambda **kw: Case(f64=f64, mode=QUANT, out=False, **kw)  # noqa: E731
        rows += [
            quant(path=0, lvx="t2", las="pow2", kernel=_fused(f64, QUANT)),
            quant(path=2, lvx="t2", las="pow2", kernel=_stream(f64, QUANT, GEN)),
            quant(path=2, lvx="lvx2+tag", las="dec", kernel=_stream(f64, QUANT, GEN)),
        ]
    # fused merged-cloud assembly on one GPU: peer bulk stores (f32 Mode A / C, aligned cloud + type-2 LVX) and the
    # per-peer store loops of the generic kernel
    for mode in (RIGID, SLERP):
        for n in (1, 7):
            rows.append(Case(f64=False, mode=mode, path=2, lvx="t2", peers=n, kernel=_stream(False, mode, OUT | LVX | PB)))
    rows += [
        Case(f64=True, mode=GYRO, path=2, lvx="t2", las="dec", peers=1, kernel=_stream(True, GYRO, GEN)),
        Case(f64=True, mode=GYRO, path=2, lvx="t2", las="dec", peers=7, kernel=_stream(True, GYRO, GEN)),
        Case(f64=False, mode=GYRO, path=2, lvx="lvx2+tag", peers=7, kernel=_stream(False, GYRO, GEN)),
    ]
    return rows


TABLE = _table()
GPU_ORDER = sorted(TABLE, key=lambda c: (not c.f64, RIGID if c.mode == QUANT else c.mode))   # rows sharing inputs run together


# ------------------------------------------------------------------------------------------
# CPU: routing and coverage
# ------------------------------------------------------------------------------------------
def _plan_case(c: Case):
    """The case as a test_launch_plan driver row: a mid-tile shard of a stream larger than any one-wave grid."""
    timed = c.mode in (GYRO, SLERP)
    las_x = c.las is not None and not c.las.startswith("int:")
    return dict(f64=c.f64, mode=c.mode, path=c.path, p_begin=1237, p_end=3_000_001, ts=int(timed),
                tag=int(c.lvx == "lvx2+tag"), out=int(c.out), lvx14=int(c.lvx is not None), las_x=int(las_x),
                las_int=int(c.las is not None), lvx_mode=LVX2_OF_OUTPUT if c.lvx and c.lvx.startswith("lvx2") else LVX_TYPE2_OF_INPUT,
                n_peers=c.peers, mc=0, hold_idx=0, frame_start=int(timed), n_samp=720_001 if timed else 0)


def test_every_case_routes_to_its_kernel(plan):
    got = plan([row(_plan_case(c)) for c in TABLE])
    assert len(got) == len(TABLE)
    for c, (rc, stream, ex, *_) in zip(TABLE, got):
        assert rc == 0, c.id
        kernel = _stream(c.f64, c.mode, ex) if stream else _fused(c.f64, c.mode)
        assert kernel == c.kernel, (c.id, kernel)


def _library_kernels(path):
    exe = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    text = subprocess.run([exe, "-symbols", path], capture_output=True, text=True, check=True, timeout=300).stdout
    ks = {_fused(f == "1", int(m)) for f, m in re.findall(r"k_fusedILb([01])ELi(\d+)EE", text)}
    ks |= {_stream(f == "1", int(m), int(x)) for f, m, x in re.findall(r"k_streamILb([01])ELi(\d+)ELi(\d+)EE", text)}
    return ks


def test_table_covers_every_point_kernel():
    """The rows name exactly the library's k_fused / k_stream instantiations, multicast excepted (it needs a real multicast
    mapping), and those of sensor-frame deskew and distortion (modes 4 and 5: the tables of test_deskew_local and
    test_motion_distortion): a new variant without a row fails here."""
    path = os.environ.get("LMC_B200_LIB", _build.LIB_PATH)
    if not os.path.exists(path):
        pytest.skip(f"{path} is not built")
    built = {k for k in _library_kernels(path) if not (k[0] == "stream" and k[3] & MC) and k[2] not in (4, 5)}
    named = {c.kernel for c in TABLE}
    assert not built - named, f"kernels without a row: {sorted(built - named)}"
    assert not named - built, f"rows naming a kernel the library lacks: {sorted(named - built)}"


# ------------------------------------------------------------------------------------------
# GPU: shared inputs
# ------------------------------------------------------------------------------------------
def _edge_values(f64):
    """(n, 4) points that exercise the quantisers' edges for both LAS configurations; the f32 layout gets the nearest f32."""
    axes = [[], [], []]
    for c in range(3):
        for scale, off, _ in LAS_CFG.values():
            s, o = scale[c], off[c]
            q = [k + 0.5 for k in (-3, -2, -1, 0, 1, 2, 1000, -1001, 123456)]                   # exact ties (pow2)
            q += [2.0 ** 31 - 1025, 2.0 ** 31 - 1024, 2.0 ** 31 - 1023.5, 2.0 ** 31 - 1023,        # around the fast-path limit
                  2147483646.5, 2147483647.0, 2147483647.25, 2147483647.5, 2147483647.75, 2147483648.0,
                  -2147483647.5, -2147483648.0, -2147483648.25, -2147483648.5, -2147483648.75, -2147483649.0]
            v = [o + k * s for k in q]
            near = [o + k * s for k in (0.5, 1.5, -2.5, 12345.5, -777.5)]                        # near-ties (dec)
            v += near + [np.nextafter(x, np.inf) for x in near] + [np.nextafter(x, -np.inf) for x in near]
            axes[c] += v
        axes[c] += [2147483.647, -2147483.647, 2147483.648, -2147483.648, 2147483.6475, -2147483.6485, 1e10, -1e10]   # type-2 clip
    n = max(len(a) for a in axes)
    xyz = np.full((n, 3), 1.25)
    for c in range(3):
        xyz[:len(axes[c]), c] = axes[c]
        xyz[:, c] = np.roll(xyz[:, c], 7 * c)                     # different neighbours per axis
    special = [np.nan, np.inf, -np.inf]
    rows = [xyz]
    for s in special:
        for c in range(3):
            r = np.full((1, 3), 2.5)
            r[0, c] = s
            rows.append(r)
    rows.append(np.array([[-0.0, 0.0, -0.0], [0.0, -0.0, -0.0], [-0.0, -0.0, -0.0]]))
    xyz = np.concatenate(rows)
    inten = np.array([-0.5, 1.5, 255.5, 70000.7, np.nan, 0.0, 0.25, 1.0, 254.9, 255.0, 3.0, -0.0])
    pts = np.column_stack([xyz, np.resize(inten, len(xyz))])
    return pts if f64 else pts.astype(np.float32).astype(np.float64)


def _counts(rng, n_total, p0, n_block):
    """Frame sizes summing to n_total: random frames (empty, one-point, short and multi-tile ones), a run of 0-3 point frames,
    then the edge block's three frames [40, 1, rest] starting at point p0.  Returns (counts, index of the first block frame)."""
    def fill(total):
        c, s = [], 0
        while s < total:
            r = rng.random()
            k = 0 if r < 0.08 else 1 if r < 0.14 else int(rng.integers(2, 200)) if r < 0.3 else int(rng.integers(200, 6000))
            k = min(k, total - s)
            c.append(k)
            s += k
        return c
    head = fill(n_total // 5) + [int(x) for x in rng.integers(0, 4, 4000)]
    head += fill(p0 - sum(head))
    return np.array(head + [40, 1, n_block - 41] + fill(n_total - p0 - n_block), np.int64), len(head)


def _sm_count():
    v = ctypes.c_int32(0)
    C.check(C.lib().lmc_device_query(ctypes.byref(v), None, None))
    return v.value


def _stages(f64, mode):
    return 3 if (not f64 and mode == SLERP) else 4                # StreamCfg::STAGES (csrc/lmc_tma.cu)


@dataclass
class Inputs:
    f64: bool
    mode: int
    n: int
    pts: "torch.Tensor"
    pts64: np.ndarray
    args: tuple                    # device arguments of the mode's entry point between pts and out
    want: np.ndarray               # oracle rows (N, 4) f64 (the input itself for the stand-alone quantisers)
    tag: "torch.Tensor"
    tag_np: np.ndarray
    block: tuple                   # [p0, p1): the edge block
    b: int
    e: int
    cuts: tuple                    # three shards of [b, e), one cut inside the edge block


def _make_inputs(f64, mode):
    from livox_motion_compensation_sim_b200 import synth
    base = RIGID if mode == QUANT else mode
    tp = tile_points(f64, base)
    sms = _sm_count()
    rng = np.random.default_rng(2024 + 10 * base + f64)
    edge = _edge_values(f64)
    nb = len(edge)
    n_tiles = sms * (_stages(f64, base) + 2) + 4                  # for the [b, e) shard: STAGES + 2 tiles per CTA at least
    N = n_tiles * tp + 1237 + 911 + 2 * tp // 3
    p0 = (int(0.45 * N) // tp) * tp - 45                          # the block straddles a tile boundary
    counts, fb = _counts(rng, N, p0, nb)
    F = len(counts)
    st = synth.make_stream(F, counts, 2024 + base, device=DEV, dtype=torch.float64 if f64 else torch.float32)
    assert st.n_points == N
    st.pts[p0:p0 + nb] = torch.from_numpy(edge).to(DEV, st.pts.dtype)
    pts64 = st.pts.cpu().numpy().astype(np.float64)
    frame_start = st.frame_start.copy()
    frame_start[fb:fb + 3] += 1000                                # block points strictly inside their (identity) segments
    fidx = np.repeat(np.arange(F), counts)
    ts_off = st.ts_off.cpu().numpy().astype(np.int64)
    ts64 = frame_start[fidx] + ts_off
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    off = d(st.frame_off)
    ts = d(ts64) if f64 else st.ts_off
    # the samples that bracket the block's points carry the identity: samples 20 f .. 20 f + 1 (frames start every 100 ms, samples every 5 ms)
    around = np.concatenate([np.arange(20 * f - 1, 20 * f + 3) for f in range(fb, fb + 3)])
    if base == RIGID:
        pose = st.gps_Rt[orc.pose_lookup_hold_next_np(st.gps_t, st.frame_t)]
        pose[fb:fb + 3] = [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]
        args = (off, d(pose))
        want = pts64.copy() if mode == QUANT else orc.C.align_rigid_f64(pts64, st.frame_off, pose, threads=8)
    elif base == GYRO:
        gyro = rng.normal(0, 0.3, (len(st.sample_ts), 3))
        gyro[around] = 0.0
        args = (ts, off, d(frame_start), d(st.sample_ts), d(gyro), len(st.sample_ts))
        want = orc.C.deskew_gyro_f64(pts64, ts64, st.frame_off, frame_start, st.sample_ts, gyro)
    else:
        from livox_motion_compensation_sim_b200 import frames as FR
        quat, pos = st.sample_quat.copy(), st.sample_pos.copy()
        quat[around] = [0.0, 0.0, 0.0, 1.0]
        pos[around] = 0.0
        seg = FR.slerp_segment_table(quat, pos, st.sample_ts)
        args = (ts, off, d(frame_start), d(st.sample_ts), d(seg), len(st.sample_ts), None)
        want = orc.C.deskew_slerp_f64(pts64, ts64, st.frame_off, st.sample_ts, seg)
    blk = slice(p0, p0 + nb)
    fin = np.isfinite(pts64[blk, :3]).all(axis=1)
    assert np.array_equal(want[blk][fin], pts64[blk][fin], equal_nan=True), "the edge block's transform is not the identity"
    tag_np = rng.integers(0, 256, N).astype(np.uint8)
    b, e = 1237, N - 911
    assert b % tp and e % tp and (e - (b // tp) * tp) // tp >= sms * (_stages(f64, base) + 2)
    cuts = (b, p0 + 71, int(0.7 * N) | 1, e)                      # (the first cut falls inside the block, mid-tile)
    return Inputs(f64, mode, N, st.pts, pts64, args, want, d(tag_np), tag_np, (p0, p0 + nb), b, e, cuts)


@pytest.fixture(scope="module")
def inputs():
    """Inputs for (layout, mode), built once; the table's rows are grouped by them, so one set is kept at a time."""
    cache = {}

    def get(f64, mode):
        key = (f64, RIGID if mode == QUANT else mode)
        if key not in cache:
            cache.clear()
            torch.cuda.empty_cache()
            cache[key] = _make_inputs(*key)
        x = cache[key]
        if mode == QUANT:
            return Inputs(**{**x.__dict__, "mode": QUANT, "want": x.pts64, "b": 0, "e": x.n})
        return x
    return get


# ------------------------------------------------------------------------------------------
# GPU: one call through the C ABI, every buffer inside sentinel guard bands
# ------------------------------------------------------------------------------------------
G = 4096                                                          # guard elements on each side (keeps 32-byte alignment)


class Guarded:
    def __init__(self, n, tail, dtype, fill):
        self.fill = fill
        self.full = torch.full((n + 2 * G,) + tail, fill, dtype=dtype, device=DEV)
        self.view = self.full[G:G + n]

    def untouched_outside(self, b, e):
        return bool((self.full[:G + b] == self.fill).all()) and bool((self.full[G + e:] == self.fill).all())


class Buffers:
    def __init__(self, c: Case, x: Inputs):
        n, fdt = x.n, torch.float64 if x.f64 else torch.float32
        self.out = Guarded(n, (4,), fdt, -123.0) if c.out else None
        self.lvx = Guarded(n, (14,), torch.uint8, 0xAB) if c.lvx else None
        xyz = c.las is not None and not c.las.startswith("int:")
        self.las = [Guarded(n, (), torch.int32, -77) for _ in range(3)] if xyz else None
        self.las_int = Guarded(n, (), torch.int16, 0x5A5A) if c.las else None
        self.status = torch.zeros(1, dtype=torch.int32, device=DEV)
        self.peers = []
        for r in range(c.peers):
            if c.peers == 7 and r == 3:
                self.peers.append(None)                           # a NULL entry in the middle of the peer list
            else:
                self.peers.append((Guarded(n, (4,), fdt, -123.0), Guarded(n, (14,), torch.uint8, 0xAB) if c.lvx else None))

    def local(self):
        return [g for g in [self.out, self.lvx, self.las_int] + (self.las or []) if g is not None]

    def flags(self):
        return int(self.status.item())


def _las_cfg(c: Case):
    return LAS_CFG[c.las.split(":")[-1]]


def _call(c: Case, x: Inputs, B: Buffers, path, b, e, tag=None, peers=True):
    ex = C.LmcExport()
    ex.lvx14 = B.lvx.view.data_ptr() if B.lvx else None
    ex.lvx_mode = LVX2_OF_OUTPUT if c.lvx and c.lvx.startswith("lvx2") else LVX_TYPE2_OF_INPUT
    if c.lvx == "lvx2+tag":
        ex.tag = (x.tag if tag is None else tag).data_ptr()
    if c.las:
        scale, off, imode = _las_cfg(c)
        if B.las:
            ex.las_x, ex.las_y, ex.las_z = (g.view.data_ptr() for g in B.las)
        ex.las_intensity = B.las_int.view.data_ptr()
        ex.las_intensity_mode = imode
        for k in range(3):
            ex.las_scale[k], ex.las_offset[k] = scale[k], off[k]
    else:
        for k in range(3):
            ex.las_scale[k] = 0.01
    ex.status = B.status.data_ptr()
    if peers and B.peers:
        ex.n_peers = len(B.peers)
        for r, p in enumerate(B.peers):
            ex.peer_out[r] = p[0].view.data_ptr() if p else None
            ex.peer_lvx14[r] = p[1].view.data_ptr() if p and p[1] else None
    L = C.lib()
    pts, out = x.pts.data_ptr(), B.out.view.data_ptr() if B.out else None
    st = torch.cuda.current_stream().cuda_stream
    C.set_path(path)
    try:
        if c.mode == QUANT:
            rc = (L.lmc_quantize_f64 if x.f64 else L.lmc_quantize_f32)(pts, x.n, ctypes.byref(ex), st)
        else:
            F = x.args[0 if c.mode == RIGID else 1].shape[0] - 1
            a = [v.data_ptr() if isinstance(v, torch.Tensor) else v for v in x.args]
            fn = {RIGID: (L.lmc_align_rigid_f64, L.lmc_align_rigid_f32), GYRO: (L.lmc_deskew_gyro_f64, L.lmc_deskew_gyro_f32),
                  SLERP: (L.lmc_deskew_slerp_f64, L.lmc_deskew_slerp_f32)}[c.mode][0 if x.f64 else 1]
            rc = fn(pts, *a, out, x.n, F, b, e, ctypes.byref(ex), st)
    finally:
        C.set_path(C.PATH_AUTO)
    torch.cuda.synchronize()
    return rc


def _bytes(t):
    """A buffer's bytes with every NaN made the same NaN (payloads are not part of the contract)."""
    if t.dtype in (torch.float32, torch.float64):
        t = torch.where(torch.isnan(t), torch.full_like(t, float("nan")), t)
    return t.contiguous().view(torch.uint8)


def _same(g1: Guarded, g2: Guarded):
    return torch.equal(_bytes(g1.full), _bytes(g2.full))


def _all_same(B1: Buffers, B2: Buffers, peers=True):
    pairs = list(zip(B1.local(), B2.local()))
    if peers:
        for p1, p2 in zip(B1.peers, B2.peers):
            if p1:
                pairs += [(p1[0], p2[0])] + ([(p1[1], p2[1])] if p1[1] else [])
    return all(_same(a, b) for a, b in pairs)


# ------------------------------------------------------------------------------------------
# GPU: what the oracle says
# ------------------------------------------------------------------------------------------
def _check_rows(f64, mode, got, want):
    """got: the device's rows, want: the oracle's (f64).  Rows holding a NaN are compared by NaN mask."""
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w), np.argwhere(nan_g != nan_w)[:5]
    ok = ~nan_w
    if mode in (RIGID, QUANT):                                     # bit-identical (f64) / one rounding of the f64 result (f32)
        w = want if f64 else want.astype(np.float32)
        assert np.array_equal(got[ok].view(np.uint64 if f64 else np.uint32), w[ok].view(np.uint64 if f64 else np.uint32))
        return
    g64 = got.astype(np.float64)
    inf = np.isinf(want) & ok
    assert np.array_equal(g64[inf], want[inf])
    fin = ok & ~inf
    assert np.abs(g64[fin] - want[fin]).max(initial=0.0) <= (1e-10 if f64 else TOL_M)
    if not f64:
        assert int((got[fin] != want[fin].astype(np.float32)).sum()) <= 4


def _expected_exports(c: Case, x: Inputs, rows, b, e):
    """(dict of integer buffers, status flags) the oracle quantisers give on [b, e).  rows: what the LAS / LVX2 quantisers see."""
    want, fl = {}, 0
    if c.lvx == "t2":
        want["lvx"], f = orc.C.quantize_lvx_type2(x.pts64[b:e])
        fl |= f
    elif c.lvx:
        want["lvx"], f = orc.C.quantize_lvx2(rows, x.tag_np[b:e] if c.lvx == "lvx2+tag" else None)
        fl |= f
    if c.las:
        scale, off, imode = _las_cfg(c)
        X, Y, Z, I, f = orc.C.quantize_las(rows, scale, off, imode)
        if c.las.startswith("int:"):
            f = orc.C.quantize_las(np.column_stack([np.zeros((len(rows), 3)), rows[:, 3]]), scale, off, imode)[4]
        else:
            want["las"] = (X, Y, Z)
        want["las_int"] = I
        fl |= f
    return want, fl


def _check_exports(B: Buffers, want, b, e):
    if "lvx" in want:
        got = B.lvx.view[b:e].cpu().numpy()
        bad = np.flatnonzero((got != want["lvx"]).any(axis=1))
        assert bad.size == 0, (b + bad[:5], got[bad[:3]], want["lvx"][bad[:3]])
    if "las" in want:
        for g, w in zip(B.las, want["las"]):
            got = g.view[b:e].cpu().numpy()
            bad = np.flatnonzero(got != w)
            assert bad.size == 0, (b + bad[:5], got[bad[:5]], w[bad[:5]])
    if "las_int" in want:
        got = B.las_int.view[b:e].cpu().numpy().view(np.uint16)
        bad = np.flatnonzero(got != want["las_int"])
        assert bad.size == 0, (b + bad[:5], got[bad[:5]], want["las_int"][bad[:5]])


# ------------------------------------------------------------------------------------------
# GPU: the cases
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c", GPU_ORDER, ids=[c.id for c in GPU_ORDER])
def test_kernel_variant_vs_oracle(c: Case, inputs):
    x = inputs(c.f64, c.mode)
    b, e = x.b, x.e
    p0, p1 = x.block
    B = Buffers(c, x)
    C.check(_call(c, x, B, c.path, b, e))

    # rows
    if c.out:
        got = B.out.view[b:e].cpu().numpy()
        _check_rows(c.f64, c.mode, got, x.want[b:e])
    # integer exports against the oracle quantisers: on the oracle rows, except f64 Modes B / C, where the device's own rows
    # are quantised (the rows themselves are only within 1e-10 m of the oracle's)
    rows = x.want[b:e]
    if c.f64 and c.mode in (GYRO, SLERP):
        if c.out:
            rows = B.out.view[b:e].cpu().numpy()
        else:                                                       # the same call with the aligned cloud gives the rows
            co = Case(**{**c.__dict__, "out": True})
            Bo = Buffers(co, x)
            C.check(_call(co, x, Bo, c.path, b, e))
            rows = Bo.out.view[b:e].cpu().numpy()
    want, fl = _expected_exports(c, x, rows, b, e)
    _check_exports(B, want, b, e)
    # status: the OR of the oracle's flags over [b, e) -- NaN and overflow in the edge block
    assert B.flags() == fl, (B.flags(), fl)
    if c.lvx or c.las:
        assert fl != 0 and b <= p0 and p1 <= e                     # the block reached the quantisers
    # bounds: nothing outside [b, e), nothing outside the buffers; peer copies equal the local result
    for g in B.local():
        assert g.untouched_outside(b, e)
    for p in B.peers:
        if p:
            assert _same(p[0], B.out) and (p[1] is None or _same(p[1], B.lvx))

    # the other kernel family (peer stores exist in the streaming kernels only: the direct call has none) -- same bytes, same status
    B2 = Buffers(c, x)
    C.check(_call(c, x, B2, 2 if c.path == 0 else 0, b, e, peers=False))
    assert _all_same(B, B2, peers=False) and B2.flags() == B.flags()

    if c.mode != QUANT:
        # three odd-cut shards compose to the single launch (peers included)
        B3 = Buffers(c, x)
        for lo, hi in zip(x.cuts[:-1], x.cuts[1:]):
            C.check(_call(c, x, B3, c.path, lo, hi))
        assert _all_same(B, B3) and B3.flags() == B.flags()
        # a call whose NaN / overflow points all lie outside its range reports nothing
        B4 = Buffers(c, x)
        C.check(_call(c, x, B4, c.path, b, p0 - 1))
        assert B4.flags() == 0
    else:
        # the stand-alone quantisers take no range: the flag-free run of points before the block, as a view
        lo, hi = 16 * 7, (p0 // 16) * 16
        y = Inputs(**{**x.__dict__, "pts": x.pts[lo:hi], "n": hi - lo, "tag": x.tag[lo:hi]})
        B4 = Buffers(c, y)
        C.check(_call(c, y, B4, c.path, 0, y.n))
        assert B4.flags() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [True, False], ids=["f64", "f32"])
def test_unaligned_tag(f64, inputs):
    """fill_export does not require the tag array to be aligned; the plan sends a tag the TMA engine cannot read to the direct
    kernel.  An LVX2 call on the streaming path with the tag one byte off its allocation gives the bytes of the aligned tag;
    with peers (streaming only) the same call is refused as a bad argument and writes nothing."""
    x = inputs(f64, GYRO)
    c = Case(f64=f64, mode=GYRO, path=2, lvx="lvx2+tag", kernel=_stream(f64, GYRO, OUT | LVX | LVX2))
    raw = torch.zeros(x.n + 1, dtype=torch.uint8, device=DEV)
    raw[1:] = x.tag
    shifted = raw[1:]
    assert shifted.data_ptr() % 16 == 1
    A, U = Buffers(c, x), Buffers(c, x)
    C.check(_call(c, x, A, 2, x.b, x.e))
    C.check(_call(c, x, U, 2, x.b, x.e, tag=shifted))
    assert _all_same(A, U) and A.flags() == U.flags() != 0
    cp = Case(**{**c.__dict__, "peers": 1})
    P = Buffers(cp, x)
    assert _call(cp, x, P, 2, x.b, x.e, tag=shifted) == C.ERR_INVALID
    assert P.flags() == 0
    for g in P.local() + [g for p in P.peers for g in p]:
        assert g.untouched_outside(0, 0)
