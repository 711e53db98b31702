"""The three binary file writers -- k_lvx_v11 (LVX v1.1), k_lvx_cs (LVX2 / LVX3 / legacy LVX) and k_las_records + k_las_header
(LAS 1.2 PF3) -- and the sharded writers built on them, against host expectations made from the oracle quantisers.

Each writer assembles a CTA's byte range in shared memory at the destination's 16-byte phase and writes it with one TMA bulk
store and byte-wise ragged ends.  So the streams here put frame sizes around each writer's unit of work (96-point packages and
8-package CTAs, 1024-point CTAs, 512-point tiles with a funnel-shift full-tile path and a halfword tail path), records at every
byte phase, and one edge-value block of the quantisers' edges (`_edge_values` of test_kernel_variants plus each format's own)
into every stream.  Checked: the bytes, the status word against the oracle's flags (and 0 on the same stream with the flagged
edge rows replaced), byte ranges of a shard against the whole file, shards composing to the whole file, sentinel guard bands
around every buffer a C entry point writes, and refusal of a range buffer off its file phase.

CPU: the expectation builders reproduce the reference writers' own golden files, and the LAS header test's extremes are ones
where one rounding (fma) and NumPy's two roundings differ."""
import ctypes
import json
import os
import struct
from fractions import Fraction

import numpy as np
import pytest

from tests.test_kernel_variants import LAS_CFG, _edge_values

torch = pytest.importorskip("torch")

from livox_motion_compensation_sim_b200 import _capi as C                  # noqa: E402
from livox_motion_compensation_sim_b200.lvx import (DeviceInfo, build_lvx_v11_file, frame_layout,  # noqa: E402
                                                     lvx_cs_prefix)
from oracle import lmc_oracle as orc                                      # noqa: E402  (checker only)

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
DEV = "cuda:0"
G = 4096                                                                  # sentinel bytes on each side of a guarded buffer
FILL = 0xA5
YEAR, DAY = 2026, 293
FLT_MAX = float(np.finfo(np.float32).max)

gpu = pytest.mark.gpu
needs_gpu = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")


# ------------------------------------------------------------------------------------------
# Host expectations
# ------------------------------------------------------------------------------------------
def first_diff(got, want):
    """'' when the byte arrays are equal, else where and how they first differ."""
    got, want = np.asarray(got, np.uint8).ravel(), np.asarray(want, np.uint8).ravel()
    if got.shape == want.shape and np.array_equal(got, want):
        return ""
    n = min(len(got), len(want))
    bad = np.flatnonzero(got[:n] != want[:n])
    if bad.size == 0:
        return f"sizes {len(got)} != {len(want)}"
    i = int(bad[0])
    return (f"{bad.size} bytes differ, first at offset {i}: got {got[i:i + 16].tobytes().hex()} want {want[i:i + 16].tobytes().hex()}"
            + ("" if len(got) == len(want) else f"; sizes {len(got)} != {len(want)}"))


def lvx_v11_expected(pts64, frame_off, frame_time, frame_id):
    """(whole LVX v1.1 file, status flags): the host container around the oracle's type-2 records."""
    rec, fl = orc.C.quantize_lvx_type2(pts64)
    return build_lvx_v11_file(rec, frame_off, frame_time, frame_id), fl


def _pack_f32(v):
    """struct.pack('<f', v), and the f32 conversion (+-inf) where struct.pack raises: (4 bytes, overflowed)."""
    try:
        return struct.pack("<f", v), False
    except OverflowError:
        with np.errstate(over="ignore"):
            return np.float32(v).tobytes(), True


def legacy_records(pts64, tag):
    """Legacy LVX records struct.pack('<fffBB', x, y, z, intensity, tag) one by one; the intensity byte and its flags are the
    LVX2 quantiser's (both formats copy it the same way).  Returns ((N, 14) uint8, flags)."""
    n = len(pts64)
    ib, fl = orc.C.quantize_lvx2(np.column_stack([np.zeros((n, 3)), pts64[:, 3]]), tag)
    out = np.empty((n, 14), np.uint8)
    for i, (x, y, z, _) in enumerate(pts64.tolist()):
        try:
            b = struct.pack("<fffBB", x, y, z, int(ib[i, 12]), int(ib[i, 13]))
        except OverflowError:
            parts = [_pack_f32(v) for v in (x, y, z)]
            fl |= orc.FLAG_OVERFLOW if any(o for _, o in parts) else 0
            b = b"".join(p for p, _ in parts) + bytes([ib[i, 12], ib[i, 13]])
        out[i] = np.frombuffer(b, np.uint8)
    return out, fl


def lvx_cs_records(pts64, tag, fmt):
    if fmt == C.LVXCS_LVX2:
        return orc.C.quantize_lvx2(pts64, tag)
    return legacy_records(pts64, tag)


def lvx_cs_expected(pts64, tag, frame_off, frame_ts, prefix, fmt, records=None):
    """(whole LVX2 / legacy file, status flags): the container of orc.lvx_cs_file_np (on a copy whose records are all zero, so
    that no edge value reaches its packer), with the records of lvx_cs_records patched in."""
    rec, fl = records if records is not None else lvx_cs_records(pts64, tag, fmt)
    out = orc.lvx_cs_file_np(np.zeros_like(pts64), None, frame_off, frame_ts, prefix, fmt)
    n, F = len(pts64), len(frame_off) - 1
    H = C.LVXCS_FRAME_BYTES[fmt]
    if n:
        fr = np.repeat(np.arange(F), np.diff(frame_off))
        dst = len(prefix) + H * (fr + 1) + 14 * np.arange(n)              # frame f starts at prefix + H f + 14 off[f]
        assert not out[dst[:, None] + np.arange(14)].any()
        out[dst[:, None] + np.arange(14)] = rec
    return out, fl


LAS_REC = np.dtype([("X", "<i4"), ("Y", "<i4"), ("Z", "<i4"), ("I", "<u2"), ("zero6", "u1", 6), ("gps", "<f8"), ("rgb", "<u2", 3)])


def las_records(pts64, scale, offset, mode, gps):
    """(34-byte PF3 records as uint8 (N, 34), (X, Y, Z), flags): the oracle's X / Y / Z / intensity, gps_time bit for bit."""
    X, Y, Z, I, fl = orc.C.quantize_las(pts64, scale, offset, mode)
    r = np.zeros(len(pts64), LAS_REC)
    r["X"], r["Y"], r["Z"], r["I"] = X, Y, Z, I
    if gps is not None:
        r["gps"] = gps.view(np.float64)
    return r.view(np.uint8).reshape(-1, 34), (X, Y, Z), fl


def las_extreme(q, scale, offset):
    """X * scale + offset as laspy's update_header evaluates it in NumPy: a rounded product, then a rounded sum."""
    return float(np.float64(q) * np.float64(scale) + np.float64(offset))


def las_header(n, scale, offset, mins, maxs):
    """The 227-byte LAS 1.2 public header block of an n-record PF3 file without VLRs (LAS 1.2 specification, the fields the
    reference sets; the integer extremes mins / maxs per axis give the scaled ones)."""
    h = bytearray(227)
    h[0:4] = b"LASF"
    h[24], h[25] = 1, 2
    h[26:31] = b"OTHER"
    h[58:71] = b"livox_mc_b200"
    struct.pack_into("<HHHI", h, 90, DAY, YEAR, 227, 227)
    struct.pack_into("<BHI", h, 104, 3, 34, n)
    struct.pack_into("<3d", h, 131, *scale)
    struct.pack_into("<3d", h, 155, *offset)
    for c in range(3):
        mx = las_extreme(maxs[c], scale[c], offset[c]) if n else 0.0
        mn = las_extreme(mins[c], scale[c], offset[c]) if n else 0.0
        struct.pack_into("<dd", h, 179 + 16 * c, mx, mn)
    return np.frombuffer(bytes(h), np.uint8)


def las_expected(pts64, scale, offset, mode, gps):
    rec, xyz, fl = las_records(pts64, scale, offset, mode, gps)
    n = len(pts64)
    mins = [int(q.min()) if n else 0 for q in xyz]
    maxs = [int(q.max()) if n else 0 for q in xyz]
    return np.concatenate([las_header(n, scale, offset, mins, maxs), rec.ravel()]), fl


def fma_extreme(q, scale, offset):
    """X * scale + offset with ONE rounding (exact rational arithmetic, one correctly rounded conversion)."""
    f = Fraction(int(q)) * Fraction(scale) + Fraction(offset)
    return f.numerator / f.denominator                       # int / int true division is correctly rounded


# header extremes where the one-rounding and the two-rounding values differ: (scale, offset, integer X values)
HEADER_CASES = []


def _header_cases():
    if not HEADER_CASES:
        rng = np.random.default_rng(291)
        for scale, offset in [(0.001, 1000.0), (0.001, 10.0), (0.01, 0.3), (0.002, 123.456)]:
            xs = []
            for x in rng.integers(-2 ** 31, 2 ** 31, 200_000):
                if las_extreme(x, scale, offset) != fma_extreme(x, scale, offset):
                    xs.append(int(x))
                    if len(xs) == 6:
                        break
            HEADER_CASES.append((scale, offset, xs))
    return HEADER_CASES


def row_flags(quantise, rows):
    """The oracle's flags of each row on its own."""
    return np.array([quantise(rows[i:i + 1]) for i in range(len(rows))], np.int64)


def clean(pts64, flags):
    """The rows whose oracle flags are non-zero replaced by a quiet value (so the stream must report status 0)."""
    out = pts64.copy()
    out[flags != 0] = [1.25, -2.5, 3.75, 7.0]
    return out


# ------------------------------------------------------------------------------------------
# CPU: the expectation builders reproduce the reference writers' golden files
# ------------------------------------------------------------------------------------------
def test_lvx_v11_expectation_reproduces_reference_file():
    g = np.load(os.path.join(GOLDEN, "lvx_file.npz"))
    off = g["frame_off"]
    want, fl = lvx_v11_expected(g["raw"], off, g["timestamps"], np.arange(len(off) - 1))
    assert fl == 0
    assert not first_diff(want, g["file_bytes"]), first_diff(want, g["file_bytes"])


@pytest.mark.parametrize("ver,key", [("lvx2", "file_lvx2"), ("lvx", "file_legacy")])
def test_lvx_cs_expectation_reproduces_reference_file(ver, key):
    g = np.load(os.path.join(GOLDEN, "lvx_cs.npz"))
    off = g["frame_off"]
    di = DeviceInfo(**json.loads(bytes(g["device_info_json"]).decode()))
    fmt = C.LVXCS_LEGACY if ver == "lvx" else C.LVXCS_LVX2
    want, fl = lvx_cs_expected(g["pts"], g["tag"], off, g["frame_ts"], lvx_cs_prefix(ver, di, len(off) - 1), fmt)
    assert fl == 0
    assert not first_diff(want, g[key]), first_diff(want, g[key])


def test_legacy_record_packer_edges():
    """struct.pack's own results where the device has to match it: NaN keeps its sign and payload, the largest finite values
    round to FLT_MAX or raise (and then the record holds inf), f32 subnormals round to nearest-even."""
    rows = np.array([[np.nan, -np.nan, 0.0, 1.0], [FLT_MAX, -FLT_MAX, 2.0 ** 128, 2.0],
                     [2.0 ** -150, 3 * 2.0 ** -150, -(2.0 ** -149), 3.0]])
    rec, fl = legacy_records(rows, None)
    words = rec[:, :12].copy().view("<u4")
    assert words[0].tolist() == [0x7FC00000, 0xFFC00000, 0]
    assert words[1].tolist() == [0x7F7FFFFF, 0xFF7FFFFF, 0x7F800000] and fl == orc.FLAG_OVERFLOW
    assert words[2].tolist() == [0, 2, 0x80000001]
    assert rec[:, 12].tolist() == [1, 2, 3] and not rec[:, 13].any()


def test_las_header_cases_separate_the_two_roundings():
    """Every header case has extremes where fma(X, scale, offset) is not NumPy's X * scale + offset, so a header written with
    the wrong rounding fails test_las_header_extremes_are_numpys."""
    for scale, offset, xs in _header_cases():
        assert len(xs) == 6, (scale, offset)
        assert all(las_extreme(x, scale, offset) != fma_extreme(x, scale, offset) for x in xs)


# ------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def _points(f64, pts64):
    """The device tensor of the layout, and the f64 values it holds (what every expectation is computed from)."""
    t = torch.from_numpy(np.ascontiguousarray(pts64)).to(DEV, torch.float64 if f64 else torch.float32)
    return t, t.cpu().numpy().astype(np.float64)


class GuardedBytes:
    """n bytes at file position pos0: a view congruent to pos0 modulo 16 inside an allocation filled with a sentinel."""

    def __init__(self, n, pos0, shift=0):
        self.n, self.start = n, G + pos0 % 16 + shift
        self.full = torch.full((G + 32 + n + G,), FILL, dtype=torch.uint8, device=DEV)
        self.ptr = self.full.data_ptr() + self.start

    def host(self):
        torch.cuda.synchronize()
        return self.full.cpu().numpy()

    def inside(self):
        return self.host()[self.start:self.start + self.n]

    def outside_untouched(self):
        h = self.host()
        return bool((h[:self.start] == FILL).all() and (h[self.start + self.n:] == FILL).all())

    def untouched(self):
        return bool((self.host() == FILL).all())


def _status():
    return torch.zeros(1, dtype=torch.int32, device=DEV)


# ------------------------------------------------------------------------------------------
# LVX v1.1
# ------------------------------------------------------------------------------------------
LVX11_COUNTS = [0, 1, 95, 96, 97, 767, 768, 769, 1535, 1537, 0, 20_013, 3, 0, 2, 1, 0]
LVX11_BLOCK = (9, 700)                        # the edge block: frame 9 (1537 points), from its point 700 (crosses a CTA's 768)


def _lvx11_inputs(f64, with_block=True):
    rng = np.random.default_rng(1101 + f64)
    counts = np.array(LVX11_COUNTS, np.int64)
    off = np.zeros(len(counts) + 1, np.int64)
    np.cumsum(counts, out=off[1:])
    n = int(off[-1])
    pts = np.column_stack([rng.uniform(-250, 250, (n, 3)), rng.uniform(0, 1, n)])
    edge = _edge_values(f64)
    p0 = int(off[LVX11_BLOCK[0]]) + LVX11_BLOCK[1]
    pts[p0:p0 + len(edge)] = edge
    if not with_block:
        pts[p0:p0 + len(edge)] = clean(edge, row_flags(lambda r: orc.C.quantize_lvx_type2(r)[1], edge))
    F = len(counts)
    ft = 0.1 * np.arange(F)                                               # int(t * 1e9) truncates for several of these
    ft[F // 2:] += 1e4
    ids = rng.integers(0, 2 ** 40, F).astype(np.int64)
    t, p64 = _points(f64, pts)
    return t, p64, off, ft, ids


@pytest.fixture(scope="module", params=[True, False], ids=["f64", "f32"])
def lvx11(request):
    t, p64, off, ft, ids = _lvx11_inputs(request.param)
    want, fl = lvx_v11_expected(p64, off, ft, ids)
    return dict(f64=request.param, pts=t, p64=p64, off=off, ft=ft, ids=ids, want=want, flags=fl)


@gpu
@needs_gpu
def test_lvx_v11_whole_file(lvx11):
    from livox_motion_compensation_sim_b200 import ops
    x = lvx11
    _, fpos = frame_layout(x["off"])
    data, status = ops.build_lvx_v11(x["pts"], dev(x["off"]), dev(fpos), dev(x["ft"]), dev(x["ids"]), int(np.diff(x["off"]).max()))
    assert not first_diff(data.cpu().numpy(), x["want"]), first_diff(data.cpu().numpy(), x["want"])
    assert x["flags"] == C.FLAG_NAN and int(status.item()) == x["flags"]
    # the same stream with the flagged edge rows replaced: status 0, bytes still the oracle's
    t, p64, off, ft, ids = _lvx11_inputs(x["f64"], with_block=False)
    want, fl = lvx_v11_expected(p64, off, ft, ids)
    data, status = ops.build_lvx_v11(t, dev(off), dev(fpos), dev(ft), dev(ids), int(np.diff(off).max()))
    assert fl == 0 and int(status.item()) == 0
    assert not first_diff(data.cpu().numpy(), want), first_diff(data.cpu().numpy(), want)


def _lvx11_ranges(off):
    from livox_motion_compensation_sim_b200 import sharding
    F = len(off) - 1
    big = int(np.argmax(np.diff(off)))
    ranges = [(0, F), (0, F - 3), (10, F), (1, F - 3), (big + 1, F), (F - 1, F), (5, 5), (0, 0), (F, F), (10, 11), (2, big + 1)]
    parts = []
    for W in (3, 7):
        cuts, _ = sharding.shard_ranges(off, W)
        parts.append([(int(a), int(b)) for a, b in zip(cuts[:-1], cuts[1:])])
    return ranges, parts


@gpu
@needs_gpu
def test_lvx_v11_shards(lvx11):
    """sharding.lvx_v11_shard over a cut table: each shard is its byte range of the whole file (a shard's last frame keeps the
    next frame's offset unless it is the file's last), its status the oracle's flags over its points, and the shards of a
    partition concatenate to the whole file."""
    from livox_motion_compensation_sim_b200 import sharding
    x = lvx11
    off = x["off"]
    assert LVX11_COUNTS[0] == 0 and LVX11_COUNTS[10] == 0 and LVX11_COUNTS[1] == 1
    ranges, parts = _lvx11_ranges(off)

    def shard(fb, fe):
        out, pos0, status = sharding.lvx_v11_shard(x["pts"], off, x["ft"], x["ids"], fb, fe)
        got = out.cpu().numpy()
        want = x["want"][pos0:pos0 + len(got)]
        _, fpos = frame_layout(off)
        assert len(got) == (int(fpos[fe]) - pos0 if fe > fb else 0), (fb, fe)
        assert not first_diff(got, want), ((fb, fe), first_diff(got, want))
        fl = orc.C.quantize_lvx_type2(x["p64"][off[fb]:off[fe]])[1] if fe > fb else 0
        assert int(status.item()) == fl, (fb, fe)
        return got

    for fb, fe in ranges:
        shard(fb, fe)
    for p in parts:
        assert p[0][0] == 0 and p[-1][1] == len(off) - 1
        whole = np.concatenate([shard(fb, fe) for fb, fe in p])
        assert not first_diff(whole, x["want"]), (p, first_diff(whole, x["want"]))


@gpu
@needs_gpu
def test_lvx_v11_stays_inside_its_buffers(lvx11):
    """The C entry points on guarded buffers: the whole file and frame ranges, each at its file phase, write exactly their bytes;
    a range buffer one byte off its phase is refused with ERR_ALIGN and nothing is written."""
    x = lvx11
    L = C.lib()
    off, F, n = x["off"], len(x["off"]) - 1, len(x["p64"])
    _, fpos = frame_layout(off)
    keep = [dev(a) for a in (off, fpos, x["ft"], x["ids"])]
    args = (x["pts"].data_ptr(), *(t.data_ptr() for t in keep))
    mx = int(np.diff(off).max())
    build = L.lmc_lvx_v11_build_f64 if x["f64"] else L.lmc_lvx_v11_build_f32
    rng_fn = L.lmc_lvx_v11_build_range_f64 if x["f64"] else L.lmc_lvx_v11_build_range_f32
    B, s = GuardedBytes(int(fpos[-1]), 0), _status()
    C.check(build(*args, B.ptr, n, F, mx, s.data_ptr(), _stream_ptr()))
    assert B.outside_untouched() and not first_diff(B.inside(), x["want"]), first_diff(B.inside(), x["want"])
    assert int(s.item()) == x["flags"]
    for fb, fe in [(0, F - 3), (1, F), (10, 12), (F - 1, F), (9, 10)]:
        pos0 = 0 if fb == 0 else int(fpos[fb])
        nb = int(fpos[fe]) - pos0
        B, s = GuardedBytes(nb, pos0), _status()
        C.check(rng_fn(*args, B.ptr, pos0, n, F, fb, fe, mx, s.data_ptr(), _stream_ptr()))
        assert B.outside_untouched(), (fb, fe)
        assert not first_diff(B.inside(), x["want"][pos0:pos0 + nb]), ((fb, fe), first_diff(B.inside(), x["want"][pos0:pos0 + nb]))
        Bad, s = GuardedBytes(nb, pos0, shift=1), _status()
        assert rng_fn(*args, Bad.ptr, pos0, n, F, fb, fe, mx, s.data_ptr(), _stream_ptr()) == C.ERR_ALIGN
        assert Bad.untouched() and int(s.item()) == 0, (fb, fe)


# ------------------------------------------------------------------------------------------
# LVX2 / legacy
# ------------------------------------------------------------------------------------------
CS_COUNTS = [0, 1, 1023, 1024, 1025, 2047, 2049, 3, 0, 500, 0]
CS_BLOCK = (6, 960)                           # the edge block: frame 6 (2049 points), from its point 960 (crosses a CTA's 1024)


def _cs_edges(f64):
    """_edge_values plus the LVX2 and legacy edges: '<iii' overflow only after truncation, intensities around the byte,
    values that round to +-inf in f32 with FLT_MAX's neighbours, f32 subnormals, signed zeros, +-inf, NaN and -NaN."""
    nx = lambda v, d: float(np.nextafter(v, d))                           # noqa: E731
    half_up = 2.0 ** 128 - 2.0 ** 103                                     # FLT_MAX + half an ulp: rounds (to even) to inf
    xyz = [2147483.6475, -2147483.6475, 2147483.648, -2147483.648, 2147483.6474999, -2147483.6485, -2147483.649, 2147483.647,
           FLT_MAX, -FLT_MAX, nx(FLT_MAX, np.inf), nx(-FLT_MAX, -np.inf), nx(FLT_MAX, 0), nx(half_up, 0), -nx(half_up, 0), half_up,
           -half_up, 2.0 ** 128, 3.5e38, -3.5e38, 1e300,
           2.0 ** -149, -(2.0 ** -149), 2.0 ** -150, 3 * 2.0 ** -150, 2.0 ** -126 - 2.0 ** -149, 2.0 ** -126, 1e-320, -1e-320, 1e-40,
           0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan]
    rows = np.full((len(xyz) + 2, 4), 1.5)
    for i, v in enumerate(xyz):
        rows[i, i % 3] = v
    rows[-2, :3] = [np.nan, -np.nan, np.nan]
    rows[-1, :3] = [-np.nan, 0.0, -0.0]
    rows[:, 3] = np.resize([-1.0, 255.0, 255.5, 256.0, np.nan, 0.0, 254.0, 1.0], len(rows))
    edge = np.concatenate([_edge_values(f64), rows])
    with np.errstate(over="ignore"):
        return edge if f64 else edge.astype(np.float32).astype(np.float64)


def _cs_inputs(f64, with_block=True):
    rng = np.random.default_rng(2202 + f64)
    counts = np.array(CS_COUNTS, np.int64)
    off = np.zeros(len(counts) + 1, np.int64)
    np.cumsum(counts, out=off[1:])
    n = int(off[-1])
    pts = np.column_stack([rng.uniform(-300, 300, (n, 3)), rng.integers(0, 256, n).astype(np.float64)])
    tag = rng.integers(0, 256, n).astype(np.uint8)
    edge = _cs_edges(f64)
    p0 = int(off[CS_BLOCK[0]]) + CS_BLOCK[1]
    pts[p0:p0 + len(edge)] = edge
    tag[p0:p0 + len(edge)] = np.resize([0, 255, 7], len(edge))
    t, p64 = _points(f64, pts)
    if not with_block:
        blk = p64[p0:p0 + len(edge)]
        f2 = row_flags(lambda r: orc.C.quantize_lvx2(r)[1], blk)
        fl = row_flags(lambda r: legacy_records(r, None)[1], blk)
        pts[p0:p0 + len(edge)] = clean(blk, f2 | fl)
        t, p64 = _points(f64, pts)
    ts = np.sort(rng.integers(0, 2 ** 62, len(counts))).astype(np.int64)
    return t, p64, tag, off, ts


@pytest.fixture(scope="module", params=[True, False], ids=["f64", "f32"])
def cs(request):
    t, p64, tag, off, ts = _cs_inputs(request.param)
    rec = {fmt: lvx_cs_records(p64, tag, fmt) for fmt in (C.LVXCS_LVX2, C.LVXCS_LEGACY)}
    return dict(f64=request.param, pts=t, p64=p64, tag=tag, off=off, ts=ts, rec=rec)


@gpu
@needs_gpu
@pytest.mark.parametrize("fmt", [C.LVXCS_LVX2, C.LVXCS_LEGACY], ids=["lvx2", "legacy"])
def test_lvx_cs_whole_file(cs, fmt):
    """Every prefix length moves the records to another byte parity and 16-byte phase; the status is the oracle's per format,
    and 0 on the same stream with the flagged edge rows replaced."""
    from livox_motion_compensation_sim_b200 import ops
    x = cs
    mx = int(np.diff(x["off"]).max())
    rng = np.random.default_rng(5)
    tag_d, off_d, ts_d = dev(x["tag"]), dev(x["off"]), dev(x["ts"])
    for plen in (0, 1, 60, 88, 96):
        prefix = bytes(rng.integers(0, 256, plen).astype(np.uint8))
        want, fl = lvx_cs_expected(x["p64"], x["tag"], x["off"], x["ts"], prefix, fmt, records=x["rec"][fmt])
        data, status = ops.build_lvx_cs(x["pts"], tag_d, off_d, ts_d, prefix, fmt, mx)
        got = data.cpu().numpy()
        assert not first_diff(got, want), (plen, first_diff(got, want))
        assert int(status.item()) == fl, (plen, int(status.item()), fl)
    assert fl == (C.FLAG_NAN | C.FLAG_OVERFLOW)
    t, p64, tag, off, ts = _cs_inputs(x["f64"], with_block=False)
    want, fl = lvx_cs_expected(p64, tag, off, ts, prefix, fmt)
    data, status = ops.build_lvx_cs(t, dev(tag), dev(off), dev(ts), prefix, fmt, mx)
    assert fl == 0 and int(status.item()) == 0
    assert not first_diff(data.cpu().numpy(), want), first_diff(data.cpu().numpy(), want)


@gpu
@needs_gpu
@pytest.mark.parametrize("fmt", [C.LVXCS_LVX2, C.LVXCS_LEGACY], ids=["lvx2", "legacy"])
def test_lvx_cs_stays_inside_its_buffer(cs, fmt):
    x = cs
    L = C.lib()
    fn = L.lmc_lvx_cs_build_f64 if x["f64"] else L.lmc_lvx_cs_build_f32
    prefix = bytes(range(60, 120))
    want, fl = lvx_cs_expected(x["p64"], x["tag"], x["off"], x["ts"], prefix, fmt, records=x["rec"][fmt])
    keep = [dev(x["tag"]), dev(x["off"]), dev(x["ts"])]
    pre = (ctypes.c_uint8 * len(prefix)).from_buffer_copy(prefix)
    B, s = GuardedBytes(len(want), 0), _status()
    F, n = len(x["off"]) - 1, len(x["p64"])
    C.check(fn(x["pts"].data_ptr(), *(k.data_ptr() for k in keep), pre, len(prefix), fmt, B.ptr, n, F, int(np.diff(x["off"]).max()),
               s.data_ptr(), _stream_ptr()))
    assert B.outside_untouched() and not first_diff(B.inside(), want), first_diff(B.inside(), want)
    assert int(s.item()) == fl


# ------------------------------------------------------------------------------------------
# LAS 1.2 PF3
# ------------------------------------------------------------------------------------------
LAS_TILE = 512
LAS_N = 12 * LAS_TILE + 301
LAS_BLOCK = 12 * LAS_TILE - 40                # the edge block straddles the last full tile and the tail


def _las_inputs(f64, with_block=True, cfg="dec", mode=C.LAS_INTENSITY_RAW):
    rng = np.random.default_rng(3303 + f64)
    n = LAS_N
    pts = np.column_stack([rng.uniform(-500, 500, (n, 3)), rng.uniform(0, 1, n)])
    edge = _edge_values(f64)
    pts[LAS_BLOCK:LAS_BLOCK + len(edge)] = edge
    gps = np.sort(rng.uniform(0, 3600, n)).view(np.uint64).copy()
    gps[LAS_BLOCK:LAS_BLOCK + 6] = np.array([np.nan, -0.0, np.inf, 5e-324, -1e300, 0.0]).view(np.uint64)
    gps[LAS_BLOCK + 6] = 0x7FF0000000000123                                 # a signalling NaN's payload travels as bits
    t, p64 = _points(f64, pts)
    if not with_block:
        scale, offset, _ = LAS_CFG[cfg]
        blk = p64[LAS_BLOCK:LAS_BLOCK + len(edge)]
        pts[LAS_BLOCK:LAS_BLOCK + len(edge)] = clean(blk, row_flags(lambda r: orc.C.quantize_las(r, scale, offset, mode)[4], blk))
        t, p64 = _points(f64, pts)
    return t, p64, gps


LAS_RUNS = [("pow2", C.LAS_INTENSITY_UNIT, True), ("pow2", C.LAS_INTENSITY_RAW, False), ("dec", C.LAS_INTENSITY_RAW, True),
            ("dec", C.LAS_INTENSITY_UNIT, False)]


@pytest.fixture(scope="module", params=[True, False], ids=["f64", "f32"])
def las(request):
    t, p64, gps = _las_inputs(request.param)
    return dict(f64=request.param, pts=t, p64=p64, gps=gps)


def _las_kw(cfg, mode, gps_d):
    scale, offset, _ = LAS_CFG[cfg]
    return dict(scale=scale, offset=offset, intensity_mode=mode, gps_time=gps_d)


@gpu
@needs_gpu
@pytest.mark.parametrize("cfg,mode,with_gps", LAS_RUNS, ids=[f"{c}-{'unit' if m == 0 else 'raw'}{'-gps' if g else ''}" for c, m, g in LAS_RUNS])
def test_las_file_ranges_and_shards(las, cfg, mode, with_gps):
    """The whole file (records, header with NumPy's extremes, status); record ranges starting at every p_begin modulo 8 (every
    16-byte phase), each with two full tiles and a tail; a shard set composed as las_pf3_shard does it (records per range, host
    min / max of the returned extremes, one empty shard with the neutral pair, header into the first shard); las_pf3_shard
    itself with torch.distributed uninitialised."""
    from livox_motion_compensation_sim_b200 import ops, sharding
    x = las
    n = len(x["p64"])
    gps_d = dev(x["gps"].view(np.float64)) if with_gps else None
    gps = x["gps"] if with_gps else None
    kw = _las_kw(cfg, mode, gps_d)
    scale, offset = kw["scale"], kw["offset"]
    want, fl = las_expected(x["p64"], scale, offset, mode, gps)
    assert fl != 0
    data, status = ops.build_las_pf3(x["pts"], year=YEAR, day_of_year=DAY, **kw)
    got = data.cpu().numpy()
    assert not first_diff(got[:227], want[:227]), ("header", first_diff(got[:227], want[:227]))
    assert not first_diff(got, want), first_diff(got, want)
    assert int(status.item()) == fl
    X, Y, Z, _, _ = orc.C.quantize_las(x["p64"], scale, offset, mode)
    mx = struct.unpack_from("<6d", got.tobytes(), 179)
    for c, q in enumerate((X, Y, Z)):                                   # exactly, not to a tolerance
        assert mx[2 * c] == las_extreme(q.max(), scale[c], offset[c]) and mx[2 * c + 1] == las_extreme(q.min(), scale[c], offset[c])

    for r in range(8):
        pb = 8 * (600 + 3 * r) + r
        pe = n if r % 2 == 0 else pb + 2 * LAS_TILE + 97 + 13 * r
        pos0 = 227 + 34 * pb
        out, mm, status = ops.las_pf3_records(x["pts"], pb, pe, pos0, **kw)
        part = want[pos0:227 + 34 * pe]
        assert pe - pb > 2 * LAS_TILE and (pe - pb) % LAS_TILE
        assert not first_diff(out.cpu().numpy(), part), ((pb, pe), first_diff(out.cpu().numpy(), part))
        q = [a[pb:pe] for a in (X, Y, Z)]
        assert mm.cpu().numpy().tolist() == [v for a in q for v in (int(a.min()), int(a.max()))], (pb, pe)
        assert int(status.item()) == orc.C.quantize_las(x["p64"][pb:pe], scale, offset, mode)[4], (pb, pe)

    cuts = [0, 1237, 1237, 3001, LAS_BLOCK + 51, n]
    outs, mms = [], []
    for rank, (pb, pe) in enumerate(zip(cuts[:-1], cuts[1:])):
        pos0 = 0 if rank == 0 else 227 + 34 * pb
        out, mm, _ = ops.las_pf3_records(x["pts"], pb, pe, pos0, **kw)
        if pe == pb:
            assert out.numel() == 0 and mm.cpu().numpy().tolist() == [2 ** 31 - 1, -2 ** 31] * 3
        outs.append(out)
        mms.append(mm.cpu().numpy())
    mm = np.stack(mms)
    red = np.empty(6, np.int32)
    red[0::2], red[1::2] = mm[:, 0::2].min(axis=0), mm[:, 1::2].max(axis=0)
    ops.las_pf3_header(outs[0], dev(red), n, scale=scale, offset=offset, year=YEAR, day_of_year=DAY)
    whole = np.concatenate([o.cpu().numpy() for o in outs])
    assert not first_diff(whole, want), first_diff(whole, want)

    out, pos0, status = sharding.las_pf3_shard(x["pts"], 0, n, 0, year=YEAR, day_of_year=DAY, **kw)
    assert pos0 == 0 and int(status.item()) == fl
    assert not first_diff(out.cpu().numpy(), want), first_diff(out.cpu().numpy(), want)


@gpu
@needs_gpu
@pytest.mark.parametrize("f64", [True, False], ids=["f64", "f32"])
def test_las_clean_stream_reports_nothing(f64):
    """The LAS stream with the flagged edge rows replaced: status 0 over the whole file and over a range, same bytes."""
    from livox_motion_compensation_sim_b200 import ops
    for cfg, mode, _ in LAS_RUNS:
        t, p64, gps = _las_inputs(f64, with_block=False, cfg=cfg, mode=mode)
        kw = _las_kw(cfg, mode, dev(gps.view(np.float64)))
        want, fl = las_expected(p64, kw["scale"], kw["offset"], mode, gps)
        data, status = ops.build_las_pf3(t, year=YEAR, day_of_year=DAY, **kw)
        assert fl == 0 and int(status.item()) == 0, (cfg, mode)
        assert not first_diff(data.cpu().numpy(), want), (cfg, mode, first_diff(data.cpu().numpy(), want))
        pb = 8 * 700 + 5
        out, _, status = ops.las_pf3_records(t, pb, len(p64), 227 + 34 * pb, **kw)
        assert int(status.item()) == 0 and not first_diff(out.cpu().numpy(), want[227 + 34 * pb:])


@gpu
@needs_gpu
def test_las_header_extremes_are_numpys():
    """las_pf3_header from integer extremes chosen where fma(X, scale, offset) and NumPy's X * scale + offset differ."""
    from livox_motion_compensation_sim_b200 import ops
    for scale, offset, xs in _header_cases():
        for k in range(0, len(xs) - 1, 2):
            lo, hi = sorted(xs[k:k + 2])
            mins, maxs = [lo, lo - 1, -5], [hi, hi + 1, 7]
            mm = np.array([v for c in range(3) for v in (mins[c], maxs[c])], np.int32)
            sc, of = (scale,) * 3, (offset, offset, 0.5)
            out = torch.full((227,), FILL, dtype=torch.uint8, device=DEV)
            ops.las_pf3_header(out, dev(mm), 12345, scale=sc, offset=of, year=YEAR, day_of_year=DAY)
            want = las_header(12345, sc, of, mins, maxs)
            assert not first_diff(out.cpu().numpy(), want), ((scale, offset, lo, hi), first_diff(out.cpu().numpy(), want))


@gpu
@needs_gpu
def test_las_stays_inside_its_buffers(las):
    """The C entry points on guarded buffers: the whole file at phase 0 and record ranges at every file phase write exactly their
    bytes; a range buffer one byte off its phase is refused with ERR_ALIGN and writes nothing (not even the extremes)."""
    x = las
    L = C.lib()
    n = len(x["p64"])
    cfg, mode = "dec", C.LAS_INTENSITY_RAW
    scale, offset, _ = LAS_CFG[cfg]
    want, fl = las_expected(x["p64"], scale, offset, mode, x["gps"])
    gps_d = dev(x["gps"].view(np.float64))
    sc, of = (ctypes.c_double * 3)(*scale), (ctypes.c_double * 3)(*offset)
    build = L.lmc_las_pf3_build_f64 if x["f64"] else L.lmc_las_pf3_build_f32
    rec = L.lmc_las_pf3_records_f64 if x["f64"] else L.lmc_las_pf3_records_f32
    mm = torch.empty(6, dtype=torch.int32, device=DEV)
    B, s = GuardedBytes(len(want), 0), _status()
    C.check(build(x["pts"].data_ptr(), gps_d.data_ptr(), n, sc, of, mode, YEAR, DAY, B.ptr, mm.data_ptr(), s.data_ptr(), _stream_ptr()))
    assert B.outside_untouched() and not first_diff(B.inside(), want), first_diff(B.inside(), want)
    assert int(s.item()) == fl
    for pb, pe in [(8 * 500 + r, n - 3 * r) for r in range(8)] + [(0, 2 * LAS_TILE + 5)]:
        pos0 = 0 if pb == 0 else 227 + 34 * pb
        nb = 227 + 34 * pe - pos0
        B, s = GuardedBytes(nb, pos0), _status()
        C.check(rec(x["pts"].data_ptr(), gps_d.data_ptr(), n, pb, pe, sc, of, mode, B.ptr, pos0, mm.data_ptr(), s.data_ptr(), _stream_ptr()))
        got = B.inside()
        lo = 227 if pb == 0 else 0                                        # rank 0's header bytes are written later
        assert B.outside_untouched(), (pb, pe)
        assert not first_diff(got[lo:], want[pos0 + lo:pos0 + nb]), ((pb, pe), first_diff(got[lo:], want[pos0 + lo:pos0 + nb]))
        mm_bad = torch.full((6,), -7, dtype=torch.int32, device=DEV)
        Bad, s = GuardedBytes(nb, pos0, shift=1), _status()
        assert rec(x["pts"].data_ptr(), gps_d.data_ptr(), n, pb, pe, sc, of, mode, Bad.ptr, pos0, mm_bad.data_ptr(), s.data_ptr(),
                   _stream_ptr()) == C.ERR_ALIGN
        assert Bad.untouched() and int(s.item()) == 0 and mm_bad.cpu().tolist() == [-7] * 6, (pb, pe)


# ------------------------------------------------------------------------------------------
# ASCII PCD
# ------------------------------------------------------------------------------------------
@gpu
@needs_gpu
@pytest.mark.parametrize("f64", [True, False], ids=["f64", "f32"])
def test_pcd_ascii_shards(f64):
    """pcd_ascii_shard with torch.distributed uninitialised is header + the whole body; odd row cuts placed with file_offsets
    compose to the same file."""
    from livox_motion_compensation_sim_b200 import ops, sharding
    from livox_motion_compensation_sim_b200.simulator import LiDARMotionSimulator
    rng = np.random.default_rng(4404)
    n = 3001
    pts = rng.uniform(-1500, 1500, (n, 4))
    pts[::97, 1] = 1e7
    pts[5::89, 2] = -0.0000004
    t, p64 = _points(f64, pts)
    header = LiDARMotionSimulator._pcd_header(n)
    want = header + "".join("%.6f %.6f %.6f %.6f\n" % tuple(r) for r in p64).encode()
    text, pos0, hdr, status = sharding.pcd_ascii_shard(t, n, 0)
    assert hdr == header and pos0 == len(header) and int(status.item()) == 0
    assert hdr + text.cpu().numpy().tobytes() == want
    cuts = [0, 1, 777, 778, 2001, n]
    texts = [ops.pcd_ascii_body(t[a:b])[0].cpu().numpy() for a, b in zip(cuts[:-1], cuts[1:])]
    off = sharding.file_offsets([len(s) for s in texts], len(header))
    assert int(off[-1]) == len(want)
    img = np.zeros(int(off[-1]), np.uint8)
    img[:len(header)] = np.frombuffer(header, np.uint8)
    for r, s in enumerate(texts):
        p = int(off[r]) + (len(header) if r == 0 else 0)
        img[p:p + len(s)] = s
    assert img.tobytes() == want
