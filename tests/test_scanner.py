"""The scanner (csrc/lmc_scan.cu: k_scan_mark, k_scan_count, k_scan_offsets, k_scan_emit<false|true>, driven by
ops.scan_frames) against scan_frame_np, the restatement of LMC:701-770 with the reference's own NumPy calls, one table row
per scene: environment sizes around the 256-point tile, runs longer than the 65535 frames one launch can carry, per-frame
visible counts around the subsample boundaries, points exactly at range_max / range_min and one ulp off, signed zeros and
points at the sensor position with range_min = 0, identity / exact-zero / negative-first-column rotations, a 360 x 180 FOV
(straight behind, straight up, clip saturating), NaN / inf rows and points a few ulp either side of each FOV limit.

CPU: the restatement replays the reference's golden runs (raw-scan sha256), the C oracle equals it byte for byte on every
scene, and scan_frames refuses points_per_frame < 1.
GPU: the entry points called directly (flags, uncertainty marks, tile offsets, visible counts, recount, emitted rows and
environment indices, nothing written outside the buffers, n_env above LMC_SCAN_MAX_ENV refused before any write), and
ops.scan_frames (every decision and byte, frame offsets, the slot each noise row lands in, the global-RNG stream over frame
chunks, motion-distorted scans)."""
import json
import os
from dataclasses import dataclass

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from oracle import lmc_oracle as orc                                      # checker only

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
MAN = json.load(open(os.path.join(GOLDEN, "MANIFEST.json")))
DEV = "cuda:0"
EDGE_EPS = 1e-9                                                            # ops.scan_frames' default edge_eps_deg
MAX_ENV = 2147483647                                                       # LMC_SCAN_MAX_ENV
GUARD = 256                                                                # sentinel bytes either side of every output
SENTINEL = 0xA5
R_NEG = Rotation.from_euler('xyz', [-2.96843364, 1.59286984, 0.23966151]).as_matrix().reshape(9)   # first column < 0
R_ZERO = np.array([0.0, -1.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0])        # 90 deg about z, exact zeros
R_ID = np.eye(3).reshape(9)


def _cfg(**kw):
    c = dict(range_max=60.0, range_min=0.05, fov_horizontal=70.0, fov_vertical=77.2, points_per_frame=1500)
    c.update(kw)
    return c


@dataclass
class Scene:
    env: np.ndarray                # (M,4) f64
    pos: np.ndarray                # (P,3) the scene's distinct sensor positions
    R: np.ndarray                  # (P,9) row-major
    fp: np.ndarray                 # (F,) pose of every frame
    cfg: dict

    @property
    def F(self):
        return len(self.fp)


def _rot(rng, n, s=0.3):
    return Rotation.from_euler('xyz', rng.normal(0, s, (n, 3))).as_matrix().reshape(n, 9)


def _random(M, F, ppf, seed):
    """Half the rows in front of the sensors, half all around, some beyond range_max; 7 poses repeat over the frames (7 is
    coprime to 65535, so a frame chunk that starts at the wrong pose or flag row shows)."""
    rng = np.random.default_rng(seed)
    h = M // 2
    front = np.column_stack([rng.uniform(2, 50, h), rng.uniform(-25, 25, h), rng.uniform(-25, 25, h)])
    around = rng.uniform(-70, 70, (M - h, 3))
    xyz = np.concatenate([front, around])[rng.permutation(M)]
    env = np.column_stack([xyz, rng.uniform(0.1, 0.9, M)]) if M else np.zeros((0, 4))
    P = min(F, 7)
    return Scene(env, rng.uniform(-3, 3, (P, 3)), _rot(rng, P), np.arange(F) % P, _cfg(points_per_frame=ppf))


def _counts(maxp, seed):
    """Frame f sees exactly counts[f] points (0, 1, max-1, max, max+1, 2max-1, 2max, 2max+1, 3max+2), interleaved with
    points behind it; the blocks of the other frames are out of range.  Rows are shuffled over the tiles."""
    rng = np.random.default_rng(seed)
    counts = [0, 1, maxp - 1, maxp, maxp + 1, 2 * maxp - 1, 2 * maxp, 2 * maxp + 1, 3 * maxp + 2]
    F = len(counts)
    pos = np.column_stack([1000.0 * np.arange(F), np.zeros(F), np.zeros(F)])
    R = _rot(rng, F, 0.05)
    rows = []
    for f, c in enumerate(counts):
        seen = np.column_stack([rng.uniform(5, 40, c), rng.uniform(-0.3, 0.3, (c, 2))])
        seen[:, 1:] *= seen[:, :1]
        behind = np.column_stack([rng.uniform(-40, -5, c + 3), rng.uniform(-5, 5, (c + 3, 2))])
        for blk in (seen, behind):
            rows.append(pos[f] + (R[f].reshape(3, 3) @ blk.T).T)
    xyz = np.concatenate(rows)
    xyz = xyz[rng.permutation(len(xyz))]
    env = np.column_stack([xyz, rng.uniform(0.1, 0.9, len(xyz))])
    return Scene(env, pos, R, np.arange(F), _cfg(points_per_frame=maxp))


def _up(v):
    return np.nextafter(v, np.inf)


def _down(v):
    return np.nextafter(v, -np.inf)


def _range_edges():
    """d2 exactly range_max^2 and one ulp outside / inside; range exactly range_min and one ulp inside."""
    rm, rn = 10.0, 0.5
    rel = [(rm, 0, 0), (0, rm, 0), (8, 0, 6), (0, 8, 6), (6, 0, -8), (_down(rm), 0, 0), (0, _down(rm), 0),
           (rn, 0, 0), (0, rn, 0), (0.3, 0, 0.4), (0, 0.3, -0.4)]
    rel0 = [(_up(rm), 0, 0), (0, _up(rm), 0), (8, 0, _up(6.0)), (0, 8, _up(6.0)), (_down(rn), 0, 0), (0, _down(rn), 0),
            (_up(rn), 0, 0)]                                               # ulp offsets: exact only around the origin
    p1 = np.array([1.25, -3.5, 2.0])
    xyz = [np.array(r, float) for r in rel + rel0] + [p1 + np.array(r, float) for r in rel]
    env = np.column_stack([np.array(xyz), np.linspace(0.1, 0.9, len(xyz))])
    pos = np.array([[0.0, 0, 0], p1, [0.0, 0, 0], p1])
    return Scene(env, pos, np.array([R_ID, R_ID, R_ZERO, R_ZERO]), np.arange(4), _cfg(range_max=rm, range_min=rn))


def _signed_zeros(fov_h=70.0, fov_v=77.2):
    """range_min = 0: points at the sensor position (R with a negative first column: all three products -0.0), environment
    coordinates of -0.0 with sensors on 0.0, under identity, exact-zero and negative-first-column rotations."""
    z, s = 0.0, np.array([3.0, -2.0, 1.5])
    xyz = [s, (-z, -z, -z), (z, z, z), (-z, z, -z), (z, -z, -z), (-z, -z, 2.0), (2.0, -z, -z), (-z, 2.0, -z), (-2.0, -z, z),
           (z, -z, -2.0), s + (1.0, 0.0, 0.0), (5.0, 1.0, -1.0)]
    env = np.column_stack([np.array(xyz, float), np.linspace(0.1, 0.9, len(xyz))])
    rng = np.random.default_rng(41)
    pos = np.array([s, s, [z, z, z], [z, z, z], [z, z, z], [z, z, z], s])
    R = np.array([R_NEG, R_ID, R_ID, R_ZERO, R_NEG, _rot(rng, 1)[0], -R_ID])
    return Scene(env, pos, R, np.arange(len(pos)), _cfg(range_max=90.0, range_min=0.0, fov_horizontal=fov_h, fov_vertical=fov_v))


def _fov_full():
    """360 x 180: straight behind (y = +-0.0), straight up / down, and points along each pose's third axis, whose rotated z
    comes out a rounding above the range so that clip saturates."""
    rng = np.random.default_rng(42)
    P = 5
    R = np.concatenate([R_ID[None], R_ZERO[None], R_NEG[None], _rot(rng, P - 3, 1.0)])
    xyz = [(-5.0, 0.0, 0.0), (-5.0, -0.0, 0.0), (-5.0, 0.0, -0.0), (0.0, 0.0, 5.0), (-0.0, 0.0, 5.0), (0.0, -0.0, -5.0),
           (0.0, 0.0, 0.0)]
    for p in range(P):
        for sgn in (1.0, -1.0):
            xyz += list(sgn * rng.uniform(0.5, 50, 40)[:, None] * R[p].reshape(3, 3)[:, 2][None])
    xyz += list(rng.uniform(-50, 50, (200, 3)))
    env = np.column_stack([np.array(xyz, float), rng.uniform(0.1, 0.9, len(xyz))])
    sc = Scene(env, np.zeros((P, 3)), R, np.arange(P), _cfg(range_min=0.0, fov_horizontal=360.0, fov_vertical=180.0))
    q = []
    for p in range(P):
        rot = (R[p].reshape(3, 3).T @ env[:, :3].T).T
        q.append(np.abs(rot[:, 2]) / np.maximum(np.sqrt(np.sum(env[:, :3] ** 2, axis=1)), 1e-6))
    assert (np.concatenate(q) > 1.0).any(), "no point saturates the clip"
    return sc


def _nan_inf():
    rng = np.random.default_rng(43)
    sc = _random(600, 3, 1500, 44)
    n, i = np.nan, np.inf
    bad = [(n, 0, 0), (10, n, 0), (10, 0, n), (n, n, n), (i, 0, 0), (-i, 0, 0), (10, i, 0), (10, 0, -i), (i, i, i), (i, -i, n)]
    bad = np.column_stack([np.array(bad, float), rng.uniform(0.1, 0.9, len(bad))])
    odd = np.array([[10.0, 0.5, 0.5, n], [12.0, -0.5, 0.5, i], [14.0, 0.5, -0.5, -i]])   # visible, odd intensities
    env = np.concatenate([sc.env[:300], bad, odd, sc.env[300:], bad])
    return Scene(env, np.zeros((3, 3)), np.array([R_ID, R_ZERO, R_NEG]), np.arange(3), sc.cfg)


def _fov_edges():
    """Points a few ulp either side of each azimuth / elevation limit (flagged uncertain and re-decided on the host), and points
    1e-8 .. 1e-5 deg off the limits (decided on the device)."""
    cfg = _cfg()
    h, v = cfg['fov_horizontal'] / 2, cfg['fov_vertical'] / 2
    xyz = []
    for r in (3.0, 17.0, 55.0):
        for lim, ax in ((h, 1), (v, 2)):
            for off in (0.0, 1e-8, -1e-8, 2e-6, -2e-6, 1e-5, -1e-5):
                t = np.deg2rad(lim + off)
                c, s = r * np.cos(t), r * np.sin(t)
                for k in ((-3, -2, -1, 0, 1, 2, 3) if off == 0.0 else (0,)):
                    sk = s
                    for _ in range(abs(k)):
                        sk = _up(sk) if k > 0 else _down(sk)
                    for sgn in (1.0, -1.0):
                        p = [c, 0.0, 0.0]
                        p[ax] = sgn * sk
                        xyz.append(p)
    env = np.column_stack([np.array(xyz), np.linspace(0.1, 0.9, len(xyz))])
    rng = np.random.default_rng(45)
    return Scene(env, np.zeros((2, 3)), np.array([R_ID, _rot(rng, 1, 1e-9)[0]]), np.arange(2), cfg)


SCENES = {
    **{f"M{M}": (lambda M=M: _random(M, 7, 97 if M > 300 else 1500, 100 + M)) for M in (0, 1, 255, 256, 257, 4097)},
    "M60001": lambda: _random(60001, 7, 1500, 7),
    "F1-M4097": lambda: _random(4097, 1, 150, 8),
    "F65535-M300": lambda: _random(300, 65535, 9, 9),
    "F65537-M300": lambda: _random(300, 65537, 9, 10),
    "counts-max7": lambda: _counts(7, 11),
    "counts-max300": lambda: _counts(300, 12),
    "counts-max1": lambda: _counts(1, 13),
    "range-edges": _range_edges,
    "signed-zeros": _signed_zeros,
    "signed-zeros-360x180": lambda: _signed_zeros(360.0, 180.0),
    "fov-360x180": _fov_full,
    "nan-inf": _nan_inf,
    "fov-edges": _fov_edges,
}
SMALL = [k for k in SCENES if not k.startswith("F655")]

_cache = {}


def scene(name):
    if name not in _cache:
        _cache[name] = SCENES[name]()
    return _cache[name]


def expect(name):
    """Per distinct pose: the restatement's visible rows before the subsample, its kept rows and indices, and which rows are
    at least 1e-6 deg from every FOV limit (certain) or within 1e-10 deg of one (near)."""
    key = ("expect", name)
    if key not in _cache:
        sc = scene(name)
        cfg = sc.cfg
        h, v = cfg['fov_horizontal'] / 2, cfg['fov_vertical'] / 2
        out = []
        for p in range(len(sc.pos)):
            vis_idx, _ = orc.scan_frame_np(sc.env, sc.pos[p], sc.R[p], dict(cfg, points_per_frame=len(sc.env) + 1))
            idx, rows = orc.scan_frame_np(sc.env, sc.pos[p], sc.R[p], cfg)
            d2, rng_, az, el = orc.scan_geometry_np(sc.env, sc.pos[p], sc.R[p])
            vis = np.zeros(len(sc.env), bool)
            vis[vis_idx] = True
            with np.errstate(invalid='ignore'):
                live = (d2 <= cfg['range_max'] ** 2) & (rng_ >= cfg['range_min'])
                dist = np.minimum(np.abs(np.abs(az) - h), np.abs(np.abs(el) - v))
                out.append(dict(vis=vis, idx=idx, rows=rows, certain=~live | (dist >= 1e-6), near=live & (dist <= 1e-10)))
        _cache[key] = out
    return _cache[key]


# ------------------------------------------------------------------------------------------
# CPU: the restatement and the C oracle
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["C1a", "C2a", "C3"])
def test_restatement_reproduces_reference_raw_scans(golden, name):
    """scan_frame_np with the reference's per-frame np.random.normal draws, replayed from the saved global-RNG state, gives the
    reference run's raw-scan sha256."""
    import hashlib
    g = golden(f"scan_{name}.npz")
    cfg = json.loads(g['config_json'].tobytes().decode())
    np.random.set_state(('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached'])))
    times = np.linspace(0, cfg['duration'], int(cfg['duration'] * cfg['lidar_fps']))
    idx = orc.pose_lookup_hold_next_np(g['traj_time'], times)
    frames = orc.scan_frames_np(g['environment'], g['traj_position_gps'][idx], g['traj_orientation_imu'][idx], cfg)
    assert hashlib.sha256(np.ascontiguousarray(np.vstack(frames)).tobytes()).hexdigest() == MAN['lmc'][name]['raw_sha256']


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_restatement(name):
    """orc_scan_frame (the kernel's arithmetic in C) == scan_frame_np byte for byte, signed zeros and NaN bits included, on
    the rows at least 1e-6 deg from every FOV limit: closer than that, the C library's atan2 / asin may decide otherwise than
    NumPy's, which is why the scanner re-decides such points on the host (the GPU tests hold it to the restatement there)."""
    sc = scene(name)
    for p, e in enumerate(expect(name)):
        env = sc.env[e['certain']]
        got = orc.C.scan_frame(env, sc.pos[p], sc.R[p], sc.cfg)
        _, want = orc.scan_frame_np(env, sc.pos[p], sc.R[p], sc.cfg)
        assert got.shape == want.shape, (p, got.shape, want.shape)
        assert got.tobytes() == want.tobytes(), p


def test_scene_edges_are_reached():
    """The edge scenes really contain what their names say (against the restatement)."""
    e = expect("range-edges")
    assert e[0]['vis'][[0, 2, 5, 7, 17]].all() and not e[0]['vis'][[11, 13, 15]].any()       # identity: along x
    assert e[2]['vis'][[1, 3, 6, 8]].all() and not e[2]['vis'][[12, 14, 16]].any()           # R_ZERO: along y
    z = expect("signed-zeros")[0]                                      # the sensor-coincident point, R_NEG, default FOV
    assert z['vis'][0] and z['rows'][0, :3].tobytes() == bytes(24)
    assert any(e_['near'].any() for e_ in expect("fov-edges")) and any(e_['near'].any() for e_ in expect("fov-360x180"))
    assert any((~e_['certain'] & ~e_['near']).any() for e_ in expect("fov-edges"))
    c = expect("counts-max7")
    assert [int(x['vis'].sum()) for x in c] == [0, 1, 6, 7, 8, 13, 14, 15, 23]
    assert [len(x['idx']) for x in c] == [0, 1, 6, 7, 7, 7, 7, 7, 7]


def test_scan_frames_refuses_points_per_frame_below_one(monkeypatch):
    """points_per_frame < 1 is a ValueError before any library call (the kept counts would otherwise silently be 0)."""
    import torch
    from livox_motion_compensation_sim_b200 import _capi, ops

    def no_lib():
        raise AssertionError("library called")
    monkeypatch.setattr(_capi, "lib", no_lib)
    env, pos, Rm = torch.zeros((4, 4), dtype=torch.float64), torch.zeros((2, 3), dtype=torch.float64), torch.zeros((2, 9), dtype=torch.float64)
    for ppf in (0, -1):
        with pytest.raises(ValueError, match="points_per_frame"):
            ops.scan_frames(env, pos, Rm, range_max=90.0, range_min=0.05, fov_horizontal=70.0, fov_vertical=77.2,
                            points_per_frame=ppf, noise_std=0.0)


# ------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------
class Guarded:
    """A device buffer with GUARD sentinel bytes either side (32-byte aligned inside)."""

    def __init__(self, torch, nbytes):
        self.n = int(nbytes)
        self.buf = torch.full((2 * GUARD + self.n,), SENTINEL, dtype=torch.uint8, device=DEV)

    @property
    def ptr(self):
        return self.buf.data_ptr() + GUARD

    def host(self, dtype):
        return self.buf[GUARD:GUARD + self.n].cpu().numpy().view(dtype)

    def intact(self):
        b = self.buf.cpu().numpy()
        return bool((b[:GUARD] == SENTINEL).all() and (b[GUARD + self.n:] == SENTINEL).all())

    def untouched(self):
        return bool((self.buf.cpu().numpy() == SENTINEL).all())


def _gpu():
    torch = pytest.importorskip("torch")
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    return torch, C, ops


def _d(torch, a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(DEV)


def _frame_expect(name):
    sc, e = scene(name), expect(name)
    fp = sc.fp
    kept = np.array([len(e[p]['idx']) for p in fp], np.int64)
    off = np.zeros(sc.F + 1, np.int64)
    np.cumsum(kept, out=off[1:])
    return sc, e, off


def _stack(e, fp, key):
    parts = [e[p][key] for p in fp]
    return np.concatenate(parts) if parts else np.zeros((0,) + e[0][key].shape[1:], e[0][key].dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_scan_entry_points(name):
    """lmc_scan_mark / lmc_scan_recount / lmc_scan_emit / lmc_scan_emit_index called directly, every output guarded:
    bit 0 of the flags == the restatement where a point is >= 1e-6 deg from every FOV limit (bit 1 clear there), bit 1 set
    within 1e-10 deg of one, *n_uncertain == the number of bit-1 flags, tile_off / n_visible == host prefix sums of bit 0.
    After the host re-decision of the flagged points (as ops.scan_frames does it), the emitted rows and environment
    indices == the restatement byte for byte."""
    torch, C, ops = _gpu()
    sc, e, off = _frame_expect(name)
    M, F, cfg = len(sc.env), sc.F, sc.cfg
    tiles = (M + C.SCAN_TILE - 1) // C.SCAN_TILE
    L = C.lib()
    env = _d(torch, sc.env if M else np.zeros((1, 4)))
    pos, R = _d(torch, sc.pos[sc.fp]), _d(torch, sc.R[sc.fp])
    flags = Guarded(torch, F * M)
    toff = Guarded(torch, 4 * F * (tiles + 1))
    nvis = Guarded(torch, 4 * F)
    nunc = Guarded(torch, 4)
    args = (float(cfg['range_max'] ** 2), float(cfg['fov_horizontal'] / 2), float(cfg['fov_vertical'] / 2), float(cfg['range_min']))
    C.check(L.lmc_scan_mark(env.data_ptr(), M, pos.data_ptr(), R.data_ptr(), F, *args, EDGE_EPS, flags.ptr, toff.ptr, nvis.ptr,
                            nunc.ptr, ops._stream_ptr()))
    torch.cuda.synchronize()
    assert flags.intact() and toff.intact() and nvis.intact() and nunc.intact()
    fl = flags.host(np.uint8).reshape(F, M)
    vis = _stack(e, sc.fp, 'vis').reshape(F, M) if M else np.zeros((F, 0), bool)
    certain = _stack(e, sc.fp, 'certain').reshape(F, M) if M else np.zeros((F, 0), bool)
    near = _stack(e, sc.fp, 'near').reshape(F, M) if M else np.zeros((F, 0), bool)
    assert set(np.unique(fl)) <= {0, 1, 2, 3}
    bad = np.argwhere(certain & (((fl & 1) != 0) != vis))
    assert len(bad) == 0, f"{len(bad)} decisions differ, first (frame, point) {bad[:5].tolist()}"
    assert not (certain & ((fl & 2) != 0)).any()
    assert ((fl & 2) != 0)[near].all()
    assert int(nunc.host(np.int32)[0]) == int(((fl & 2) != 0).sum())

    def prefix(bits):
        cnt = np.zeros((F, tiles), np.int64)
        if M:
            padded = np.zeros((F, tiles * C.SCAN_TILE), np.int64)
            padded[:, :M] = bits
            cnt = padded.reshape(F, tiles, C.SCAN_TILE).sum(axis=2)
        want = np.zeros((F, tiles + 1), np.int64)
        np.cumsum(cnt, axis=1, out=want[:, 1:])
        return want
    want = prefix(fl & 1)
    assert np.array_equal(toff.host(np.int32).reshape(F, tiles + 1), want)
    assert np.array_equal(nvis.host(np.int32), want[:, -1])
    # the host re-decision of the uncertain points, then the recount (what ops.scan_frames does)
    unc = (fl & 2) != 0
    fl2 = np.where(unc, vis.astype(np.uint8), fl)
    if M:
        flags.buf[GUARD:GUARD + F * M] = _d(torch, fl2.reshape(-1))
    C.check(L.lmc_scan_recount(flags.ptr, M, F, toff.ptr, nvis.ptr, ops._stream_ptr()))
    want = prefix(fl2 & 1)
    assert np.array_equal(toff.host(np.int32).reshape(F, tiles + 1), want) and np.array_equal(want[:, -1], vis.sum(axis=1))
    assert toff.intact() and nvis.intact()
    n = int(off[-1])
    raw, idx = Guarded(torch, 32 * n), Guarded(torch, 8 * n)
    fo = _d(torch, off)
    common = (env.data_ptr(), M, pos.data_ptr(), R.data_ptr(), F, args[0], flags.ptr, toff.ptr, nvis.ptr, fo.data_ptr(),
              int(cfg['points_per_frame']))
    C.check(L.lmc_scan_emit(*common, None, raw.ptr, ops._stream_ptr()))
    C.check(L.lmc_scan_emit_index(*common, idx.ptr, ops._stream_ptr()))
    torch.cuda.synchronize()
    assert raw.intact() and idx.intact() and flags.intact()
    assert np.array_equal(idx.host(np.int64), _stack(e, sc.fp, 'idx'))
    assert raw.host(np.float64).tobytes() == _stack(e, sc.fp, 'rows').tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_scan_frames_vs_restatement(name):
    """ops.scan_frames with noise off: frame offsets and every emitted byte == the restatement, in one chunk and (small scenes)
    in chunks of 3 frames."""
    torch, C, ops = _gpu()
    sc, e, off = _frame_expect(name)
    want = _stack(e, sc.fp, 'rows')
    kw = dict(range_max=sc.cfg['range_max'], range_min=sc.cfg['range_min'], fov_horizontal=sc.cfg['fov_horizontal'],
              fov_vertical=sc.cfg['fov_vertical'], points_per_frame=sc.cfg['points_per_frame'], noise_std=0.0)
    env, pos, R = _d(torch, sc.env.reshape(-1, 4)), _d(torch, sc.pos[sc.fp]), _d(torch, sc.R[sc.fp])
    for mfb in ((1 << 30, 3 * max(len(sc.env), 1)) if sc.F < 1000 else (1 << 30,)):
        raw, fo = ops.scan_frames(env, pos, R, max_flag_bytes=mfb, **kw)
        assert np.array_equal(fo, off)
        assert raw.cpu().numpy().tobytes() == want.tobytes()


def _noise_scene():
    return _counts(40, 21)


def _kw(sc, **over):
    c = sc.cfg
    return dict(dict(range_max=c['range_max'], range_min=c['range_min'], fov_horizontal=c['fov_horizontal'],
                     fov_vertical=c['fov_vertical'], points_per_frame=c['points_per_frame']), **over)


@pytest.mark.gpu
def test_scan_noise_lands_in_its_slot():
    """A noise_fn whose rows are distinct per slot: each emitted row == the restatement row + that slot's noise, one IEEE add,
    over ragged, subsampled frames in chunks of 2."""
    torch, C, ops = _gpu()
    sc = _noise_scene()
    e = [orc.scan_frame_np(sc.env, sc.pos[p], sc.R[p], sc.cfg) for p in sc.fp]
    rng = np.random.default_rng(22)
    drawn = []

    def noise_fn(n):
        drawn.append(rng.uniform(-1e-2, 1e-2, (n, 3)))
        return drawn[-1]
    raw, off = ops.scan_frames(_d(torch, sc.env), _d(torch, sc.pos), _d(torch, sc.R), noise_std=0.02, noise_fn=noise_fn,
                               max_flag_bytes=2 * len(sc.env), **_kw(sc))
    rows = np.concatenate([r for _, r in e])
    noise = np.concatenate(drawn)
    assert len(drawn) == 5 and len(np.unique(noise[:, 0])) == len(noise)
    want = rows.copy()
    want[:, :3] = rows[:, :3] + noise
    assert np.array_equal(np.diff(off), [len(i) for i, _ in e])
    assert raw.cpu().numpy().tobytes() == want.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 2, 3])
def test_scan_global_rng_noise_over_chunks(chunk):
    """Default noise (the global legacy RNG), frames in chunks of `chunk`: the rows and the final np.random.get_state() ==
    the reference's per-frame np.random.normal draws (frames with no point draw nothing)."""
    torch, C, ops = _gpu()
    sc = _noise_scene()
    std = 0.02
    np.random.seed(1234)
    want = []
    for p in sc.fp:
        _, r = orc.scan_frame_np(sc.env, sc.pos[p], sc.R[p], sc.cfg)
        if len(r):
            r[:, :3] += np.random.normal(0, std, (len(r), 3))
        want.append(r)
    state_want = np.random.get_state()
    np.random.seed(1234)
    raw, off = ops.scan_frames(_d(torch, sc.env), _d(torch, sc.pos), _d(torch, sc.R), noise_std=std,
                               max_flag_bytes=chunk * len(sc.env), **_kw(sc))
    state = np.random.get_state()
    assert raw.cpu().numpy().tobytes() == np.concatenate(want).tobytes()
    assert state[0] == state_want[0] and np.array_equal(state[1], state_want[1]) and state[2:] == state_want[2:]


@pytest.mark.gpu
@pytest.mark.parametrize("noise", [False, True], ids=["noise-off", "noise-fn"])
def test_scan_motion_ragged_subsampled_chunked(noise):
    """motion=: ragged (0 .. 3max+2 visible) and subsampled frames in chunks of 2: the environment rows == the restatement's
    kept rows, the point times follow frame_start + (j * period) // m_f, and the rows == odis.C.distort_slerp_f64(env[idx])
    within 1e-10 m, noise added to that in its slot with one IEEE add."""
    from oracle import lmc_oracle_distort as odis
    torch, C, ops = _gpu()
    sc = _noise_scene()
    F = sc.F
    rng = np.random.default_rng(23)
    S = 3 * F + 4
    s_ts = np.cumsum(rng.integers(20_000_000, 60_000_000, S)).astype(np.int64)
    quat = Rotation.from_euler('xyz', np.cumsum(rng.normal(0, 0.01, (S, 3)), axis=0)).as_quat()
    spos = np.column_stack([1000.0 * (s_ts - s_ts[0]) / 100_000_000, rng.normal(0, 0.1, (S, 2))])   # along the frames' blocks
    seg = orc.slerp_segment_table(quat, spos, s_ts)
    period = 100_000_000
    fstart = s_ts[0] + np.arange(F, dtype=np.int64) * period + 7
    e = [orc.scan_frame_np(sc.env, sc.pos[p], sc.R[p], sc.cfg) for p in sc.fp]
    drawn = []

    def noise_fn(n):
        drawn.append(rng.uniform(-1e-2, 1e-2, (n, 3)))
        return drawn[-1]
    args = (_d(torch, sc.env), _d(torch, sc.pos), _d(torch, sc.R))
    kw = _kw(sc, noise_std=0.0, max_flag_bytes=2 * len(sc.env), motion=(_d(torch, s_ts), _d(torch, seg), fstart, period))
    raw0, off, ts, idx = ops.scan_frames(*args, **kw)
    idx_h = idx.cpu().numpy()
    assert np.array_equal(idx_h, np.concatenate([i for i, _ in e]))
    m = np.diff(off)
    assert np.array_equal(m, [len(i) for i, _ in e]) and m.max() == 40 and (m == 0).any()
    fidx = np.repeat(np.arange(F), m)
    assert np.array_equal(ts, fstart[fidx] + ((np.arange(off[-1]) - off[fidx]) * period) // m[fidx])
    want = odis.C.distort_slerp_f64(sc.env[idx_h], ts, s_ts, seg)
    r0 = raw0.cpu().numpy()
    assert np.abs(r0 - want).max() <= 1e-10 and np.array_equal(r0[:, 3], sc.env[idx_h, 3])
    if noise:
        raw1, off1, ts1, idx1 = ops.scan_frames(*args, **dict(kw, noise_std=0.02, noise_fn=noise_fn))
        assert np.array_equal(off1, off) and np.array_equal(ts1, ts) and torch.equal(idx1, idx)
        w = r0.copy()
        w[:, :3] = r0[:, :3] + np.concatenate(drawn)
        assert raw1.cpu().numpy().tobytes() == w.tobytes()


@pytest.mark.gpu
def test_scan_recount_counts_bit_zero():
    """lmc_scan_recount on random flag bytes 0..3: tile_off / n_visible == host prefix sums of bit 0, over a frame count
    past one launch's 65535."""
    torch, C, ops = _gpu()
    rng = np.random.default_rng(24)
    L = C.lib()
    for M, F in ((1, 3), (257, 5), (4097, 2), (300, 65537)):
        tiles = (M + C.SCAN_TILE - 1) // C.SCAN_TILE
        fl = rng.integers(0, 4, (F, M)).astype(np.uint8)
        flags = _d(torch, fl)
        toff, nvis = Guarded(torch, 4 * F * (tiles + 1)), Guarded(torch, 4 * F)
        C.check(L.lmc_scan_recount(flags.data_ptr(), M, F, toff.ptr, nvis.ptr, ops._stream_ptr()))
        torch.cuda.synchronize()
        padded = np.zeros((F, tiles * C.SCAN_TILE), np.int64)
        padded[:, :M] = fl & 1
        want = np.zeros((F, tiles + 1), np.int64)
        np.cumsum(padded.reshape(F, tiles, C.SCAN_TILE).sum(axis=2), axis=1, out=want[:, 1:])
        assert np.array_equal(toff.host(np.int32).reshape(F, tiles + 1), want), (M, F)
        assert np.array_equal(nvis.host(np.int32), want[:, -1]) and toff.intact() and nvis.intact()


@pytest.mark.gpu
def test_scan_refuses_env_above_int32():
    """n_env = LMC_SCAN_MAX_ENV + 1: all four entry points return LMC_ERR_INVALID and write nothing (n_uncertain included),
    with small real buffers behind every pointer."""
    torch, C, ops = _gpu()
    L = C.lib()
    env, pos, R = _d(torch, np.ones((4, 4))), _d(torch, np.zeros((1, 3))), _d(torch, R_ID[None])
    flags, toff, nvis, nunc, raw, idx = (Guarded(torch, 64) for _ in range(6))
    fo = _d(torch, np.array([0, 1], np.int64))
    big = MAX_ENV + 1
    rcs = [L.lmc_scan_mark(env.data_ptr(), big, pos.data_ptr(), R.data_ptr(), 1, 100.0, 35.0, 38.6, 0.05, EDGE_EPS, flags.ptr,
                           toff.ptr, nvis.ptr, nunc.ptr, ops._stream_ptr()),
           L.lmc_scan_recount(flags.ptr, big, 1, toff.ptr, nvis.ptr, ops._stream_ptr()),
           L.lmc_scan_emit(env.data_ptr(), big, pos.data_ptr(), R.data_ptr(), 1, 100.0, flags.ptr, toff.ptr, nvis.ptr, fo.data_ptr(),
                           1, None, raw.ptr, ops._stream_ptr()),
           L.lmc_scan_emit_index(env.data_ptr(), big, pos.data_ptr(), R.data_ptr(), 1, 100.0, flags.ptr, toff.ptr, nvis.ptr,
                                 fo.data_ptr(), 1, idx.ptr, ops._stream_ptr())]
    torch.cuda.synchronize()
    assert rcs == [C.ERR_INVALID] * 4
    assert all(b.untouched() for b in (flags, toff, nvis, nunc, raw, idx))
    # the limit itself is accepted by the argument checks (nothing launched: no frames)
    assert L.lmc_scan_recount(flags.ptr, MAX_ENV, 0, toff.ptr, nvis.ptr, ops._stream_ptr()) == C.OK
