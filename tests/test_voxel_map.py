"""Voxel-grid map (lmc_voxel.cu, ops.voxel_downsample, LiDARMotionSimulator.voxel_map) against the NumPy oracle
(oracle/lmc_oracle_voxel.py), which is itself checked against a per-point dict restatement with exact integer sums.
The device results are compared byte for byte: centroids, counts, point_voxel, V and the status word."""
import ctypes
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import lmc_oracle_voxel as ov                                  # checker only

LEAF_C3, ORIGIN_C3 = 0.5, (0.123456789, 0.234567891, 0.0987654321)      # every C3 environment row >= 8e-6 m from a face


# ---------------------------------------------------------------------------------------------------- clouds
def _cloud(n, seed, extent=20.0, refl=False, dtype=np.float64, center=(0.0, 0.0, 0.0)):
    rng = np.random.default_rng(seed)
    p = np.empty((n, 4), np.float64)
    p[:, :3] = np.asarray(center) + rng.uniform(-extent, extent, (n, 3))
    p[:, 3] = rng.integers(0, 256, n) if refl else rng.uniform(0.0, 1.0, n)
    return p.astype(dtype)


def _on_faces(n, seed, leaf, origin):
    """Points exactly on voxel faces (o + j L, j integer, representable): they belong to the voxel above the face."""
    rng = np.random.default_rng(seed)
    j = rng.integers(-8, 8, (n, 3)).astype(np.float64)
    p = np.empty((n, 4))
    p[:, :3] = np.asarray(origin) + j * np.asarray(leaf)
    p[:, 3] = rng.uniform(0, 1, n)
    return p


def _edge_block():
    """Rows at the edges of the contract (leaf 1, origin 0): the q clamp, the key range, non-finite values, |I| near 256."""
    tiny = 5e-324
    kl = float(1 << 20)
    rows = [[-tiny, 0.5, 0.5, 0.5], [0.5, -tiny, -tiny, 0.25],                       # u = -tiny: k = -1, q = 2^32 - 1
            [-kl, 0.0, 0.0, 0.1], [kl - 0.5, kl - 0.5, -kl, 0.2],                   # keys -2^20 and 2^20 - 1: kept
            [-kl - 0.5, 0.0, 0.0, 0.3], [0.0, kl, 0.0, 0.3], [0.0, 0.0, -kl - 1, 0.3],   # -2^20 - 1 and 2^20: dropped
            [0.5, 0.5, 0.5, np.nextafter(256.0, 0.0)], [0.5, 0.5, 0.5, -np.nextafter(256.0, 0.0)],   # |I| = 256 - ulp: kept
            [0.5, 0.5, 0.5, 256.0], [0.5, 0.5, 0.5, -256.0]]                         # |I| = 256: dropped
    for c in range(4):
        for v in (np.nan, np.inf, -np.inf):
            r = [0.5, 0.5, 0.5, 0.5]
            r[c] = v
            rows.append(r)
    return np.array(rows, np.float64)


# ---------------------------------------------------------------------------------------------------- CPU: the oracle
def _dict_voxels(pts, leaf, origin):
    """Per-point Python restatement: key -> [first index, n, S_x, S_y, S_z, S_I] with Python ints, exact means."""
    L = [float(v) for v in np.broadcast_to(np.asarray(leaf, np.float64), (3,))]
    o = [float(v) for v in np.broadcast_to(np.asarray(origin, np.float64), (3,))]
    vox, flags, pv_key = {}, 0, []
    for i, row in enumerate(np.asarray(pts).astype(np.float64)):
        x = [float(v) for v in row]
        if not all(math.isfinite(v) for v in x):
            flags |= ov.FLAG_NAN
            pv_key.append(None)
            continue
        u = [(x[c] - o[c]) / L[c] for c in range(3)]
        k = [math.floor(v) if math.isfinite(v) else None for v in u]
        if any(kk is None or not -(1 << 20) <= kk < (1 << 20) for kk in k) or abs(x[3]) >= 256.0:
            flags |= ov.FLAG_OVERFLOW
            pv_key.append(None)
            continue
        q = [min(int((u[c] - k[c]) * 2.0 ** 32), 2 ** 32 - 1) for c in range(3)]
        qi = round(x[3] * 2.0 ** 24)                                   # Python round: half to even
        key = tuple(k)
        e = vox.setdefault(key, [i, 0, 0, 0, 0, 0])
        e[1] += 1
        for c in range(3):
            e[2 + c] += q[c]
        e[5] += qi
        pv_key.append(key)
    keys = sorted(vox, key=lambda kk: vox[kk][0])
    rank = {kk: r for r, kk in enumerate(keys)}
    cent = np.empty((len(keys), 4))
    cnt = np.empty(len(keys), np.int32)
    for r, kk in enumerate(keys):
        _, n, sx, sy, sz, si = vox[kk]
        assert max(abs(sx), abs(sy), abs(sz), abs(si)) < 2 ** 53                # f64(S) exact: one rounding of S / n
        for c, s in enumerate((sx, sy, sz)):
            cent[r, c] = o[c] + (kk[c] + float(Fraction(s, n)) * 2.0 ** -32) * L[c]
        cent[r, 3] = float(Fraction(si, n)) * 2.0 ** -24
        cnt[r] = n
    pv = np.array([-1 if kk is None else rank[kk] for kk in pv_key], np.int32)
    return cent, cnt, pv, flags


def _cpu_cases():
    neg = _cloud(3000, 1, extent=3.0, center=(-10.0, -5.0, -2.0))
    yield "negative", neg, 0.5, (0.0, 0.0, 0.0)
    yield "faces", _on_faces(2000, 2, 0.25, (0.5, -1.0, 2.0)), 0.25, (0.5, -1.0, 2.0)
    yield "anisotropic", _cloud(4000, 3, extent=4.0), (0.3, 0.7, 1.9), (0.0, 0.0, 0.0)
    yield "origin", _cloud(4000, 4, extent=4.0, center=(100.0, -200.0, 3.0)), 0.4, (97.31, -203.17, 1.01)
    yield "reflectivity", _cloud(4000, 5, extent=4.0, refl=True), 1.0, (0.0, 0.0, 0.0)
    yield "f32", _cloud(4000, 6, extent=4.0, dtype=np.float32), 0.2, (0.05, 0.0, -0.05)
    yield "edges", _edge_block(), 1.0, (0.0, 0.0, 0.0)


@pytest.mark.parametrize("name,pts,leaf,origin", list(_cpu_cases()), ids=[c[0] for c in _cpu_cases()])
def test_oracle_vs_dict(name, pts, leaf, origin):
    cent, cnt, pv, fl = ov.voxel_downsample(pts, leaf, origin)
    dc, dn, dpv, dfl = _dict_voxels(pts, leaf, origin)
    if pts.dtype == np.float32:
        dc = dc.astype(np.float32)
    assert cent.dtype == pts.dtype and cent.tobytes() == dc.tobytes()
    assert np.array_equal(cnt, dn) and np.array_equal(pv, dpv) and fl == dfl
    assert 1 < len(cnt) < len(pts)                                          # (voxels shared and distinct)


def test_oracle_edge_values():
    e = _edge_block()
    keep, k, q, qi, fl = ov.point_keys(e, 1.0)
    assert fl == ov.FLAG_NAN | ov.FLAG_OVERFLOW
    assert keep[:4].all() and not keep[4:7].any() and keep[7:9].all() and not keep[9:].any()
    assert k[0, 0] == -1 and q[0, 0] == 2 ** 32 - 1 and k[1, 1] == k[1, 2] == -1 and q[1, 1] == q[1, 2] == 2 ** 32 - 1
    assert k[2, 0] == -(1 << 20) and k[3, 0] == k[3, 1] == (1 << 20) - 1 and k[3, 2] == -(1 << 20)
    assert qi[7] == round(float(np.nextafter(256.0, 0.0)) * 2 ** 24) and qi[8] == -qi[7]
    assert (ov.point_keys(e[:4], 1.0)[4], ov.point_keys(e[4:7], 1.0)[4], ov.point_keys(e[9:11], 1.0)[4]) == (0, ov.FLAG_OVERFLOW, ov.FLAG_OVERFLOW)
    for c in range(4):                                                    # one non-finite value per column: NAN only
        assert ov.point_keys(e[11 + 3 * c: 14 + 3 * c], 1.0)[4] == ov.FLAG_NAN
    cent, cnt, pv, _ = ov.voxel_downsample(e, 1.0)
    assert np.array_equal(pv[4:7], [-1] * 3) and (pv[9:] == -1).all() and (pv[:4] >= 0).all()
    assert cent[pv[2], 0] == -float(1 << 20) and cent[pv[0], 0] == -2.0 ** -32      # the clamp: just below the face


def _keyed(pts, leaf, origin, cent, cnt, pv):
    """key -> (centroid bytes, count) of a map, the key taken from any member point."""
    keep, k, _, _, _ = ov.point_keys(pts, leaf, origin)
    keys = ov.pack_keys(k)
    kr = np.empty(len(cnt), np.int64)
    kr[pv[keep]] = keys[keep]
    return {int(kk): (cent[r].tobytes(), int(cnt[r])) for r, kk in enumerate(kr)}


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_oracle_permutation_invariance(dtype):
    p = _cloud(20000, 7, extent=3.0, dtype=dtype)
    perm = np.random.default_rng(8).permutation(len(p))
    a = ov.voxel_downsample(p, 0.3, (0.1, 0.2, 0.3))
    b = ov.voxel_downsample(p[perm], 0.3, (0.1, 0.2, 0.3))
    assert _keyed(p, 0.3, (0.1, 0.2, 0.3), a[0], a[1], a[2]) == _keyed(p[perm], 0.3, (0.1, 0.2, 0.3), b[0], b[1], b[2])


def test_c3_environment_clear_of_voxel_faces(golden):
    """The grid of the C3 Mode C map test: no environment row within 1e-6 m of a voxel face (Mode C recovers the rows
    to 1e-9 m), so the recovered points and the environment rows fill the same voxels."""
    env = golden("scan_C3.npz")['environment']
    u = (env[:, :3] - np.asarray(ORIGIN_C3)) / LEAF_C3
    fr = u - np.floor(u)
    assert np.minimum(fr, 1.0 - fr).min() * LEAF_C3 > 1e-6


# ---------------------------------------------------------------------------------------------------- GPU
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _check_device(pts, leaf, origin):
    from livox_motion_compensation_sim_b200 import ops
    cent, cnt, pv, status = ops.voxel_downsample(_dev(pts), leaf, origin, point_voxel=True)
    want = ov.voxel_downsample(pts, leaf, origin)
    got = (cent.cpu().numpy(), cnt.cpu().numpy(), pv.cpu().numpy(), int(status.item()))
    assert got[0].dtype == want[0].dtype and got[0].shape == want[0].shape
    assert got[0].tobytes() == want[0].tobytes(), "centroids"
    assert np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]) and got[3] == want[3]
    return got


def _one_voxel():
    p = np.empty((1_000_000, 4))
    p[:, :3] = np.random.default_rng(9).uniform(0.0, 0.99, (1_000_000, 3))
    p[:, 3] = np.random.default_rng(10).integers(0, 256, 1_000_000)
    return p, 1.0, (0.0, 0.0, 0.0)


def _one_per_voxel():
    j = np.arange(300_000)
    g = np.stack([j % 100, (j // 100) % 100, j // 10_000, np.full(len(j), 0.5)], 1).astype(np.float64)
    g[:, :3] = g[:, :3] * 0.2 + 0.1
    return g[np.random.default_rng(11).permutation(len(j))], 0.2, (0.0, 0.0, 0.0)


def _edges_in_stream():
    p = _cloud(200_000, 14, extent=8.0)
    e = _edge_block()
    p[np.sort(np.random.default_rng(15).choice(len(p), len(e), replace=False))] = e
    return p, 1.0, (0.0, 0.0, 0.0)


GPU_CASES = {
    "single": lambda: (np.array([[1.25, -2.5, 3.75, 0.5]]), 0.5, (0.0, 0.0, 0.0)),
    "one_voxel_1e6": _one_voxel,
    "one_per_voxel": _one_per_voxel,
    **{f"n{n}": (lambda n=n: (_cloud(n, n, extent=2.0), 0.5, (0.0, 0.0, 0.0)))
       for n in (255, 256, 257, 511, 1023, 1024, 1025, 262_143, 262_145)},
    **{f"leaf{leaf}": (lambda leaf=leaf: (_cloud(400_000, 12, extent=60.0, refl=leaf == 5.0), leaf, (0.0, 0.0, 0.0)))
       for leaf in (0.01, 0.2, 5.0)},
    "utm": lambda: (_cloud(500_000, 13, extent=50.0, center=(5.0e5, 4.4e6, 50.0)), 0.1, (5.0e5 - 37.5, 4.4e6 + 12.25, 0.0)),
    "edges_in_stream": _edges_in_stream,
}


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_device_vs_oracle(name, f32):
    pts, leaf, origin = GPU_CASES[name]()
    _check_device(pts.astype(np.float32) if f32 else pts, leaf, origin)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_empty_input(dtype):
    import torch
    from livox_motion_compensation_sim_b200 import ops
    cent, cnt, pv, status = ops.voxel_downsample(torch.empty((0, 4), dtype=getattr(torch, dtype), device="cuda:0"), 0.5, point_voxel=True)
    assert cent.shape == (0, 4) and cent.dtype == getattr(torch, dtype) and cnt.shape == (0,) and pv.shape == (0,) and int(status.item()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_deterministic_and_permutation_invariant(f32):
    from livox_motion_compensation_sim_b200 import ops
    p = _cloud(2_000_000, 16, extent=30.0, dtype=np.float32 if f32 else np.float64)
    runs = [ops.voxel_downsample(_dev(p), 0.25, (0.1, 0.0, -0.1), point_voxel=True) for _ in range(2)]
    a = [t.cpu().numpy() for t in runs[0][:3]]
    b = [t.cpu().numpy() for t in runs[1][:3]]
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    perm = np.random.default_rng(17).permutation(len(p))
    c = [t.cpu().numpy() for t in ops.voxel_downsample(_dev(p[perm]), 0.25, (0.1, 0.0, -0.1), point_voxel=True)[:3]]
    assert _keyed(p, 0.25, (0.1, 0.0, -0.1), *a) == _keyed(p[perm], 0.25, (0.1, 0.0, -0.1), *c)


G = 4096                                                                  # sentinel elements on each side


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_abi_guard_bands_and_refusals(f32):
    import torch
    from livox_motion_compensation_sim_b200 import _capi as C
    from tests.test_kernel_variants import Guarded
    L = C.lib()
    fdt = torch.float32 if f32 else torch.float64
    sfx = "f32" if f32 else "f64"
    index, reduce = getattr(L, f"lmc_voxel_index_{sfx}"), getattr(L, f"lmc_voxel_reduce_{sfx}")
    pts_h = _cloud(70_001, 18, extent=3.0, dtype=np.float32 if f32 else np.float64)
    pts_h[123] = [np.nan, 0, 0, 0]
    n = len(pts_h)
    pts = _dev(pts_h)
    want = ov.voxel_downsample(pts_h, 0.5, (0.0, 0.1, 0.2))
    V = len(want[1])
    d3 = lambda *v: (ctypes.c_double * 3)(*v)                              # noqa: E731
    leaf, org = d3(0.5, 0.5, 0.5), d3(0.0, 0.1, 0.2)
    ws = torch.empty(L.lmc_voxel_workspace_bytes(n), dtype=torch.uint8, device="cuda:0")
    nv = torch.full((3,), -5, dtype=torch.int64, device="cuda:0")
    status = torch.zeros(3, dtype=torch.int32, device="cuda:0")
    out, cnt, pv = Guarded(V, (4,), fdt, -123.0), Guarded(V, (), torch.int32, -77), Guarded(n, (), torch.int32, -77)
    st = torch.cuda.current_stream().cuda_stream

    def idx(p=pts.data_ptr(), nn=n, lf=leaf, og=org, w=ws.data_ptr(), v=nv[1:].data_ptr(), s=status[1:].data_ptr()):
        return index(p, nn, lf, og, w, v, s, st)

    def red(p=pts.data_ptr(), nn=n, lf=leaf, og=org, w=ws.data_ptr(), vv=V, o=out.view.data_ptr(), c=cnt.view.data_ptr(), q=pv.view.data_ptr()):
        return reduce(p, nn, lf, og, w, vv, o, c, q, st)

    def untouched():
        torch.cuda.synchronize()
        return (out.untouched_outside(0, 0) and cnt.untouched_outside(0, 0) and pv.untouched_outside(0, 0)
                and (nv == -5).all().item() and (status == 0).all().item())

    nan, inf = float("nan"), float("inf")
    bad_index = [dict(nn=-1), dict(nn=1 << 31), dict(lf=d3(0.5, 0.0, 0.5)), dict(lf=d3(-0.5, 0.5, 0.5)), dict(lf=d3(nan, 0.5, 0.5)),
                 dict(lf=d3(0.5, 0.5, inf)), dict(og=d3(0.0, nan, 0.0)), dict(og=d3(0.0, 0.0, -inf)), dict(p=None), dict(w=None),
                 dict(v=None), dict(s=None), dict(lf=None), dict(og=None)]
    for kw in bad_index:
        assert idx(**kw) == C.ERR_INVALID, kw
    assert idx(p=pts.data_ptr() + 16) == C.ERR_ALIGN and idx(w=ws.data_ptr() + 8) == C.ERR_ALIGN
    assert untouched()
    assert idx() == C.OK
    torch.cuda.synchronize()
    assert int(nv[1].item()) == V and int(nv[0].item()) == int(nv[2].item()) == -5
    assert int(status[1].item()) == want[3] == C.FLAG_NAN and int(status[0].item()) == int(status[2].item()) == 0
    bad_reduce = [dict(vv=-1), dict(vv=n + 1), dict(o=None), dict(c=None), dict(nn=-1), dict(lf=d3(0.5, 0.5, 0.0)), dict(og=d3(inf, 0, 0)),
                  dict(w=None), dict(p=None)]
    for kw in bad_reduce:
        assert red(**kw) == C.ERR_INVALID, kw
    assert red(o=out.view.data_ptr() + 16) == C.ERR_ALIGN and red(q=pv.view.data_ptr() + 4) == C.ERR_ALIGN
    torch.cuda.synchronize()
    assert out.untouched_outside(0, 0) and cnt.untouched_outside(0, 0) and pv.untouched_outside(0, 0)
    assert red() == C.OK
    torch.cuda.synchronize()
    assert out.untouched_outside(0, V) and cnt.untouched_outside(0, V) and pv.untouched_outside(0, n)
    assert out.view.cpu().numpy().tobytes() == want[0].tobytes()
    assert np.array_equal(cnt.view.cpu().numpy(), want[1]) and np.array_equal(pv.view.cpu().numpy(), want[2])
    assert L.lmc_voxel_workspace_bytes(-1) == C.ERR_INVALID and L.lmc_voxel_workspace_bytes(1 << 31) == C.ERR_INVALID


@pytest.mark.gpu
def test_full_size_m1h():
    """The M-1H aligned cloud (3.6e8 float4 points, a 2^30-slot table): whole-map properties, and 1000 sampled voxels
    recomputed by the oracle from their member points."""
    import torch
    import bench
    from livox_motion_compensation_sim_b200 import ops, synth
    dev = torch.device("cuda:0")
    st = synth.make_stream(bench.N_FRAMES, bench.PTS_PER_FRAME, bench.SEED, device=dev, dtype=torch.float32)
    N = st.n_points
    out, _ = ops.deskew_slerp(st.pts, st.ts_off, _dev(st.frame_off), _dev(st.frame_start), _dev(st.sample_ts), _dev(st.seg))
    leaf, origin = 0.5, tuple(float(v) for v in st.seg[0, 9:12])                # the first pose sample's position
    cent, cnt, pv, status = ops.voxel_downsample(out, leaf, origin, point_voxel=True)
    V = cnt.shape[0]
    assert int(status.item()) == 0 and 0 < V < N
    assert int(cnt.sum(dtype=torch.int64).item()) == N
    pvl = pv.long()
    assert torch.equal(torch.bincount(pvl, minlength=V), cnt.long())
    first = torch.full((V,), N, dtype=torch.int64, device=dev).scatter_reduce_(0, pvl, torch.arange(N, device=dev), "amin")
    assert bool((first[1:] > first[:-1]).all().item())
    del pvl, first
    sample = torch.from_numpy(np.sort(np.random.default_rng(19).choice(V, 1000, replace=False))).to(dev)
    members = torch.nonzero(torch.isin(pv, sample.int()), as_tuple=True)[0]
    sub = out[members].cpu().numpy()
    sub_pv = pv[members].cpu().numpy()
    c, n, spv, fl = ov.voxel_downsample(sub, leaf, origin)
    assert fl == 0 and len(n) == 1000
    s_h = sample.cpu().numpy()
    assert np.array_equal(s_h[spv], sub_pv)                                     # same voxels, same order (first occurrence)
    assert c.tobytes() == cent[sample].cpu().numpy().tobytes() and np.array_equal(n, cnt[sample].cpu().numpy())


@pytest.mark.gpu
def test_c3_map_sharpness_and_mode_c_map(golden):
    """C3 with motion distortion: the Mode C map occupies fewer voxels than the frame-rigid one; with noise off it has
    exactly the voxels and counts of the environment rows the scans observed (test_c3_environment_clear_of_voxel_faces)."""
    from tests.test_motion_distortion import _c3_run
    sim_s, res_s, _, _, _ = _c3_run(golden, motion_distortion=True, pose_interpolation='slerp')
    sim_h, res_h, _, _, _ = _c3_run(golden, motion_distortion=True)
    ms, mh = sim_s.voxel_map(res_s, LEAF_C3, ORIGIN_C3), sim_h.voxel_map(res_h, LEAF_C3, ORIGIN_C3)
    print(f"C3 distorted, leaf {LEAF_C3} m: slerp {len(ms['counts'])} voxels, hold_next {len(mh['counts'])} voxels")
    assert len(ms['counts']) < len(mh['counts'])
    assert ms['counts'].sum() == mh['counts'].sum() == sum(len(a) for a in res_s['aligned_pointclouds'])

    sim, res, _, g, _ = _c3_run(golden, motion_distortion=True, lidar_range_noise=0.0, pose_interpolation='slerp')
    m = sim.voxel_map(res, LEAF_C3, ORIGIN_C3)
    idx = np.concatenate([s['env_index'] for s in res['raw_scans']])
    env_pts = g['environment'][idx]
    want_c, want_n, want_pv, _ = ov.voxel_downsample(env_pts, LEAF_C3, ORIGIN_C3)
    assert np.array_equal(m['counts'], want_n)
    aligned = np.vstack(res['aligned_pointclouds'])
    assert np.array_equal(ov.pack_keys(ov.point_keys(aligned, LEAF_C3, ORIGIN_C3)[1]), ov.pack_keys(ov.point_keys(env_pts, LEAF_C3, ORIGIN_C3)[1]))
    assert np.abs(m['points'] - want_c).max() <= 1e-8
    assert m['points'].tobytes() == ov.voxel_downsample(aligned, LEAF_C3, ORIGIN_C3)[0].tobytes()
