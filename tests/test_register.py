"""Prior point map, exact fixed-radius nearest neighbours and per-frame pose refinement (lmc_register.cu, ops.build_point_map /
map_nearest / register_frames, LiDARMotionSimulator.register_scans) against the NumPy oracle (oracle/lmc_oracle_register.py),
which is itself checked against scipy's cKDTree and Rotation."""
import ctypes
import json

import numpy as np
import pytest

from oracle import lmc_oracle as orc                                       # checker only
from oracle import lmc_oracle_register as org
from oracle import lmc_oracle_voxel as ov


def _cloud(n, seed, extent=5.0, center=(0.0, 0.0, 0.0)):
    rng = np.random.default_rng(seed)
    p = np.empty((n, 4))
    p[:, :3] = np.asarray(center) + rng.uniform(-extent, extent, (n, 3))
    p[:, 3] = rng.uniform(0.0, 1.0, n)
    return p


def _perturb(pose, seed, dt=0.03, dr=0.01):
    """A pose row moved by dt metres and rotated by dr radians about a random axis (left-multiplied)."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    u, v = rng.normal(size=3), rng.normal(size=3)
    out = np.array(pose, np.float64)
    out[:9] = (Rotation.from_rotvec(dr * v / np.linalg.norm(v)).as_matrix() @ out[:9].reshape(3, 3)).reshape(9)
    out[9:12] += dt * u / np.linalg.norm(u)
    return out


def _c3_frames(golden, frames=(3, 7, 13)):
    """Noise-free C3 scans from the golden trajectory's poses: (env, points, frame_off, true pose table)."""
    from scipy.spatial.transform import Rotation
    g = golden("scan_C3.npz")
    cfg = json.loads(bytes(g['config_json']).decode())
    env = g['environment']
    pts, off, poses = [], [0], []
    for k in frames:
        pos, R = g['traj_position_gps'][k * 10], Rotation.from_euler('xyz', g['traj_orientation_imu'][k * 10]).as_matrix()
        _, rows = orc.scan_frame_np(env, pos, R, cfg)
        pts.append(rows)
        off.append(off[-1] + len(rows))
        poses.append(np.r_[R.reshape(9), pos])
    return env, np.vstack(pts), np.array(off, np.int64), np.array(poses)


# ---------------------------------------------------------------------------------------------------- CPU: the oracle
@pytest.mark.parametrize("case", ["random", "c3"])
def test_oracle_nearest_vs_ckdtree(case, golden):
    from scipy.spatial import cKDTree
    if case == "random":
        mp, q, leaf, origin = _cloud(20_000, 1), _cloud(5_000, 2, extent=6.0), 0.7, (0.1, -0.2, 0.3)
    else:
        env, pts, _, poses = _c3_frames(golden, (5,))
        mp, leaf, origin = env, 1.0, tuple(poses[0, 9:12])
        q = pts.copy()
        q[:, :3] = org.transform(pts, _perturb(poses[0], 3))[1]
    M = org.build_map(mp, leaf, origin)
    idx, d2, fl = org.nearest(q, M, leaf)
    dist, j = cKDTree(mp[:, :3]).query(q[:, :3], distance_upper_bound=leaf)
    assert fl == 0
    found = np.isfinite(dist)
    assert np.array_equal(found, idx >= 0) and found.sum() > len(q) // 2
    assert np.abs(np.sqrt(d2[found]) - dist[found]).max() <= 1e-12
    dist2, j2 = cKDTree(mp[:, :3]).query(q[found, :3], k=2)
    untied = dist2[:, 1] - dist2[:, 0] > 1e-9
    assert np.array_equal(idx[found][untied], j[found][untied])


def test_oracle_map_csr():
    p = _cloud(3000, 4, extent=2.0)
    M = org.build_map(p, 0.5, (0.0, 0.1, 0.2))
    assert np.array_equal(np.sort(M['index']), np.arange(len(p)))
    keep, k, _, _, _ = ov.point_keys(M['pts'], 0.5, (0.0, 0.1, 0.2))
    keys = ov.pack_keys(k)
    V = len(M['vox_off']) - 1
    r = np.repeat(np.arange(V), np.diff(M['vox_off']))
    assert keep.all() and np.array_equal(keys, M['keys'][r]) and len(np.unique(M['keys'])) == V
    with pytest.raises(ValueError):
        org.build_map(np.array([[np.nan, 0, 0, 0]]), 1.0)
    with pytest.raises(OverflowError):
        org.build_map(np.array([[3e6, 0, 0, 0]]), 1.0)


def test_oracle_registration_recovers_c3_poses(golden):
    """Noise off, 3 cm / 0.01 rad off, 1 m gate: the true pose to 1e-9 m and 1e-12 rad within 30 iterations."""
    from scipy.spatial.transform import Rotation
    env, pts, off, poses = _c3_frames(golden)
    init = np.array([_perturb(p, 10 + i) for i, p in enumerate(poses)])
    M = org.build_map(env, 1.0, tuple(poses[0, 9:12]))
    pose, inl, rms, its, fl = org.register_frames(pts, off, init, M, 1.0)
    assert (fl == org.CONVERGED).all() and (its <= 30).all()
    assert np.abs(pose[:, 9:12] - poses[:, 9:12]).max() <= 1e-9
    dR = Rotation.from_matrix(pose[:, :9].reshape(-1, 3, 3)) * Rotation.from_matrix(poses[:, :9].reshape(-1, 3, 3)).inv()
    assert np.linalg.norm(dR.as_rotvec(), axis=1).max() <= 1e-12
    assert np.array_equal(inl, np.diff(off)) and rms.max() <= 1e-9


def test_scan_pose_source_checks():
    from livox_motion_compensation_sim_b200 import LiDARMotionSimulator

    class WithScan:
        trajectory = {}
        environment = np.zeros((1, 4))

        def scan(self, i, t, pose):                                        # pragma: no cover
            return np.zeros((0, 4))
    with pytest.raises(ValueError, match="scan_pose_source"):
        LiDARMotionSimulator({'scan_pose_source': 'truth', 'device': 'cpu'}).run_simulation(WithScan())
    with pytest.raises(ValueError, match="device scanner"):
        LiDARMotionSimulator({'scan_pose_source': 'true', 'device': 'cpu'}).run_simulation(WithScan())
    assert LiDARMotionSimulator({'device': 'cpu'}).config['scan_pose_source'] == 'measured'


# ---------------------------------------------------------------------------------------------------- GPU
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _check_map(mp, leaf, origin):
    from livox_motion_compensation_sim_b200 import ops
    pm = ops.build_point_map(_dev(mp), leaf, origin)
    M = org.build_map(mp, leaf, origin)
    assert pm.pts.cpu().numpy().tobytes() == M['pts'].tobytes()
    assert np.array_equal(pm.index.cpu().numpy(), M['index']) and np.array_equal(pm.vox_off.cpu().numpy(), M['vox_off'])
    assert np.array_equal(np.sort(pm.index.cpu().numpy()), np.arange(len(mp)))
    keys, ranks = pm.keys.cpu().numpy(), pm.ranks.cpu().numpy()
    full = keys != -1
    V = len(M['vox_off']) - 1
    assert full.sum() == V and np.array_equal(np.sort(ranks[full]), np.arange(V))
    assert np.array_equal(M['keys'][ranks[full]], keys[full])
    return pm, M


MAP_CASES = {
    "empty": lambda: (np.zeros((0, 4)), 1.0, (0.0, 0.0, 0.0)),
    "one": lambda: (np.array([[0.3, -0.2, 0.1, 0.5]]), 1.0, (0.0, 0.0, 0.0)),
    "one_voxel_1e5": lambda: (np.c_[np.random.default_rng(5).uniform(0.0, 0.99, (100_000, 3)), np.zeros(100_000)], 1.0, (0.0, 0.0, 0.0)),
    "random": lambda: (_cloud(200_000, 6, extent=20.0), 0.5, (0.1, 0.2, 0.3)),
    "utm": lambda: (_cloud(100_000, 7, extent=30.0, center=(5.0e5, 4.4e6, 50.0)), 1.0, (5.0e5 - 3.25, 4.4e6 + 1.5, 40.0)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MAP_CASES))
def test_build_point_map(name):
    _check_map(*MAP_CASES[name]())


def _nearest_queries(leaf, origin, rng):
    """Queries on cell faces and corners, near map points, equidistant pairs, exact-gate and beyond-gate distances,
    non-finite rows and cells outside the key range (the map is on an integer lattice of spacing leaf / 4)."""
    o = np.asarray(origin)
    q = [o + rng.integers(-12, 12, (400, 3)) * leaf,                                   # corners
         o + np.c_[rng.integers(-12, 12, (400, 1)) * leaf, rng.uniform(-3, 3, (400, 2))],   # faces
         o + rng.uniform(-3, 3, (2000, 3))]
    q = np.vstack(q)
    q4 = np.c_[q, np.zeros(len(q))]
    bad = np.array([[np.nan, 0, 0, 0], [0, np.inf, 0, 0], [0, 0, -np.inf, 0], [3e6, 0, 0, 0], [0, -3e6, 0, 0]], np.float64)
    return np.vstack([q4, bad])


def _lattice_map(leaf, origin, rng):
    """Map points on a lattice of spacing leaf / 4 (duplicated rows give equal distances at different indices)."""
    g = np.asarray(origin) + rng.integers(-12, 12, (6000, 3)) * (leaf / 4)
    g = np.vstack([g, g[:500]])                                                        # exact duplicates: ties
    return np.c_[g, rng.uniform(0, 1, len(g))]


def _nearest_check(q, pm, M, max_dist, f32):
    from livox_motion_compensation_sim_b200 import ops
    qq = q.astype(np.float32) if f32 else q
    idx, d2, status = ops.map_nearest(_dev(qq), pm, max_dist)
    wi, wd, wf = org.nearest(qq, M, max_dist)
    assert np.array_equal(idx.cpu().numpy(), wi) and d2.cpu().numpy().tobytes() == wd.tobytes()
    assert int(status.item()) == wf
    return wi, wd


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
@pytest.mark.parametrize("gate", ["leaf", "half"])
def test_map_nearest_vs_oracle(f32, gate):
    rng = np.random.default_rng(20)
    leaf, origin = 0.5, (0.25, -0.5, 0.125)
    mp = _lattice_map(leaf, origin, rng)
    pm, M = _check_map(mp, leaf, origin)
    max_dist = leaf if gate == "leaf" else 0.3
    q = _nearest_queries(leaf, origin, rng)
    wi, wd = _nearest_check(q, pm, M, max_dist, f32)
    assert (wi >= 0).sum() > len(q) // 10 and (wi < 0).sum() > 5
    # ties: a query at a duplicated map row has two candidates at d2 = 0; the smaller original index wins
    dup = mp[:500]
    wi2, wd2 = _nearest_check(dup, pm, M, max_dist, f32)
    first = {}
    for j, row in enumerate(map(tuple, mp[:, :3])):
        first.setdefault(row, j)
    assert (wd2 == 0).all() and np.array_equal(wi2, [first[tuple(r)] for r in dup[:, :3]])


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_map_nearest_gate_edges(f32):
    """d2 exactly r2 is accepted, one ulp beyond is rejected."""
    leaf = 1.0
    mp = np.array([[0.5, 0.5, 0.5, 0.0]])
    pm, M = _check_map(mp, leaf, (0.0, 0.0, 0.0))
    q = np.array([[1.25, 0.5, 0.5, 0.0], [np.nextafter(1.25, 2.0), 0.5, 0.5, 0.0]])      # d2 = r2 exactly, then just above
    from livox_motion_compensation_sim_b200 import ops
    idx, d2, st = ops.map_nearest(_dev(q.astype(np.float32) if f32 else q), pm, 0.75)
    assert idx.cpu().tolist() == ([0, -1] if not f32 else [0, idx.cpu().tolist()[1]])
    if not f32:
        assert d2.cpu().numpy()[0] == 0.75 * 0.75 and np.isinf(d2.cpu().numpy()[1])
    _nearest_check(q, pm, M, 0.75, f32)


@pytest.mark.gpu
def test_map_abi_refusals_and_guard_bands():
    import torch
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    from tests.test_kernel_variants import Guarded
    L = C.lib()
    mp = _cloud(5000, 21, extent=3.0)
    pm = ops.build_point_map(_dev(mp), 0.5, (0.0, 0.0, 0.0))
    M = org.build_map(mp, 0.5, (0.0, 0.0, 0.0))
    q = _cloud(3001, 22, extent=3.5)
    n = len(q)
    qd = _dev(q)
    idx, d2 = Guarded(n, (), torch.int64, -77), Guarded(n, (), torch.float64, -123.0)
    status = torch.zeros(3, dtype=torch.int32, device="cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    m = pm._c()

    def call(p=qd.data_ptr(), nn=n, mm=ctypes.byref(m), md=0.5, i=idx.view.data_ptr(), d=d2.view.data_ptr(), s=status[1:].data_ptr()):
        return L.lmc_map_nearest_f64(p, nn, mm, md, i, d, s, st)
    nan = float("nan")
    for kw in [dict(nn=-1), dict(nn=1 << 31), dict(md=0.0), dict(md=-0.1), dict(md=nan), dict(md=float("inf")), dict(md=0.5000001),
               dict(p=None), dict(i=None), dict(d=None), dict(s=None), dict(mm=None)]:
        assert call(**kw) == C.ERR_INVALID, kw
    assert call(p=qd.data_ptr() + 16) == C.ERR_ALIGN and call(d=d2.view.data_ptr() + 8) == C.ERR_ALIGN
    bad = pm._c()
    bad.leaf[1] = 0.4
    assert call(mm=ctypes.byref(bad)) == C.ERR_INVALID                                   # max_dist > min(leaf)
    bad = pm._c()
    bad.n_voxels = bad.n_points + 1
    assert call(mm=ctypes.byref(bad)) == C.ERR_INVALID
    torch.cuda.synchronize()
    assert idx.untouched_outside(0, 0) and d2.untouched_outside(0, 0) and (status == 0).all().item()
    assert call() == C.OK
    torch.cuda.synchronize()
    assert idx.untouched_outside(0, n) and d2.untouched_outside(0, n) and int(status[0]) == int(status[2]) == 0
    wi, wd, _ = org.nearest(q, M, 0.5)
    assert np.array_equal(idx.view.cpu().numpy(), wi) and d2.view.cpu().numpy().tobytes() == wd.tobytes()
    assert L.lmc_map_workspace_bytes(-1) == C.ERR_INVALID and L.lmc_register_workspace_bytes(-1, 1) == C.ERR_INVALID
    # register refusals write nothing
    F = 2
    off = _dev(np.array([0, 1000, n], np.int64))
    pose_in = _dev(np.tile(np.r_[np.eye(3).reshape(9), 0, 0, 0], (F, 1)))
    pose_out = Guarded(F, (12,), torch.float64, -5.0)
    ints = [Guarded(F, (), torch.int32, -9) for _ in range(3)]
    rms = Guarded(F, (), torch.float64, -5.0)
    ws = torch.empty(L.lmc_register_workspace_bytes(n, F), dtype=torch.uint8, device="cuda:0")

    def reg(nn=n, ff=F, md=0.5, it=30, tt=1e-9, tr=1e-12, w=ws.data_ptr(), po=pose_out.view.data_ptr()):
        return L.lmc_register_frames_f64(qd.data_ptr(), nn, off.data_ptr(), ff, pose_in.data_ptr(), ctypes.byref(m), md, it, tt, tr, w, po,
                                         ints[0].view.data_ptr(), rms.view.data_ptr(), ints[1].view.data_ptr(), ints[2].view.data_ptr(),
                                         status[1:].data_ptr(), st)
    for kw in [dict(it=0), dict(ff=0), dict(md=0.6), dict(md=nan), dict(tt=-1.0), dict(tr=nan), dict(w=None), dict(po=None), dict(nn=-1)]:
        assert reg(**kw) == C.ERR_INVALID, kw
    torch.cuda.synchronize()
    assert pose_out.untouched_outside(0, 0) and rms.untouched_outside(0, 0) and all(g.untouched_outside(0, 0) for g in ints)
    assert reg() == C.OK
    torch.cuda.synchronize()
    assert pose_out.untouched_outside(0, F) and rms.untouched_outside(0, F) and all(g.untouched_outside(0, F) for g in ints)


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_register_frames_vs_oracle(golden, f32):
    import torch
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    env, pts, off, poses = _c3_frames(golden)
    pts = pts.astype(np.float32) if f32 else pts
    init = np.array([_perturb(p, 30 + i) for i, p in enumerate(poses)])
    origin = tuple(poses[0, 9:12])
    pm = ops.build_point_map(_dev(env), 1.0, origin)
    M = org.build_map(env, 1.0, origin)
    # first iteration: the correspondences of the initial pose, exactly
    p1, s1 = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, 1.0, iters=1)
    _, inl1, rms1, _, _ = org.register_frames(pts, off, init, M, 1.0, iters=1)
    assert np.array_equal(s1.inliers.cpu().numpy(), inl1) and np.allclose(s1.rms_m.cpu().numpy(), rms1, rtol=1e-12, atol=0)
    pose, st = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, 1.0)
    want, inl, rms, its, fl = org.register_frames(pts, off, init, M, 1.0)
    ph = pose.cpu().numpy()
    assert np.abs(ph[:, 9:12] - want[:, 9:12]).max() <= 1e-9 and np.abs(ph[:, :9] - want[:, :9]).max() <= 1e-9
    if not f32:                                                             # (f32 rows hold the scan to ~1e-7 m)
        assert np.abs(ph[:, 9:12] - poses[:, 9:12]).max() <= 1e-9
    assert st.converged.all().item() and np.array_equal(st.inliers.cpu().numpy(), inl) and int(st.status.item()) == 0
    print(f"C3 frames {np.diff(off).tolist()}: iterations device {st.iterations.cpu().tolist()} oracle {its.tolist()}")
    # two calls: byte-identical
    pose2, st2 = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, 1.0)
    for a, b in ((pose, pose2), (st.inliers, st2.inliers), (st.rms_m, st2.rms_m), (st.iterations, st2.iterations), (st.flags, st2.flags)):
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()
    # a converged frame's pose stops changing: more iterations give the same bytes
    pose3, st3 = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, 1.0, iters=60)
    assert torch.equal(pose3, pose) and torch.equal(st3.iterations, st.iterations)
    assert (st.flags.cpu().numpy() == C.REG_CONVERGED).all()


@pytest.mark.gpu
def test_register_frame_sizes_and_degenerate():
    """Frames of 0, 5, 255, 256 and 257 points: fewer than 6 inliers is degenerate and keeps the input pose."""
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    rng = np.random.default_rng(40)
    mp = _cloud(40_000, 41, extent=10.0)
    sizes = [0, 5, 255, 256, 257, 3]
    take = [rng.choice(len(mp), s, replace=False) for s in sizes]
    pts = np.vstack([mp[t] for t in take])
    off = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    init = np.array([_perturb(np.r_[np.eye(3).reshape(9), 0, 0, 0], 50 + i, dt=0.01, dr=0.002) for i in range(len(sizes))])
    pm = ops.build_point_map(_dev(mp), 1.0)
    M = org.build_map(mp, 1.0)
    pose, st = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, 1.0)
    want, inl, rms, its, fl = org.register_frames(pts, off, init, M, 1.0)
    flags = st.flags.cpu().numpy()
    assert np.array_equal(flags, fl)
    deg = np.array([0, 1, 5])
    assert (flags[deg] == C.REG_DEGENERATE).all() and pose.cpu().numpy()[deg].tobytes() == init[deg].tobytes()
    assert np.array_equal(st.iterations.cpu().numpy()[deg], [1, 1, 1]) and np.isnan(st.rms_m.cpu().numpy()[0])
    assert np.abs(pose.cpu().numpy() - want).max() <= 1e-9


@pytest.mark.gpu
def test_register_many_chunks():
    """70 000 frames (one chunk each, more than a launch's 65 535 y-limit) plus a frame of 2^17 points."""
    from livox_motion_compensation_sim_b200 import ops
    mp = _cloud(200_000, 60, extent=20.0)
    rng = np.random.default_rng(61)
    F = 70_001
    sizes = np.r_[np.full(F - 1, 8), 1 << 17]
    pts = mp[rng.integers(0, len(mp), int(sizes.sum()))]
    off = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    init = np.tile(np.r_[np.eye(3).reshape(9), 0.01, -0.02, 0.005], (F, 1))
    pm = ops.build_point_map(_dev(mp), 1.0)
    pose, st = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, 1.0)
    M = org.build_map(mp, 1.0)
    sel = np.r_[0, 1, 12345, F - 2, F - 1]
    sub_off = np.r_[0, np.cumsum(sizes[sel])]
    sub = np.vstack([pts[off[f]:off[f + 1]] for f in sel])
    want, inl, _, _, fl = org.register_frames(sub, sub_off, init[sel], M, 1.0)
    assert np.array_equal(st.inliers.cpu().numpy()[sel], inl) and np.array_equal(st.flags.cpu().numpy()[sel], fl)
    assert np.abs(pose.cpu().numpy()[sel] - want).max() <= 1e-9


# ---------------------------------------------------------------------------------------------------- end to end on C3
def _noisy_run(golden, seed=70, **cfg_over):
    from livox_motion_compensation_sim_b200 import LiDARMotionSimulator
    g = golden("scan_C3.npz")
    cfg = json.loads(bytes(g['config_json']).decode())
    rng = np.random.default_rng(seed)
    truth_p, truth_o = g['traj_position_gps'], g['traj_orientation_imu']

    class Source:
        trajectory = {'time': g['traj_time'], 'position': truth_p, 'velocity': np.zeros_like(truth_p), 'orientation': truth_o,
                      'position_gps': truth_p + rng.normal(0, 0.03, truth_p.shape),
                      'orientation_imu': truth_o + rng.normal(0, 0.01, truth_o.shape)}
        environment = g['environment']
    sim = LiDARMotionSimulator(dict(cfg, scan_pose_source='true', **cfg_over))
    np.random.set_state(('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached'])))
    return sim, sim.run_simulation(Source)


# 0.01 rad of heading noise moves a point at 50 m by 0.5 m (plus 3 cm per axis of position noise): a 2 m gate on a 2 m
# leaf takes the right neighbours from the first iteration on every C3 frame
GATE = dict(leaf=2.0, max_dist=2.0)


def _point_error(sim, res, golden):
    """|aligned - env row| of an undistorted run: each frame's rows are the reference scan's (scan_frame_np, which the
    device scanner reproduces) at the true hold-next pose."""
    from scipy.spatial.transform import Rotation
    from livox_motion_compensation_sim_b200 import frames as FR
    g = golden("scan_C3.npz")
    cfg = json.loads(bytes(g['config_json']).decode())
    traj = res['trajectory']
    _, k = sim.lookup_frame_poses(traj, FR.lidar_frame_times(sim.config['duration'], sim.config['lidar_fps']))
    err = []
    for i, a in enumerate(res['aligned_pointclouds']):
        if len(a) == 0:
            continue
        idx, _ = orc.scan_frame_np(g['environment'], traj['position'][k[i]], Rotation.from_euler('xyz', traj['orientation'][k[i]]).as_matrix(), cfg)
        assert len(idx) == len(a)
        err.append(np.linalg.norm(np.asarray(a)[:, :3] - g['environment'][idx, :3], axis=1))
    err = np.concatenate(err)
    return float(err.max()), float(np.sqrt(np.mean(err * err)))


@pytest.mark.gpu
def test_c3_registration_noise_off(golden):
    sim, res = _noisy_run(golden, lidar_range_noise=0.0)
    before = _point_error(sim, res, golden)
    reg = sim.register_scans(res, **GATE)
    after = _point_error(sim, reg, golden)
    r = reg['registration']
    full = np.array([len(s['points_local']) > 0 for s in res['raw_scans']])
    print(f"C3 pose noise, range noise off: before rms {before[1]:.4f} m, after max {after[0]:.3e} m; "
          f"iterations {r['iterations'].min()}..{r['iterations'].max()}, converged {r['converged'].sum()} of {len(full)}")
    assert before[1] >= 0.1 and after[0] <= 1e-6
    assert r['converged'][full].all() and r['position'].shape == (len(full), 3) and r['rotation'].shape == (len(full), 3, 3)
    assert all(a is b for a, b in zip(reg['raw_scans'], res['raw_scans']))
    assert len(sim.voxel_map(reg, 0.5, (0.123456789, 0.234567891, 0.0987654321))['counts']) > 0


@pytest.mark.gpu
def test_c3_registration_range_noise(golden):
    sim, res = _noisy_run(golden)
    after = _point_error(sim, sim.register_scans(res, **GATE), golden)
    print(f"C3 pose noise, range noise 0.02: after rms {after[1]:.4f} m (noise floor 0.0346 m)")
    assert abs(after[1] - 0.0346) <= 0.1 * 0.0346


@pytest.mark.gpu
def test_c3_registration_distorted_hold_next(golden):
    """With motion distortion a frame-rigid pose cannot remove the smear, but registration still lowers the error."""
    sim, res = _noisy_run(golden, motion_distortion=True)
    before, after = sim.alignment_error(res), sim.alignment_error(sim.register_scans(res, **GATE))
    print(f"C3 pose noise, motion distortion, hold_next: rms before {before['rms_m']:.4f} m, after {after['rms_m']:.4f} m")
    assert after['rms_m'] < before['rms_m']


@pytest.mark.gpu
def test_c3_registration_slerp(golden):
    sim, res = _noisy_run(golden, motion_distortion=True, pose_interpolation='slerp')
    before = sim.alignment_error(res)
    after = sim.alignment_error(sim.register_scans(res, **GATE))
    print(f"C3 pose noise, motion distortion, slerp: rms before {before['rms_m']:.4f} m, after {after['rms_m']:.4f} m")
    assert after['rms_m'] < before['rms_m']


@pytest.mark.gpu
def test_c3_scan_pose_source_measured_is_the_reference(golden):
    import hashlib
    import os
    from tests.test_motion_distortion import _c3_run
    from tests.conftest import GOLDEN
    man = json.load(open(os.path.join(GOLDEN, "MANIFEST.json")))['lmc']['C3']
    _, res, _, _, _ = _c3_run(golden, scan_pose_source='measured')
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()       # noqa: E731
    assert sha(np.vstack([s['points_local'] for s in res['raw_scans']])) == man['raw_sha256']
    assert sha(np.vstack(res['aligned_pointclouds'])) == man['aligned_sha256']
