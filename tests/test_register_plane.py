"""Map normals and point-to-plane registration (lmc_register.cu k_map_normals / k_reg_accum_plane / k_reg_solve_plane,
ops.estimate_normals, ops.register_frames(normals=...), LiDARMotionSimulator.register_scans(metric='plane')) against the
NumPy oracle (oracle/lmc_oracle_plane.normals / register_frames_plane), which is itself checked against scipy's
cKDTree and numpy.linalg.eigh."""
import ctypes
import json

import numpy as np
import pytest

from oracle import lmc_oracle_plane as orp
from oracle import lmc_oracle_register as org


def _perturb(pose, seed, dt=0.03, dr=0.01):
    """A pose row moved by dt metres and rotated by dr radians about a random axis (left-multiplied)."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    u, v = rng.normal(size=3), rng.normal(size=3)
    out = np.array(pose, np.float64)
    out[:9] = (Rotation.from_rotvec(dr * v / np.linalg.norm(v)).as_matrix() @ out[:9].reshape(3, 3)).reshape(9)
    out[9:12] += dt * u / np.linalg.norm(u)
    return out


def _rows(p):
    return np.c_[p, np.full(len(p), 0.5)]


# ---------------------------------------------------------------------------------------------------- the planar scene
RADIUS, MAX_DIST = 1.0, 1.0          # leaf 1 m; patches are >= 2 RADIUS + MAX_DIST apart, so no ball straddles two


def _patch_frames():
    """(centre, u, v) of every patch: 4 x 4 m squares on a 10 m grid (the nearest points of two patches are >= 4.3 m
    apart): ground, walls facing x and y, and panels tilted about two axes."""
    def span(n):                                                          # two unit vectors across the normal n
        n = np.asarray(n, np.float64) / np.linalg.norm(n)
        u = np.cross(n, [0.0, 0.0, 1.0])
        u /= np.linalg.norm(u)
        return u, np.cross(n, u)
    ex, ey, ez = np.eye(3)
    kinds = {"ground": (ex, ey), "wall_x": (ey, ez), "wall_y": (ex, ez), "tilt_a": span([1.0, -2.0, 3.0]), "tilt_b": span([-3.0, 1.0, 2.0])}
    out = []
    for i, (name, (u, v)) in enumerate(kinds.items()):
        for j in range(4):
            c = np.array([10.0 * j - 15.0, 10.0 * i - 20.0, 0.0 if name == "ground" else 10.0])
            out.append((name, c, u / np.linalg.norm(u), v / np.linalg.norm(v)))
    return out


def _sample(patches, n_per, rng):
    return np.vstack([c + rng.uniform(-2, 2, (n_per, 1)) * u + rng.uniform(-2, 2, (n_per, 1)) * v for _, c, u, v in patches])


def _planar_scene(n_frames=4, map_per=1600, scan_per=400, seed=0, ground_frame=True, center=(0.0, 0.0, 0.0)):
    """(map rows, sensor-frame scan rows, frame_off, true pose table, origin); the last frame sees the ground only."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    patches = _patch_frames()
    ctr = np.asarray(center)
    mp = _rows(_sample(patches, map_per, rng) + ctr)
    srng = np.random.default_rng(seed + 1000)                                 # scan samples independent of the map's
    pts, off, poses = [], [0], []
    for f in range(n_frames):
        only_ground = ground_frame and f == n_frames - 1
        sel = [p for p in patches if p[0] == "ground"] if only_ground else patches
        w = _sample(sel, scan_per, srng) + ctr
        R = Rotation.from_rotvec(srng.normal(0, 0.3, 3)).as_matrix()
        t = ctr + np.array([srng.uniform(-3, 3), srng.uniform(-3, 3), 2.0])
        pts.append(_rows((w - t) @ R))                                        # p = R^T (w - t)
        off.append(off[-1] + len(w))
        poses.append(np.r_[R.reshape(9), t])
    return mp, np.vstack(pts), np.array(off, np.int64), np.array(poses), tuple(ctr + 0.25)


def _rot_err(a, b):
    from scipy.spatial.transform import Rotation
    dR = Rotation.from_matrix(a[:, :9].reshape(-1, 3, 3)) * Rotation.from_matrix(b[:, :9].reshape(-1, 3, 3)).inv()
    return np.linalg.norm(dR.as_rotvec(), axis=1)


# ---------------------------------------------------------------------------------------------------- CPU: the oracle
def _independent_normals(P, radius, min_nb):
    """cKDTree ball + eigh of the same covariance (offsets from the row): (normal with the sign rule, planarity, count)."""
    from scipy.spatial import cKDTree
    T = cKDTree(P)
    out = np.full((len(P), 3), np.nan)
    pl = np.zeros(len(P))
    cnt = np.zeros(len(P), np.int64)
    for i, nb in enumerate(T.query_ball_point(P, radius)):
        cnt[i] = len(nb)
        if len(nb) < min_nb:
            continue
        d = P[nb] - P[i]
        mu = d.mean(0)
        w, V = np.linalg.eigh(d.T @ d / len(nb) - np.outer(mu, mu))
        w = np.maximum(w, 0.0)
        if w[2] == 0.0:
            continue
        n = V[:, 0] / np.linalg.norm(V[:, 0])
        out[i] = n if n[np.argmax(np.abs(n))] > 0 else -n
        pl[i] = (w[1] - w[0]) / w[2]
    return out, pl, cnt


def _check_vs_independent(mp, leaf, origin, radius, min_nb=5, planar_min=0.3):
    M = org.build_map(mp, leaf, origin)
    N, cnt = orp.normals(M, radius, min_nb)
    P = M["pts"][:, :3]
    n_ind, pl_ind, cnt_ind = _independent_normals(P, radius, min_nb)
    assert np.array_equal(cnt, cnt_ind)
    planar = (pl_ind >= planar_min) & np.isfinite(N[:, 0])
    assert planar.sum() > 0
    dot = np.sum(N[planar, :3] * n_ind[planar], 1)
    ang = np.arctan2(np.linalg.norm(np.cross(N[planar, :3], n_ind[planar]), axis=1), dot)   # (arccos loses 1e-8 near 1)
    assert (dot > 0).all()                                                                   # same sign
    assert ang.max() <= 1e-9
    assert (np.abs(N[planar, 3] - pl_ind[planar]) <= 1e-12 * pl_ind[planar]).all()
    assert np.array_equal(np.isnan(N[:, 0]), np.isnan(n_ind[:, 0]))
    return M, N, cnt, planar


def test_oracle_normals_planar_patches():
    mp, _, _, _, origin = _planar_scene(n_frames=1)
    M, N, cnt, planar = _check_vs_independent(mp, 1.0, origin, RADIUS, planar_min=0.0)
    assert planar.all() and N[:, 3].min() >= 0.15                          # (a corner row sees a quarter disc)
    # every row's normal is its patch's
    want = np.vstack([np.repeat(np.cross(u, v)[None], 1600, 0) for _, _, u, v in _patch_frames()])[M["index"]]
    assert np.abs(np.abs(np.sum(N[:, :3] * want, 1)) - 1.0).max() <= 1e-12


@pytest.mark.parametrize("radius", [2.0, 3.0])
def test_oracle_normals_c3(golden, radius):
    g = golden("scan_C3.npz")
    M, N, cnt, planar = _check_vs_independent(g["environment"], radius, tuple(g["traj_position_gps"][0]), radius)
    few = (cnt < 5).mean()
    print(f"C3 at {radius} m: {few:.3f} of rows with < 5 neighbours, {planar.mean():.3f} planar (>= 0.3)")
    assert 0.1 <= few <= 0.5 and planar.sum() > 1000


def test_oracle_normals_utm():
    mp, _, _, _, origin = _planar_scene(n_frames=1, map_per=400, center=(5.0e5, 4.4e6, 50.0))
    _check_vs_independent(mp, 1.0, origin, RADIUS, planar_min=0.0)


def test_oracle_jacobi_edges():
    # already diagonal: no rotation, the eigenvalues are the diagonal's bits
    C = np.array([[[2.0, 0, 0], [0, 0.5, 0], [0, 0, 1e-30]]])
    lam, V = orp.jacobi3(C)
    assert np.array_equal(lam, [[2.0, 0.5, 1e-30]]) and np.array_equal(V[0], np.eye(3))
    # repeated eigenvalues: a rotated diag(1, 1, 0) and diag(1, 0, 0) reach exact zeros off the diagonal
    from scipy.spatial.transform import Rotation
    R = Rotation.from_rotvec([0.3, -0.2, 0.7]).as_matrix()
    for d in ([1.0, 1.0, 0.0], [1.0, 0.0, 0.0], [1.0, 1.0, 1.0]):
        A = (R * d) @ R.T
        lam, V = orp.jacobi3(A[None])
        assert np.allclose(np.sort(lam[0]), np.sort(d), atol=1e-15)
        assert np.allclose(V[0] @ np.diag(lam[0]) @ V[0].T, A, atol=1e-15)


def _normals_of(pts, radius=1.0, min_nb=5, leaf=1.0):
    M = org.build_map(_rows(np.asarray(pts, np.float64)), leaf, (0.0, 0.0, 0.0))
    N, cnt = orp.normals(M, radius, min_nb)
    out, c = np.empty_like(N), np.empty_like(cnt)
    out[M["index"]], c[M["index"]] = N, cnt
    return out, c


def test_oracle_normals_degenerate_neighbourhoods():
    # an axis-aligned plane: no rotation, the normal is exactly e_z
    g = np.array([[x, y, 0.3] for x in np.arange(0.1, 0.9, 0.2) for y in np.arange(0.1, 0.9, 0.2)])
    N, c = _normals_of(g)
    assert (N[:, :3] == [0.0, 0.0, 1.0]).all() and (N[:, 3] > 0.5).all()
    # collinear: planarity 0 (the normal is a unit vector across the line)
    line = np.c_[np.linspace(0.1, 0.9, 7), np.full(7, 0.4), np.full(7, 0.6)]
    N, c = _normals_of(line)
    assert (N[:, 3] == 0.0).all() and np.allclose(np.linalg.norm(N[:, :3], axis=1), 1.0) and (N[:, 0] == 0.0).all()
    # coincident: lambda_max = 0, NaN normal
    N, c = _normals_of(np.tile([[0.5, 0.5, 0.5]], (6, 1)))
    assert np.isnan(N[:, :3]).all() and (N[:, 3] == 0.0).all() and (c == 6).all()
    # exactly min_neighbours - 1 and min_neighbours neighbours
    for k, valid in ((4, False), (5, True)):
        pts = np.c_[0.5 + 0.1 * np.cos(np.arange(k)), 0.5 + 0.1 * np.sin(np.arange(k)), 0.5 + 0.01 * np.arange(k)]
        N, c = _normals_of(pts, min_nb=5)
        assert (c == k).all() and np.isfinite(N[:, 0]).all() == valid and (N[:, 3] > 0).all() == valid


def test_oracle_plane_registration_recovers_planar_scene():
    mp, pts, off, poses, origin = _planar_scene()
    init = np.array([_perturb(p, 10 + i) for i, p in enumerate(poses)])
    M = org.build_map(mp, 1.0, origin)
    N, _ = orp.normals(M, RADIUS)
    pose, inl, rms, its, fl = orp.register_frames_plane(pts, off, init, M, N, MAX_DIST, 0.1)
    pp, _, _, its_p, fl_p = org.register_frames(pts, off, init, M, MAX_DIST)
    e_plane = np.abs(pose[:-1, 9:12] - poses[:-1, 9:12]).max()
    e_point = np.abs(pp[:-1, 9:12] - poses[:-1, 9:12]).max()
    print(f"planar scene: plane {e_plane:.2e} m in {its[:-1].tolist()} iterations, point {e_point:.2e} m in {its_p[:-1].tolist()}")
    assert (fl[:-1] == org.CONVERGED).all() and e_plane <= 1e-6 and _rot_err(pose[:-1], poses[:-1]).max() <= 1e-7
    assert e_point >= 1e-3
    assert fl[-1] == org.DEGENERATE and pose[-1].tobytes() == init[-1].tobytes()


# ---------------------------------------------------------------------------------------------------- GPU
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _device_normals(mp, leaf, origin, radius, min_nb=5):
    from livox_motion_compensation_sim_b200 import ops
    pm = ops.build_point_map(_dev(mp), leaf, origin)
    N, nb = ops.estimate_normals(pm, radius, min_nb)
    N2, nb2 = ops.estimate_normals(pm, radius, min_nb)
    assert N.cpu().numpy().tobytes() == N2.cpu().numpy().tobytes() and torch_equal(nb, nb2)
    M = org.build_map(mp, leaf, origin)
    want, cnt = orp.normals(M, radius, min_nb)
    assert N.cpu().numpy().tobytes() == want.tobytes()
    assert np.array_equal(nb.cpu().numpy(), cnt)
    return pm, M, N, want


def torch_equal(a, b):
    import torch
    return torch.equal(a, b)


def _edge_map():
    """d2 = r2 exactly (included) and one ulp beyond (excluded), duplicates and isolated rows."""
    base = np.array([[0.5, 0.5, 0.5], [1.25, 0.5, 0.5], [0.5, np.nextafter(1.25, 2.0), 0.5]])     # radius 0.75 from row 0
    dup = np.tile([[4.5, 4.5, 4.5]], (7, 1))
    iso = np.array([[10.5, 10.5, 10.5], [20.5, 0.5, 0.5]])
    rng = np.random.default_rng(3)
    ring = np.c_[3.5 + 0.5 * np.cos(np.linspace(0, 6, 9)), 3.5 + 0.5 * np.sin(np.linspace(0, 6, 9)), np.full(9, 3.5)]
    cloud = 7.0 + rng.uniform(-1, 1, (300, 3))
    return _rows(np.vstack([base, ring, dup, iso, cloud]))


NORMAL_CASES = {
    "planar": lambda g: (_planar_scene(n_frames=1)[0], 1.0, _planar_scene(n_frames=1)[4], RADIUS),
    "c3_2m": lambda g: (g("scan_C3.npz")["environment"], 2.0, tuple(g("scan_C3.npz")["traj_position_gps"][0]), 2.0),
    "c3_3m": lambda g: (g("scan_C3.npz")["environment"], 3.0, tuple(g("scan_C3.npz")["traj_position_gps"][0]), 3.0),
    "utm": lambda g: (_planar_scene(n_frames=1, map_per=400, center=(5.0e5, 4.4e6, 50.0))[0], 1.0,
                      _planar_scene(n_frames=1, map_per=400, center=(5.0e5, 4.4e6, 50.0))[4], RADIUS),
    "edges": lambda g: (_edge_map(), 1.0, (0.0, 0.0, 0.0), 0.75),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NORMAL_CASES))
def test_estimate_normals_vs_oracle(golden, name):
    mp, leaf, origin, radius = NORMAL_CASES[name](golden)
    _, M, _, want = _device_normals(mp, leaf, origin, radius)
    if name == "edges":
        cnt = orp.normals(M, radius, 5)[1]
        orig = np.empty_like(cnt)
        orig[M["index"]] = cnt
        assert orig[0] == 2 and orig[1] == 2 and orig[2] == 1                # (0.5 -> 1.25 at r2 in; one ulp beyond out)
        assert (orig[12:19] == 7).all() and (orig[19:21] == 1).all()


@pytest.mark.gpu
def test_estimate_normals_min_neighbours_and_empty():
    from livox_motion_compensation_sim_b200 import ops
    mp = _planar_scene(n_frames=1, map_per=200)[0]
    for k in (3, 40, 200):
        _device_normals(mp, 1.0, (0.25, 0.25, 0.25), 1.0, k)
    pm = ops.build_point_map(_dev(np.zeros((0, 4))), 1.0)
    N, nb = ops.estimate_normals(pm, 1.0)
    assert N.shape == (0, 4) and nb.shape == (0,)


def _plane_check(pts, off, init, mp, origin, f32, min_planarity=0.1):
    from livox_motion_compensation_sim_b200 import ops
    pts = pts.astype(np.float32) if f32 else pts
    pm = ops.build_point_map(_dev(mp), 1.0, origin)
    Nd, _ = ops.estimate_normals(pm, RADIUS)
    M = org.build_map(mp, 1.0, origin)
    N, _ = orp.normals(M, RADIUS)
    _, s1 = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, MAX_DIST, iters=1, normals=Nd, min_planarity=min_planarity)
    _, inl1, rms1, _, _ = orp.register_frames_plane(pts, off, init, M, N, MAX_DIST, min_planarity, iters=1)
    assert np.array_equal(s1.inliers.cpu().numpy(), inl1)
    assert np.allclose(s1.rms_m.cpu().numpy(), rms1, rtol=1e-9, atol=1e-15, equal_nan=True)
    pose, st = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, MAX_DIST, normals=Nd, min_planarity=min_planarity)
    want, inl, rms, its, fl = orp.register_frames_plane(pts, off, init, M, N, MAX_DIST, min_planarity)
    ph = pose.cpu().numpy()
    assert np.array_equal(st.flags.cpu().numpy(), fl) and np.array_equal(st.inliers.cpu().numpy(), inl)
    assert np.abs(ph - want).max() <= 1e-9
    pose2, st2 = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, MAX_DIST, normals=Nd, min_planarity=min_planarity)
    for a, b in ((pose, pose2), (st.inliers, st2.inliers), (st.rms_m, st2.rms_m), (st.iterations, st2.iterations), (st.flags, st2.flags)):
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()
    return pm, Nd, pose, st


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_register_plane_vs_oracle(f32):
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    mp, pts, off, poses, origin = _planar_scene()
    init = np.array([_perturb(p, 30 + i) for i, p in enumerate(poses)])
    pm, Nd, pose, st = _plane_check(pts, off, init, mp, origin, f32)
    ph = pose.cpu().numpy()
    flags = st.flags.cpu().numpy()
    assert (flags[:-1] == C.REG_CONVERGED).all() and flags[-1] == C.REG_DEGENERATE and ph[-1].tobytes() == init[-1].tobytes()
    if not f32:                                                              # (f32 rows hold the scan to ~1e-6 m)
        assert np.abs(ph[:-1, 9:12] - poses[:-1, 9:12]).max() <= 1e-6 and _rot_err(ph[:-1], poses[:-1]).max() <= 1e-7
    # the same frames point-to-point: the sampling bias stays
    pp, sp = ops.register_frames(_dev(pts.astype(np.float32) if f32 else pts), _dev(off), _dev(init), pm, MAX_DIST)
    e_point = np.abs(pp.cpu().numpy()[:-1, 9:12] - poses[:-1, 9:12]).max()
    print(f"planar scene ({'f32' if f32 else 'f64'}): iterations plane {st.iterations.cpu().tolist()} "
          f"point {sp.iterations.cpu().tolist()}; position error plane "
          f"{np.abs(ph[:-1, 9:12] - poses[:-1, 9:12]).max():.2e} m, point {e_point:.2e} m")
    assert e_point >= 1e-3


@pytest.mark.gpu
def test_register_plane_frame_sizes_and_degenerate():
    """Frames of 0, 5, 255, 256 and 257 points: fewer than 6 inliers is degenerate and keeps the input pose."""
    from livox_motion_compensation_sim_b200 import _capi as C
    mp, _, _, _, origin = _planar_scene(n_frames=1)
    rng = np.random.default_rng(40)
    sizes = [0, 5, 255, 256, 257, 3]
    world = [mp[rng.choice(len(mp), s, replace=False)] for s in sizes]
    pts = np.vstack(world)
    off = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    init = np.array([_perturb(np.r_[np.eye(3).reshape(9), 0, 0, 0], 50 + i, dt=0.01, dr=0.002) for i in range(len(sizes))])
    _, _, pose, st = _plane_check(pts, off, init, mp, origin, False)
    deg = np.array([0, 1, 5])
    assert (st.flags.cpu().numpy()[deg] == C.REG_DEGENERATE).all() and pose.cpu().numpy()[deg].tobytes() == init[deg].tobytes()
    assert np.array_equal(st.iterations.cpu().numpy()[deg], [1, 1, 1]) and np.isnan(st.rms_m.cpu().numpy()[0])


@pytest.mark.gpu
def test_register_plane_many_frames():
    """70 001 frames (one chunk each, more than a launch's 65 535 y-limit) plus a frame of 2^17 points."""
    from livox_motion_compensation_sim_b200 import ops
    mp, _, _, _, origin = _planar_scene(n_frames=1)
    rng = np.random.default_rng(61)
    F = 70_001
    sizes = np.r_[np.full(F - 1, 8), 1 << 17]
    pts = mp[rng.integers(0, len(mp), int(sizes.sum()))]
    off = np.r_[0, np.cumsum(sizes)].astype(np.int64)
    init = np.tile(np.r_[np.eye(3).reshape(9), 0.01, -0.02, 0.005], (F, 1))
    pm = ops.build_point_map(_dev(mp), 1.0, origin)
    Nd, _ = ops.estimate_normals(pm, RADIUS)
    pose, st = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, MAX_DIST, normals=Nd)
    M = org.build_map(mp, 1.0, origin)
    N, _ = orp.normals(M, RADIUS)
    sel = np.r_[0, 1, 12345, F - 2, F - 1]
    sub_off = np.r_[0, np.cumsum(sizes[sel])]
    sub = np.vstack([pts[off[f]:off[f + 1]] for f in sel])
    want, inl, _, _, fl = orp.register_frames_plane(sub, sub_off, init[sel], M, N, MAX_DIST, 0.1)
    assert np.array_equal(st.inliers.cpu().numpy()[sel], inl) and np.array_equal(st.flags.cpu().numpy()[sel], fl)
    assert np.abs(pose.cpu().numpy()[sel] - want).max() <= 1e-9


@pytest.mark.gpu
def test_plane_abi_refusals_and_guard_bands():
    import torch
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    from tests.test_kernel_variants import Guarded
    L = C.lib()
    st = torch.cuda.current_stream().cuda_stream
    mp, pts, off_h, poses, origin = _planar_scene(n_frames=3)
    pm = ops.build_point_map(_dev(mp), 1.0, origin)
    m = pm._c()
    Mn = len(mp)
    normals, nb = Guarded(Mn, (4,), torch.float64, -3.0), Guarded(Mn, (), torch.int32, -7)

    def nrm(mm=ctypes.byref(m), r=RADIUS, k=5, o=normals.view.data_ptr(), c=nb.view.data_ptr()):
        return L.lmc_map_normals(mm, r, k, o, c, st)
    nan = float("nan")
    for kw in [dict(r=0.0), dict(r=-1.0), dict(r=nan), dict(r=float("inf")), dict(r=1.0000001), dict(k=2), dict(o=None), dict(mm=None)]:
        assert nrm(**kw) == C.ERR_INVALID, kw
    assert nrm(o=normals.view.data_ptr() + 8) == C.ERR_ALIGN and nrm(c=nb.view.data_ptr() + 4) == C.ERR_ALIGN
    torch.cuda.synchronize()
    assert normals.untouched_outside(0, 0) and nb.untouched_outside(0, 0)
    assert nrm() == C.OK
    torch.cuda.synchronize()
    assert normals.untouched_outside(0, Mn) and nb.untouched_outside(0, Mn)
    want, cnt = orp.normals(org.build_map(mp, 1.0, origin), RADIUS, 5)
    assert normals.view.cpu().numpy().tobytes() == want.tobytes() and np.array_equal(nb.view.cpu().numpy(), cnt)
    only = Guarded(Mn, (4,), torch.float64, -3.0)
    assert L.lmc_map_normals(ctypes.byref(m), RADIUS, 5, only.view.data_ptr(), None, st) == C.OK      # neighbours optional
    torch.cuda.synchronize()
    assert only.untouched_outside(0, Mn) and only.view.cpu().numpy().tobytes() == want.tobytes()

    n, F = len(pts), len(off_h) - 1
    qd, off, pose_in = _dev(pts), _dev(off_h), _dev(poses)
    pose_out = Guarded(F, (12,), torch.float64, -5.0)
    ints = [Guarded(F, (), torch.int32, -9) for _ in range(3)]
    rms = Guarded(F, (), torch.float64, -5.0)
    status = torch.zeros(3, dtype=torch.int32, device="cuda:0")
    assert L.lmc_register_plane_workspace_bytes(-1, 1) == C.ERR_INVALID
    ws = torch.empty(L.lmc_register_plane_workspace_bytes(n, F), dtype=torch.uint8, device="cuda:0")
    assert L.lmc_register_plane_workspace_bytes(n, F) > L.lmc_register_workspace_bytes(n, F)

    def reg(nn=n, ff=F, nv=normals.view.data_ptr(), md=MAX_DIST, mpl=0.1, it=30, tt=1e-9, tr=1e-12, w=ws.data_ptr(), po=pose_out.view.data_ptr()):
        return L.lmc_register_frames_plane_f64(qd.data_ptr(), nn, off.data_ptr(), ff, pose_in.data_ptr(), ctypes.byref(m), nv, md, mpl, it, tt,
                                               tr, w, po, ints[0].view.data_ptr(), rms.view.data_ptr(), ints[1].view.data_ptr(),
                                               ints[2].view.data_ptr(), status[1:].data_ptr(), st)
    for kw in [dict(it=0), dict(ff=0), dict(md=1.1), dict(md=nan), dict(tt=-1.0), dict(tr=nan), dict(w=None), dict(po=None), dict(nn=-1),
               dict(nv=None), dict(mpl=0.0), dict(mpl=-0.1), dict(mpl=1.0000001), dict(mpl=nan)]:
        assert reg(**kw) == C.ERR_INVALID, kw
    assert reg(nv=normals.view.data_ptr() + 8) == C.ERR_ALIGN
    torch.cuda.synchronize()
    assert pose_out.untouched_outside(0, 0) and rms.untouched_outside(0, 0) and all(g.untouched_outside(0, 0) for g in ints)
    assert (status == 0).all().item()
    assert reg(mpl=1.0) == C.OK and reg() == C.OK
    torch.cuda.synchronize()
    assert pose_out.untouched_outside(0, F) and rms.untouched_outside(0, F) and all(g.untouched_outside(0, F) for g in ints)
    assert int(status[0]) == int(status[2]) == 0


@pytest.mark.gpu
def test_register_without_normals_is_point_to_point():
    """register_frames without normals gives the bytes of the point-to-point entry point called directly."""
    import torch
    from livox_motion_compensation_sim_b200 import _capi as C, ops
    mp, pts, off, poses, origin = _planar_scene()
    init = np.array([_perturb(p, 80 + i) for i, p in enumerate(poses)])
    pm = ops.build_point_map(_dev(mp), 1.0, origin)
    pose, st = ops.register_frames(_dev(pts), _dev(off), _dev(init), pm, MAX_DIST)
    L = C.lib()
    n, F = len(pts), len(off) - 1
    ws = torch.empty(L.lmc_register_workspace_bytes(n, F), dtype=torch.uint8, device="cuda:0")
    po = torch.empty((F, 12), dtype=torch.float64, device="cuda:0")
    outs = [torch.empty(F, dtype=torch.int32, device="cuda:0"), torch.empty(F, dtype=torch.float64, device="cuda:0"),
            torch.empty(F, dtype=torch.int32, device="cuda:0"), torch.empty(F, dtype=torch.int32, device="cuda:0")]
    status = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    qd, od, idd, m = _dev(pts), _dev(off), _dev(init), pm._c()
    C.check(L.lmc_register_frames_f64(qd.data_ptr(), n, od.data_ptr(), F, idd.data_ptr(), ctypes.byref(m), MAX_DIST, 30, 1e-9, 1e-12,
                                      ws.data_ptr(), po.data_ptr(), *[o.data_ptr() for o in outs], status.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream))
    for a, b in zip((pose, st.inliers, st.rms_m, st.iterations, st.flags), [po] + outs):
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()


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


GATE = dict(leaf=2.0, max_dist=2.0)


def _point_error(sim, res, golden):
    from scipy.spatial.transform import Rotation
    from oracle import lmc_oracle as orc
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
        err.append(np.linalg.norm(np.asarray(a)[:, :3] - g['environment'][idx, :3], axis=1))
    err = np.concatenate(err)
    return float(err.max()), float(np.sqrt(np.mean(err * err)))


@pytest.mark.gpu
def test_c3_plane_registration_noise_off(golden):
    sim, res = _noisy_run(golden, lidar_range_noise=0.0)
    before = _point_error(sim, res, golden)
    reg_pt = sim.register_scans(res, **GATE)
    reg = sim.register_scans(res, metric='plane', **GATE)
    after = _point_error(sim, reg, golden)
    r, rp = reg['registration'], reg_pt['registration']
    full = np.array([len(s['points_local']) > 0 for s in res['raw_scans']])
    print(f"C3 pose noise, range noise off, plane: before rms {before[1]:.4f} m, after max {after[0]:.3e} m; iterations plane "
          f"{r['iterations'][full].tolist()}, point {rp['iterations'][full].tolist()}")
    assert before[1] >= 0.1 and after[0] <= 1e-6
    assert r['converged'][full].all() and set(r) == set(rp)
    with pytest.raises(ValueError, match="metric"):
        sim.register_scans(res, metric='planes', **GATE)
