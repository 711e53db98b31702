"""Drop-in check against the reference run C1a, from the golden fixtures the reference produced: the
INTEGRATION.md mix-in -- the reference's generators feeding this package's run_simulation / merge --
reproduces the reference run.

The generators' outputs (noisy trajectory, environment cloud, global NumPy RNG state right before the
frame loop) come from tests/golden/scan_C1a.npz, and the reference's per-frame scan_environment is
replayed by the oracle's scanner, which draws its noise from that RNG exactly as the reference does.
The two device operators used by run_simulation are replaced, for this test only, by the CPU oracle
behind the same signatures; what is verified here is the host-side logic (frame-time grid, hold-next
lookup plumbing, RNG untouched, results contract, merge quirk).  The operators themselves are
verified on the B200 in test_gpu_parity.py.
"""
import contextlib
import hashlib
import io
import json
import os

import numpy as np
import pytest

MAN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "MANIFEST.json")))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture()
def cpu_ops(monkeypatch):
    import torch
    from livox_motion_compensation_sim_b200 import _build, ops
    from oracle import lmc_oracle as orc
    _build.build_library()                                   # the host-side helpers of the C ABI (flatten, result copy)

    def pose_lookup(traj_t, traj_Rt, frame_t):
        idx = orc.C.pose_lookup_hold_next(traj_t.numpy(), frame_t.numpy())
        return torch.from_numpy(traj_Rt.numpy()[idx]), torch.from_numpy(idx)

    def align(pts, frame_off, pose_Rt, *, out=None, export=None, p_range=None, want_out=True):
        return torch.from_numpy(orc.C.align_rigid_f64(pts.numpy(), frame_off.numpy(), pose_Rt.numpy())), None
    monkeypatch.setattr(ops, "pose_lookup_hold_next", pose_lookup)
    monkeypatch.setattr(ops, "align_rigid", align)
    return ops


def test_mixin_reproduces_reference_run(golden, cpu_ops):
    from livox_motion_compensation_sim_b200 import LiDARMotionSimulator as B200Sim
    from oracle import lmc_oracle as orc
    g, want = golden("scan_C1a.npz"), golden("lmc_C1a.npz")
    cfg = dict(json.loads(g['config_json'].tobytes().decode()), **MAN['lmc']['C1a']['config'])
    b200 = B200Sim(dict(cfg, device='cpu'))
    velocity = np.arange(3 * len(g['traj_time']), dtype=np.float64).reshape(-1, 3)     # distinct rows: shows which one a frame got

    class Source:                                            # INTEGRATION.md section 3(b), generators replayed from the fixture
        trajectory = {'time': g['traj_time'], 'position': g['traj_position_gps'], 'velocity': velocity,
                      'orientation': g['traj_orientation_imu'], 'position_gps': g['traj_position_gps'],
                      'orientation_imu': g['traj_orientation_imu']}
        environment = g['environment']
        scan = staticmethod(lambda i, t, pose: orc.scan_frames(Source.environment, pose['position'], pose['orientation'], cfg)[0])
    np.random.set_state(('MT19937', g['rng_keys'], int(g['rng_pos']), int(g['rng_has_gauss']), float(g['rng_cached'])))
    with contextlib.redirect_stdout(io.StringIO()):
        res = b200.run_simulation(Source)
    raw = np.vstack([s['points_local'] for s in res['raw_scans']])
    al = np.vstack(res['aligned_pointclouds'])
    e = MAN['lmc']['C1a']
    assert len(res['raw_scans']) == e['frames'] and len(raw) == e['total_points']
    assert sha(raw) == e['raw_sha256']                       # the seeded scan stream is untouched
    assert sha(al) == e['aligned_sha256']                    # alignment == the reference's
    assert set(res) == {'raw_scans', 'aligned_pointclouds', 'motion_data', 'trajectory', 'environment'}
    assert set(res['raw_scans'][0]) == {'frame_id', 'timestamp', 'points_local', 'sensor_pose'}
    assert set(res['motion_data'][0]) == {'frame_id', 'timestamp', 'gps_lat', 'gps_lon', 'gps_alt', 'imu_roll', 'imu_pitch',
                                          'imu_yaw', 'vel_x', 'vel_y', 'vel_z'}
    # motion rows (LMC:835-847) from the reference's frame times and the pose it used for each frame
    pos, eul, vel = want['pose_position'], want['pose_euler'], velocity[want['pose_idx_all']]
    for i, row in enumerate(res['motion_data']):
        assert row['frame_id'] == i and row['timestamp'] == want['frame_t_all'][i]
        assert row['gps_lat'] == pos[i, 1] / 111320.0 + 40.0
        assert row['gps_lon'] == pos[i, 0] / (111320.0 * np.cos(np.radians(40.0))) - 74.0
        assert (row['gps_alt'], row['imu_roll'], row['imu_pitch'], row['imu_yaw']) == (pos[i, 2], *eul[i])
        assert (row['vel_x'], row['vel_y'], row['vel_z']) == tuple(vel[i])
    # merge quirk (LMC:887-891): C1a has empty frames -> no merged_aligned in strict mode
    with contextlib.redirect_stdout(io.StringIO()):
        m = b200.merge_results(res)
    assert m['merged_aligned'] is None and m['merged_raw'] is not None and len(m['merged_raw']) == e['total_points']
    b200.config['strict_reference_merge'] = False
    with contextlib.redirect_stdout(io.StringIO()):
        m = b200.merge_results(res)
    assert sha(m['merged_aligned']) == e['aligned_sha256']
