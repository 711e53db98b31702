"""
Host-side mirror of the reference's ``LiDARMotionSimulator`` for the motion-compensation hot
path (pose lookup -> per-point transform -> merge -> quantise), B200-native underneath.

Same constructor, config keys, ``ValueError`` messages, ``transform_pointcloud`` operator,
``results`` dict contract and output file names as /root/reference/lidar_motion_compensation.py
(LMC).  What changes is *how* the alignment runs: the reference's per-frame Python loop
(LMC:802-832) becomes ONE batched device call over a frame-major point buffer + CSR offsets.

Out of scope here (SURVEY.md section 2, rows 8-11, 16, 18): the trajectory / environment / scanner
generators and the plots.  ``run_simulation`` therefore takes a ``frame_source`` that supplies the
trajectory and the per-frame raw scans -- in an integration that is the reference's own generator
methods (see INTEGRATION.md for the three-line mix-in).

There is no CPU fallback: a CUDA device and liblmc_b200.so are required.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _trace
from . import _capi as C
from . import frames as FR
from . import ops
from .lvx import frame_layout



class LiDARMotionSimulator:
    # ------------------------------------------------------------------ construction (LMC:275-359)
    def __init__(self, config: Optional[Dict] = None):
        self.config = self.default_config()
        if config:
            self._validate_config(config)
            self.config.update(config)          # unknown keys accepted silently, as in LMC:285
        np.random.seed(self.config['random_seed'])          # LMC:288 (generators upstream rely on it)
        self.device = torch.device(self.config.get('device', 'cuda:0'))
        self._performance_stats = {'scan_times': [], 'transform_times': [], 'total_points_processed': 0}

    def default_config(self):
        """All 22 reference keys with the reference's defaults (LMC:297-330) + B200 knobs."""
        return {
            'duration': 60.0, 'lidar_fps': 10, 'imu_rate': 100, 'gps_rate': 5, 'random_seed': 42,
            'max_speed': 15.0, 'max_angular_vel': 0.5, 'trajectory_type': 'figure_eight',
            'fov_horizontal': 70.0, 'fov_vertical': 77.2, 'range_max': 90.0, 'range_min': 0.05,
            'points_per_frame': 96000, 'angular_resolution': 0.28,
            'gps_noise_std': 0.03, 'imu_accel_noise': 0.1, 'imu_gyro_noise': 0.01, 'lidar_range_noise': 0.02,
            'environment_complexity': 'medium', 'ground_height': 0.0, 'obstacle_density': 0.1,
            # --- additional keys (defaults reproduce the reference's behaviour) ---
            'device': 'cuda:0',
            'io_dtype': 'float64',               # 'float64' = reference-exact layout, 'float32' = throughput layout
            'strict_reference_merge': True,      # LMC:887-891: no merged_aligned if any frame is empty
            'las_scale': (0.01, 0.01, 0.01),     # laspy header default used by LMC:953
            'las_offset': (0.0, 0.0, 0.0),
            # 'hold_next' = the reference's per-frame pose (LMC:802-812); 'slerp' = per-point deskew: every point's
            # timestamp is bracketed in the trajectory samples, orientation SLERPed, position lerped (north_star Mode C)
            'pose_interpolation': 'hold_next',
            # False (default): the device scanner sees every point of a frame from the frame's hold-next pose, as the
            # reference does.  True: a moving sensor -- point j of a frame's m kept points is observed at frame time +
            # j * period / m from the pose interpolated there (Mode C's pose: SLERP + lerp of the trajectory samples), so
            # the raw scans carry the motion distortion the deskews remove; every raw scan dict gains 'point_times' (int64
            # ns) and 'env_index' (its environment rows).  Which points a frame sees is still decided at the hold-next pose,
            # so the point sets and the NumPy noise stream are the reference's.  Needs the device scanner (a frame_source
            # without .scan).
            'motion_distortion': False,
            # 'measured' (default): the device scanner observes from the measured poses (position_gps / orientation_imu),
            # as the reference does, and the alignment uses the same poses, so pose noise never reaches the aligned cloud.
            # 'true': the scanner observes from trajectory['position'] / ['orientation'] (and, with 'motion_distortion',
            # its sample table comes from those too) while alignment and deskew keep the measured poses: the pose noise
            # shows in alignment_error, and register_scans can correct it.  Which points a frame sees is then decided at
            # the true hold-next pose.  Needs the device scanner (a frame_source without .scan).
            'scan_pose_source': 'measured',
            # False (default): results are ordinary NumPy arrays -- D2H into one reusable pinned staging buffer, then a threaded
            # copy (lmc_host_copy); nothing stays page-locked behind the caller's back.
            # True: opt-in throughput knob -- results ARE page-locked blocks of torch's caching host allocator (no second copy:
            # align_frames 42 -> 7 ms on the reference's run shapes), which stay locked as long as any per-frame view of them
            # lives and are cached afterwards (~2 x 2 GB for the reference's default run)
            'pinned_results': False,
        }

    def _validate_config(self, config: Dict) -> None:
        """Same checks and messages as LMC:332-359."""
        for key in ['duration', 'lidar_fps', 'max_speed', 'range_max', 'range_min', 'points_per_frame']:
            if key in config and not isinstance(config[key], (int, float)):
                raise ValueError(f"Configuration '{key}' must be numeric")
        if 'lidar_fps' in config and config['lidar_fps'] <= 0:
            raise ValueError("LiDAR frame rate must be positive")
        if 'duration' in config and config['duration'] <= 0:
            raise ValueError("Simulation duration must be positive")
        if 'max_speed' in config and config['max_speed'] < 0:
            raise ValueError("Maximum speed cannot be negative")
        if 'range_max' in config and 'range_min' in config:
            if config['range_max'] <= config['range_min']:
                raise ValueError("Maximum range must be greater than minimum range")

    # ------------------------------------------------------------------ device helpers
    def _np_dtype(self):
        return np.float64 if self.config.get('io_dtype', 'float64') == 'float64' else np.float32

    def _pinned_stage(self, n: int, np_dtype) -> torch.Tensor:
        tdt = torch.float64 if np_dtype == np.float64 else torch.float32
        st = getattr(self, '_stage', None)
        if st is None or st.dtype != tdt or st.shape[0] < n:
            cap = max(n, 1 << 16)
            self._stage = st = torch.empty((cap, 4), dtype=tdt, pin_memory=self.device.type == 'cuda')
        return st[:n]

    def _to_dev(self, a: np.ndarray, dtype=None) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(a if dtype is None else a.astype(dtype, copy=False)))
        return t.to(self.device, non_blocking=False)

    def _to_host(self, t: torch.Tensor) -> np.ndarray:
        """Device result -> host array the caller owns."""
        if t.device.type != 'cuda' or t.numel() == 0:
            return t.cpu().numpy()
        if self.config.get('pinned_results', False):
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)      # cached block after the first call of a size
            h.copy_(t)
            return h.numpy()                                              # keeps the pinned block alive while referenced
        flat = t.reshape(-1)
        n8 = (flat.numel() * flat.element_size() + 7) // 8
        st = getattr(self, '_stage_out', None)
        if st is None or st.shape[0] < n8:
            self._stage_out = st = torch.empty(max(n8, 1 << 16), dtype=torch.int64, pin_memory=True)
        hb = st.view(torch.uint8)[:flat.numel() * flat.element_size()]
        hb.copy_(flat.view(torch.uint8))
        out = np.empty(tuple(t.shape), dtype=torch.empty(0, dtype=t.dtype).numpy().dtype)
        C.check(C.lib().lmc_host_copy(out.ctypes.data, hb.data_ptr(), out.nbytes, FR._host_threads()))
        return out

    # ------------------------------------------------------------------ (a1) LMC:802-812
    def lookup_frame_poses(self, trajectory: Dict, lidar_times: np.ndarray):
        """Hold-next pose per frame on the device. Returns (pose_Rt device (F,12), pose_idx np int32)."""
        traj_Rt = FR.pose_table(trajectory['position_gps'], trajectory['orientation_imu'])
        pose, idx = ops.pose_lookup_hold_next(self._to_dev(np.asarray(trajectory['time'], np.float64)),
                                              self._to_dev(traj_Rt),
                                              self._to_dev(np.asarray(lidar_times, np.float64)))
        return pose, idx.cpu().numpy()

    # ------------------------------------------------------------------ (a2) LMC:772-776
    def transform_pointcloud(self, points, transformation):
        """Apply transformation to point cloud -- same contract as LMC:772-776: (n,4) f64 in, new
        (n,4) f64 out, input untouched, empty in -> empty out.  Runs as a one-frame device batch."""
        points = np.asarray(points, np.float64)
        n = len(points)
        if n == 0:
            return np.column_stack([np.zeros((0, 3)), np.zeros(0)])
        pose = FR.pose_table(np.asarray(transformation['translation'], np.float64),
                             np.asarray(transformation['rotation'], np.float64))
        off = torch.tensor([0, n], dtype=torch.int64, device=self.device)
        out, _ = ops.align_rigid(self._to_dev(points), off, self._to_dev(pose))
        return out.cpu().numpy()

    # ------------------------------------------------------------------ (N4) LMC:701-770
    @_trace.traced("LiDARMotionSimulator.scan_all")
    def scan_all(self, environment, positions, eulers, keep_device: bool = False, motion=None) -> List[np.ndarray]:
        """scan_environment for every frame in ONE device pass (range / FOV cull, compaction, subsample);
        the noise is drawn on the host from the global NumPy RNG exactly as LMC:767 does, so a seeded
        run reproduces the reference's raw scans.  Returns the per-frame (n_f,4) arrays.
        motion: ops.scan_frames' motion argument (each point observed from the pose at its own time); the point times and
        environment rows are then kept in self.last_scan_motion = (point_times np.int64[N], env_index np.int64[N])."""
        from scipy.spatial.transform import Rotation
        positions = np.asarray(positions, np.float64).reshape(-1, 3)
        Rm = Rotation.from_euler('xyz', np.asarray(eulers, np.float64).reshape(-1, 3)).as_matrix().reshape(-1, 9)   # LMC:726
        c = self.config
        res = ops.scan_frames(self._to_dev(np.asarray(environment, np.float64)), self._to_dev(positions), self._to_dev(Rm),
                              range_max=c['range_max'], range_min=c['range_min'], fov_horizontal=c['fov_horizontal'],
                              fov_vertical=c['fov_vertical'], points_per_frame=c['points_per_frame'],
                              noise_std=c['lidar_range_noise'], motion=motion)
        raw, off = res[0], res[1]
        self.last_scan_motion = (res[2], res[3].cpu().numpy()) if motion is not None else None
        self._dev_scan = (raw, off) if keep_device else None      # run_simulation aligns the device copy directly
        host = self._to_host(raw)
        return [host[off[i]:off[i + 1]] if off[i + 1] > off[i] else np.array([]).reshape(0, 4) for i in range(len(off) - 1)]

    def scan_environment(self, environment, sensor_pose):
        """Same contract as LMC:701-770 for one pose (one-frame device batch)."""
        return self.scan_all(environment, [sensor_pose['position']], [sensor_pose['orientation']])[0]

    # ------------------------------------------------------------------ (a2)+(a3) batched
    @_trace.traced("LiDARMotionSimulator.align_frames")
    def align_frames(self, frames: Sequence[np.ndarray], positions: np.ndarray, eulers: np.ndarray,
                     export: Optional[ops.ExportSpec] = None):
        """The reference's frame loop body LMC:826-832 for every frame at once.

        Returns (merged (N,4) host array, frame_off, ExportBuffers|None).  The merged array is
        frame-major == np.vstack(aligned) (LMC:888); per-frame results are views of it."""
        dt = self._np_dtype()
        off = FR.frame_offsets(frames)
        n = int(off[-1])
        pose = FR.pose_table(positions, eulers)
        if n == 0:
            return np.zeros((0, 4), dt), off, None
        # frames are concatenated straight into a pinned staging buffer that is reused across calls
        # (no page faults on a fresh 100 MB array, and the H2D copy runs at the pinned rate)
        stage = self._pinned_stage(n, dt)
        FR.flatten_frames_into(frames, stage.numpy())
        pts_d = stage.to(self.device, non_blocking=True)
        out, bufs = ops.align_rigid(pts_d, self._to_dev(off), self._to_dev(pose), export=export)
        self._performance_stats['total_points_processed'] += n
        return self._to_host(out), off, bufs

    # ------------------------------------------------------------------ LMC:778-858
    @_trace.traced("LiDARMotionSimulator.run_simulation")
    def run_simulation(self, frame_source=None):
        """Run the simulation with the alignment step on the B200.

        ``frame_source`` supplies what the (out-of-scope) generators produce:
          .trajectory                -> dict with 'time','position','velocity','orientation',
                                        'position_gps','orientation_imu'  (LMC:396-428)
          .scan(i, t, sensor_pose)   -> (n,4) f64 raw sensor-frame points   (LMC:701-770); if absent,
                                        .environment is scanned on the device for all frames at once (N4)
          .environment               -> (M,4) f64 world cloud (needed when .scan is absent)
        With config 'motion_distortion' the device scanner observes every point from the pose at its own time (see
        default_config) and every raw scan dict carries 'point_times' and 'env_index'; alignment_error then measures what
        the alignment leaves of that distortion.
        Returns the reference's results dict (LMC:852-858)."""
        if frame_source is None:
            raise NotImplementedError(
                "trajectory / environment / scanner generators are outside the accelerated hot path "
                "(SURVEY.md section 2 rows 8-11); pass a frame_source, or mix this class into the "
                "reference's LiDARMotionSimulator as shown in INTEGRATION.md")
        distort = bool(self.config.get('motion_distortion', False))
        if distort and hasattr(frame_source, 'scan'):
            raise ValueError("motion_distortion needs the device scanner: a frame_source with its own .scan has no environment "
                             "rows to observe from other poses")
        source = self.config.get('scan_pose_source', 'measured')
        if source not in ('measured', 'true'):
            raise ValueError("scan_pose_source must be 'measured' or 'true'")
        if source == 'true' and hasattr(frame_source, 'scan'):
            raise ValueError("scan_pose_source 'true' needs the device scanner: a frame_source with its own .scan observes "
                             "from the poses it is given")
        scan_keys = ('position', 'orientation') if source == 'true' else ('position_gps', 'orientation_imu')
        trajectory = frame_source.trajectory
        lidar_times = FR.lidar_frame_times(self.config['duration'], self.config['lidar_fps'])
        _, pose_idx = self.lookup_frame_poses(trajectory, lidar_times)

        all_scans, motion_data = [], []
        device_scans = None
        if not hasattr(frame_source, 'scan'):           # no host scanner supplied: scan every frame on the device (N4)
            motion = None
            if distort:                                 # the pose samples the deskews read (_deskew_inputs), one table
                s_ts_d, seg = self._slerp_samples(trajectory, scan_keys)
                motion = (s_ts_d, seg, np.round(np.asarray(lidar_times, np.float64) * 1e9).astype(np.int64),
                          int(round(1e9 / float(self.config['lidar_fps']))))
            device_scans = self.scan_all(frame_source.environment, trajectory[scan_keys[0]][pose_idx],
                                         trajectory[scan_keys[1]][pose_idx], keep_device=True, motion=motion)
        scan_motion = getattr(self, 'last_scan_motion', None) if distort else None
        scan_off = self._dev_scan[1] if scan_motion is not None else None
        for i, t in enumerate(lidar_times):
            k = int(pose_idx[i])
            sensor_pose = {'position': trajectory['position_gps'][k],
                           'orientation': trajectory['orientation_imu'][k],
                           'velocity': trajectory['velocity'][k]}
            scan = device_scans[i] if device_scans is not None else frame_source.scan(i, t, sensor_pose)
            all_scans.append({'frame_id': i, 'timestamp': t, 'points_local': scan, 'sensor_pose': sensor_pose})
            if scan_motion is not None:
                a, b = int(scan_off[i]), int(scan_off[i + 1])
                all_scans[-1]['point_times'], all_scans[-1]['env_index'] = scan_motion[0][a:b], scan_motion[1][a:b]
            motion_data.append(self._motion_row(i, t, sensor_pose))
        dev_scan = getattr(self, '_dev_scan', None) if device_scans is not None else None
        self._dev_scan = None
        if self.config.get('pose_interpolation', 'hold_next') == 'slerp':
            aligned = self.deskew_scans(all_scans, trajectory, _device_raw=dev_scan, _samples=motion[:2] if distort and source == 'measured' else None)
        elif dev_scan is not None and self._np_dtype() == np.float64 and dev_scan[0].shape[0] > 0:
            # the scans are still resident: align them where they are (no flatten, no second upload)
            raw_d, off = dev_scan
            pose = FR.pose_table(trajectory['position_gps'][pose_idx], trajectory['orientation_imu'][pose_idx])
            out, _ = ops.align_rigid(raw_d, self._to_dev(off), self._to_dev(pose))
            self.last_merged, self.last_frame_off, self.last_export = self._to_host(out), off, None
            self._performance_stats['total_points_processed'] += int(off[-1])
            aligned = FR.split_frames(self.last_merged, off)
        else:
            aligned = self.align_scans(all_scans)
        return {'raw_scans': all_scans, 'aligned_pointclouds': aligned, 'motion_data': motion_data,
                'trajectory': trajectory, 'environment': getattr(frame_source, 'environment', None)}

    @staticmethod
    def _motion_row(i, t, sensor_pose):
        """LMC:835-847."""
        p, o, v = sensor_pose['position'], sensor_pose['orientation'], sensor_pose['velocity']
        return {'frame_id': i, 'timestamp': t,
                'gps_lat': p[1] / 111320.0 + 40.0,
                'gps_lon': p[0] / (111320.0 * np.cos(np.radians(40.0))) - 74.0,
                'gps_alt': p[2], 'imu_roll': o[0], 'imu_pitch': o[1], 'imu_yaw': o[2],
                'vel_x': v[0], 'vel_y': v[1], 'vel_z': v[2]}

    @_trace.traced("LiDARMotionSimulator.align_scans")
    def align_scans(self, raw_scans: List[dict], export: Optional[ops.ExportSpec] = None) -> List[np.ndarray]:
        """Batched LMC:826-832 over the reference's raw_scans list; keeps the merged buffer and the
        export buffers on ``self`` (last_merged / last_frame_off / last_export)."""
        frames = [s['points_local'] for s in raw_scans]
        pos = np.array([s['sensor_pose']['position'] for s in raw_scans], np.float64).reshape(-1, 3)
        eul = np.array([s['sensor_pose']['orientation'] for s in raw_scans], np.float64).reshape(-1, 3)
        merged, off, bufs = self.align_frames(frames, pos, eul, export=export)
        self.last_merged, self.last_frame_off, self.last_export = merged, off, bufs
        return FR.split_frames(merged, off)

    def _slerp_samples(self, trajectory: Dict, keys=('position_gps', 'orientation_imu')):
        """The pose samples of Mode C on the device: the trajectory's GPS positions / IMU orientations (or the `keys`
        given) at their own times -> (int64 ns sample times, the (S,22) pose-segment table)."""
        from scipy.spatial.transform import Rotation
        s_ts = np.round(np.asarray(trajectory['time'], np.float64) * 1e9).astype(np.int64)
        quat = Rotation.from_euler('xyz', np.asarray(trajectory[keys[1]], np.float64)).as_quat()
        s_ts_d = self._to_dev(s_ts)
        seg = ops.build_slerp_table(self._to_dev(quat), self._to_dev(np.asarray(trajectory[keys[0]], np.float64)), s_ts_d)
        return s_ts_d, seg

    def _deskew_inputs(self, raw_scans: List[dict], trajectory: Dict, _device_raw=None, _samples=None):
        """The per-point times and the pose-segment table both deskews need: (flat points on the device, frame offsets,
        frame starts, int64 ns point times, sample times, seg) -- None for the device arrays when there are no points."""
        if _device_raw is not None:                                 # scans still resident on the device (run_simulation)
            flat_d, off = _device_raw
        else:
            flat, off = FR.flatten_frames([s['points_local'] for s in raw_scans], np.float64)
            flat_d = None
        n = int(off[-1])
        if n == 0:
            return None, off, None, None, None, None
        if flat_d is None:
            flat_d = self._to_dev(flat)
        period_ns = int(round(1e9 / float(self.config['lidar_fps'])))
        fstart = np.round(np.array([s['timestamp'] for s in raw_scans], np.float64) * 1e9).astype(np.int64)   # same conversion as the sample times below
        ts = np.empty(n, np.int64)
        for i, s in enumerate(raw_scans):
            m = int(off[i + 1] - off[i])
            if m:
                pt = s.get('point_times')
                ts[off[i]:off[i + 1]] = pt if pt is not None else fstart[i] + (np.arange(m, dtype=np.int64) * period_ns) // m
        s_ts_d, seg = self._slerp_samples(trajectory) if _samples is None else _samples
        return flat_d, off, fstart, ts, s_ts_d, seg

    @_trace.traced("LiDARMotionSimulator.deskew_scans")
    def deskew_scans(self, raw_scans: List[dict], trajectory: Dict, export: Optional[ops.ExportSpec] = None,
                     _device_raw=None, _samples=None) -> List[np.ndarray]:
        """Per-point deskew + alignment (north_star Mode C; the reference has no such step -- parity is against the
        builder's SciPy Slerp + lerp oracle).  Pose samples = the trajectory's GPS positions / IMU orientations at
        their own times (LMC:396-428); a point's time is ``scan['point_times']`` (int64 ns) when the scan dict has
        it, else frame time + i * (frame period / n_f) (SURVEY 8d M-C3).  Points outside the sample span hold the
        end pose.  Returns the per-frame world clouds; merged buffer kept as in align_scans."""
        flat_d, off, fstart, ts, s_ts_d, seg = self._deskew_inputs(raw_scans, trajectory, _device_raw, _samples)
        if flat_d is None:
            self.last_merged, self.last_frame_off, self.last_export = np.zeros((0, 4)), off, None
            return FR.split_frames(self.last_merged, off)
        out, bufs = ops.deskew_slerp(flat_d, self._to_dev(ts), self._to_dev(off), self._to_dev(fstart), s_ts_d, seg,
                                     export=export)
        self.last_merged, self.last_frame_off, self.last_export = self._to_host(out), off, bufs
        return FR.split_frames(self.last_merged, off)

    @_trace.traced("LiDARMotionSimulator.deskew_scans_local")
    def deskew_scans_local(self, raw_scans: List[dict], trajectory: Dict, reference='end',
                           export: Optional[ops.ExportSpec] = None) -> List[np.ndarray]:
        """Per-point deskew into the sensor frame of one instant per frame: rotation and translation removed, the
        product scan registration, odometry and LVX recording expect.  Point times and pose samples as deskew_scans.
        reference: 'start' (the frame's start time, the MotionCompensator convention), 'end' (the time of the frame's
        last point; frame start for an empty frame) or an int64 ns array with one entry per frame.  The reference pose
        is Mode C's pose at that time (ops.slerp_pose_at).  Returns the per-frame sensor-frame clouds; the merged buffer
        and the export buffers are kept as in align_scans."""
        bad_ref = ValueError("reference must be 'start', 'end' or an int64 ns array with one entry per frame")
        if isinstance(reference, str) and reference not in ('start', 'end'):
            raise bad_ref
        flat_d, off, fstart, ts, s_ts_d, seg = self._deskew_inputs(raw_scans, trajectory)
        if flat_d is None:
            self.last_merged, self.last_frame_off, self.last_export = np.zeros((0, 4)), off, None
            return FR.split_frames(self.last_merged, off)
        if isinstance(reference, str):
            if reference == 'start':
                ref_ts = fstart
            else:
                ref_ts = fstart.copy()
                full = np.flatnonzero(np.diff(off) > 0)
                ref_ts[full] = ts[off[full + 1] - 1]
        else:
            ref_ts = np.asarray(reference)
            if ref_ts.shape != (len(raw_scans),) or not np.issubdtype(ref_ts.dtype, np.integer):
                raise bad_ref
            ref_ts = ref_ts.astype(np.int64)
        ref_pose = ops.slerp_pose_at(s_ts_d, seg, self._to_dev(ref_ts))
        self.last_ref_pose = ref_pose
        out, bufs = ops.deskew_slerp_local(flat_d, self._to_dev(ts), self._to_dev(off), self._to_dev(fstart), s_ts_d, seg, ref_pose,
                                           export=export)
        self.last_merged, self.last_frame_off, self.last_export = self._to_host(out), off, bufs
        return FR.split_frames(self.last_merged, off)

    def alignment_error(self, results) -> Dict:
        """How far the aligned clouds of a run are from the environment points they observed: |aligned_i - env[env_index_i]|
        (Euclidean, metres) over every point, on the device.  Needs a run with 'motion_distortion' (the raw scans carry
        'env_index').  Returns {'max_m', 'rms_m', 'per_frame_max_m'} (per-frame list; 0.0 for an empty frame)."""
        scans = results['raw_scans']
        if not scans or any(s.get('env_index') is None for s in scans):
            raise ValueError("alignment_error needs the environment rows of the raw points: run with 'motion_distortion': True")
        aligned = results['aligned_pointclouds']
        off = FR.frame_offsets(aligned)
        if not np.array_equal(off, FR.frame_offsets([s['env_index'] for s in scans])):
            raise ValueError("aligned clouds and raw scans differ in their point counts")
        n = int(off[-1])
        if n == 0:
            return {'max_m': 0.0, 'rms_m': 0.0, 'per_frame_max_m': [0.0] * len(scans)}
        flat, _ = FR.flatten_frames([np.asarray(a).reshape(-1, 4) for a in aligned], np.float64)
        idx = self._to_dev(np.concatenate([np.asarray(s['env_index'], np.int64) for s in scans]))
        env = self._to_dev(np.asarray(results['environment'], np.float64))
        err = torch.linalg.vector_norm(self._to_dev(flat)[:, :3] - env[idx, :3], dim=1)
        fidx = self._to_dev(np.repeat(np.arange(len(scans)), np.diff(off)))
        per = torch.zeros(len(scans), dtype=torch.float64, device=self.device).scatter_reduce(0, fidx, err, 'amax')
        return {'max_m': float(err.max().item()), 'rms_m': float(torch.sqrt(torch.mean(err * err)).item()),
                'per_frame_max_m': per.cpu().numpy().tolist()}

    def voxel_map(self, results, leaf, origin=(0.0, 0.0, 0.0)) -> Dict[str, np.ndarray]:
        """Voxel-grid map of the run's aligned cloud (the merged buffer, frame-major), built on the device by
        ops.voxel_downsample: the centroid and point count of every voxel of edge `leaf` (one value or three) on the grid
        anchored at `origin`, voxels in the order the run first reaches them.  A sharper alignment fills fewer voxels.
        Keys are limited to 2^20 cells from the origin on each axis and the arithmetic is f64, so a UTM-scale cloud needs
        an origin near the data (e.g. the first pose).  Returns {'points': (V,4) host array in the run's layout,
        'counts': int32[V]}.  ValueError for a NaN / inf point, OverflowError for a point beyond the key range or an
        |intensity| >= 256, as ExportBuffers.raise_for_flags."""
        aligned = results['aligned_pointclouds']
        base = getattr(self, 'last_merged', None)
        if base is not None and len(aligned) and aligned[0].base is base:
            pts = base
        else:
            pts = np.vstack([np.asarray(a).reshape(-1, 4) for a in aligned]) if len(aligned) else np.zeros((0, 4), self._np_dtype())
        cent, counts, _, status = ops.voxel_downsample(self._to_dev(pts), leaf, origin)
        ops.ExportBuffers(status=status).raise_for_flags()
        return {'points': self._to_host(cent), 'counts': counts.cpu().numpy()}

    def register_scans(self, results, leaf=1.0, max_dist=1.0, iters=30, map_points=None, origin=None, metric='point',
                       normal_radius=None, min_planarity=ops.MIN_PLANARITY) -> Dict:
        """Refine every frame's pose against a prior point map on the device (ops.build_point_map + ops.register_frames:
        exact nearest neighbours within max_dist, Gauss-Newton) and re-align the run with the refined poses.  metric
        'point' minimises point-to-point distances; 'plane' estimates the map's normals within normal_radius (default
        min(leaf); ops.estimate_normals) and minimises the distances along them, pairing only map rows with planarity >=
        min_planarity.
        The map defaults to results['environment'] (the prior map) on a grid of edge `leaf` anchored at `origin` (default:
        the first frame's pose, so UTM-scale maps keep their keys in range); max_dist <= leaf.  A 'hold_next' run
        registers its raw scans from their hold-next measured poses; a 'slerp' run registers deskew_scans_local(reference=
        'end') from the Mode C poses at the frames' last point times.  Returns a new results dict: the raw scans untouched,
        'aligned_pointclouds' = ops.align_rigid of those clouds with the refined poses, and 'registration': {'position'
        (F,3), 'rotation' (F,3,3), 'inliers', 'rms_m', 'iterations', 'converged', 'degenerate'} (per frame; a frame with
        fewer than 6 inliers is degenerate and keeps its pose).  alignment_error and voxel_map work on it unchanged."""
        if metric not in ('point', 'plane'):
            raise ValueError("metric must be 'point' or 'plane'")
        scans = results['raw_scans']
        env = results.get('environment') if map_points is None else map_points
        if env is None:
            raise ValueError("register_scans needs a map: pass map_points, or a run whose results carry 'environment'")
        if self.config.get('pose_interpolation', 'hold_next') == 'slerp':
            local = self.deskew_scans_local(scans, results['trajectory'], reference='end')
            off = FR.frame_offsets(local)
            flat = self.last_merged
            pose0 = self.last_ref_pose if int(off[-1]) else self._to_dev(np.zeros((len(scans), 12)))
        else:
            flat, off = FR.flatten_frames([s['points_local'] for s in scans], np.float64)
            pose0 = self._to_dev(FR.pose_table(np.array([s['sensor_pose']['position'] for s in scans], np.float64).reshape(-1, 3),
                                               np.array([s['sensor_pose']['orientation'] for s in scans], np.float64).reshape(-1, 3)))
        if origin is None:
            origin = tuple(float(v) for v in scans[0]['sensor_pose']['position']) if scans else (0.0, 0.0, 0.0)
        pmap = ops.build_point_map(self._to_dev(np.asarray(env, np.float64).reshape(-1, 4)), leaf, origin)
        pts_d = self._to_dev(np.asarray(flat, np.float64).reshape(-1, 4))
        off_d = self._to_dev(off)
        if metric == 'plane':
            radius = min(pmap.leaf) if normal_radius is None else normal_radius
            normals, _ = ops.estimate_normals(pmap, radius)
            pose, st = ops.register_frames(pts_d, off_d, pose0, pmap, max_dist, iters=iters, normals=normals, min_planarity=min_planarity)
        else:
            pose, st = ops.register_frames(pts_d, off_d, pose0, pmap, max_dist, iters=iters)
        ops.ExportBuffers(status=st.status).raise_for_flags()
        if int(off[-1]):
            out, _ = ops.align_rigid(pts_d if self._np_dtype() == np.float64 else pts_d.float(), off_d, pose)
            self.last_merged, self.last_frame_off, self.last_export = self._to_host(out), off, None
        else:
            self.last_merged, self.last_frame_off, self.last_export = np.zeros((0, 4), self._np_dtype()), off, None
        ph = pose.cpu().numpy()
        reg = {'position': ph[:, 9:12].copy(), 'rotation': ph[:, :9].reshape(-1, 3, 3).copy(),
               'inliers': st.inliers.cpu().numpy(), 'rms_m': st.rms_m.cpu().numpy(), 'iterations': st.iterations.cpu().numpy(),
               'converged': st.converged.cpu().numpy(), 'degenerate': st.degenerate.cpu().numpy()}
        return dict(results, aligned_pointclouds=FR.split_frames(self.last_merged, off), registration=reg)

    # ------------------------------------------------------------------ (a3) LMC:886-899
    def _merge_flags(self, results):
        """The reference's two merge guards (LMC:887-899) with its warnings: (merged_aligned exists, merged_raw exists)."""
        aligned = results['aligned_pointclouds']
        strict = self.config.get('strict_reference_merge', True)
        has_aligned = bool(aligned) and (all(len(pc) > 0 for pc in aligned) or not strict)
        if not has_aligned:
            print("Warning: No aligned point clouds to merge")
        has_raw = any(len(s['points_local']) > 0 for s in results['raw_scans'])
        if not has_raw:
            print("Warning: No raw point clouds to merge")
        return has_aligned, has_raw

    def merge_results(self, results) -> Dict[str, Optional[np.ndarray]]:
        """merged_aligned / merged_raw with the reference's guards."""
        aligned = results['aligned_pointclouds']
        out: Dict[str, Optional[np.ndarray]] = {'merged_aligned': None, 'merged_raw': None}
        has_aligned, has_raw = self._merge_flags(results)
        if has_aligned:
            base = getattr(self, 'last_merged', None)
            same = base is not None and len(aligned) and aligned[0].base is base
            out['merged_aligned'] = base if same else np.vstack(aligned)
        if has_raw:
            out['merged_raw'] = np.vstack([s['points_local'] for s in results['raw_scans'] if len(s['points_local']) > 0])
        return out

    # ------------------------------------------------------------------ (a4) LMC:252-272 / 965-990
    def quantize_lvx(self, results) -> tuple:
        """int32-millimetre LVX type-2 records of the RAW scans (LMC:973-978), on the device.
        Returns ((N,14) uint8 host array, frame_off)."""
        flat, off = FR.flatten_frames([s['points_local'] for s in results['raw_scans']], np.float64)
        if len(flat) == 0:
            return np.zeros((0, 14), np.uint8), off
        bufs = ops.quantize(self._to_dev(flat), ops.ExportSpec(lvx=True, lvx_mode=C.LVX_TYPE2_OF_INPUT))
        bufs.raise_for_flags()
        return self._to_host(bufs.lvx14), off

    # ------------------------------------------------------------------ (a5) LMC:950-963
    def quantize_las(self, points: np.ndarray):
        """LAS integer X/Y/Z + uint16 intensity of the merged cloud (parity unpinned: laspy)."""
        bufs = ops.quantize(self._to_dev(np.asarray(points, np.float64)),
                            ops.ExportSpec(las=True, las_scale=self.config['las_scale'],
                                           las_offset=self.config['las_offset'],
                                           las_intensity_mode=C.LAS_INTENSITY_UNIT))
        bufs.raise_for_flags()
        return (bufs.las_x.cpu().numpy(), bufs.las_y.cpu().numpy(), bufs.las_z.cpu().numpy(),
                bufs.las_intensity.cpu().numpy())

    # ------------------------------------------------------------------ LMC:860-930 (hot-path outputs)
    @_trace.traced("LiDARMotionSimulator.save_results")
    def save_results(self, results, output_dir='lidar_simulation_output'):
        """Writes the reference's hot-path outputs under the reference's names:
        aligned_scans_pcd/aligned_frame_%04d.pcd, raw_scans_pcd/frame_%04d.pcd, merged_aligned.pcd,
        merged_raw_overlapped.pcd, merged_aligned.las, lidar_data.lvx -- plus the two small tables
        motion_data.csv / trajectory.csv (LMC:866-868, 916-927; plain pandas, as in the reference)."""
        os.makedirs(output_dir, exist_ok=True)
        print(f"Saving results to {output_dir}...")
        import pandas as pd
        if results.get('motion_data') is not None:
            pd.DataFrame(results['motion_data']).to_csv(os.path.join(output_dir, 'motion_data.csv'), index=False)
        # LMC:870-899: every per-frame PCD and the two merged PCDs.  One formatting pass per cloud family: the text
        # of the frame-major buffer IS the merged file's body, and each per-frame body is a slice of it
        has_aligned, has_raw = self._merge_flags(results)
        pcd_dir = os.path.join(output_dir, 'raw_scans_pcd'); os.makedirs(pcd_dir, exist_ok=True)
        self.save_pcd_frames([scan['points_local'] for scan in results['raw_scans']],
                             [os.path.join(pcd_dir, f'frame_{scan["frame_id"]:04d}.pcd') for scan in results['raw_scans']],
                             os.path.join(output_dir, 'merged_raw_overlapped.pcd') if has_raw else None)
        aligned_dir = os.path.join(output_dir, 'aligned_scans_pcd'); os.makedirs(aligned_dir, exist_ok=True)
        aligned = results['aligned_pointclouds']
        aligned_d = self.save_pcd_frames(aligned, [os.path.join(aligned_dir, f'aligned_frame_{i:04d}.pcd') for i in range(len(aligned))],
                                         os.path.join(output_dir, 'merged_aligned.pcd') if has_aligned else None)
        try:
            if not has_aligned:
                raise UnboundLocalError("merged_aligned")           # what LMC:903 hits when the merge was skipped
            self.save_las(np.zeros((0, 4)) if aligned_d is None else None, os.path.join(output_dir, 'merged_aligned.las'),
                          _device_pts=aligned_d)                                    # the aligned cloud is still resident
            print("LAS format saved successfully")
        except Exception as e:                                       # LMC:905-906 swallows and prints
            print(f"Could not save LAS format: {e}")
        del aligned_d
        try:
            self.save_lvx(results, os.path.join(output_dir, 'lidar_data'))
            print("LVX formats saved successfully")
        except Exception as e:                                       # LMC:913-914
            print(f"Could not save LVX formats: {e}")
        traj = results.get('trajectory')
        if traj is not None and all(k in traj for k in ('time', 'position', 'position_gps')):
            pd.DataFrame({'time': traj['time'], 'x': traj['position'][:, 0], 'y': traj['position'][:, 1], 'z': traj['position'][:, 2],
                          'x_gps': traj['position_gps'][:, 0], 'y_gps': traj['position_gps'][:, 1],
                          'z_gps': traj['position_gps'][:, 2]}).to_csv(os.path.join(output_dir, 'trajectory.csv'), index=False)
        print("Results saved successfully!")
        return output_dir

    @staticmethod
    def _pcd_header(n: int) -> bytes:
        """LMC:934-945."""
        return ("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z intensity\n"
                "SIZE 4 4 4 4\nTYPE F F F F\nCOUNT 1 1 1 1\n"
                f"WIDTH {n}\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS {n}\nDATA ascii\n").encode('ascii')

    def save_pcd(self, points, filename):
        """ASCII PCD, byte-identical to LMC:932-948 ('%.6f' per field); the point lines are formatted on the GPU."""
        points = np.asarray(points, np.float64).reshape(-1, 4)
        n = len(points)
        with open(filename, 'wb') as f:
            f.write(self._pcd_header(n))
            if n:
                body, status = ops.pcd_ascii_body(self._to_dev(points))       # (N2) '%.6f' formatting on the device
                if int(status.item()):
                    raise OverflowError("save_pcd: |value| >= 9.2e12 is outside the device formatter's range")
                f.write(body.cpu().numpy().tobytes())

    @_trace.traced("LiDARMotionSimulator.save_pcd_frames")
    def save_pcd_frames(self, frames: Sequence[np.ndarray], filenames: Sequence[str], merged_filename: Optional[str] = None):
        """save_pcd for a whole list of frames (LMC:870-884) plus their np.vstack (LMC:893-899) with ONE upload and
        ONE formatting pass: the frame-major buffer is formatted once, frame f's file body is the byte range between
        the offsets of its first and one-past-last row (``lmc_pcd_ascii_row_offsets``), the merged file's body is the
        whole text.  Every file is byte-identical to what save_pcd writes.  Returns the device copy of the
        frame-major (N,4) f64 buffer (None when there are no points)."""
        if len(frames) != len(filenames):
            raise ValueError("one filename per frame")
        off = FR.frame_offsets(frames)
        n = int(off[-1])
        pts_d = None
        if n:
            stage = self._pinned_stage(n, np.float64)
            FR.flatten_frames_into(frames, stage.numpy())
            pts_d = stage.to(self.device, non_blocking=True)
            text_d, boff_d, status = ops.pcd_ascii_frames(pts_d, self._to_dev(off))   # (syncs: the staging buffer is free again)
            if int(status.item()):
                raise OverflowError("save_pcd: |value| >= 9.2e12 is outside the device formatter's range")
            text = memoryview(self._to_host(text_d))
            boff = boff_d.cpu().numpy()
        for i, fn in enumerate(filenames):
            m = int(off[i + 1] - off[i])
            with open(fn, 'wb') as f:
                f.write(self._pcd_header(m))
                if m:
                    f.write(text[int(boff[i]):int(boff[i + 1])])
        if merged_filename is not None:
            with open(merged_filename, 'wb') as f:
                f.write(self._pcd_header(n))
                if n:
                    f.write(text)
        return pts_d

    @_trace.traced("LiDARMotionSimulator.save_las")
    def save_las(self, points, filename, _device_pts: Optional[torch.Tensor] = None):
        """merged_aligned.las (LMC:950-963): LAS 1.2 / point format 3 with the laspy header defaults the
        reference relies on (scale 0.01, offset 0; config 'las_scale' / 'las_offset'), intensity scaled to
        16 bits.  The whole file image -- header extremes included -- is built on the device.  Parity
        with laspy's bytes is unpinned (laspy is not available); the file follows the LAS 1.2 spec."""
        import datetime
        today = datetime.date.today()
        pts_d = _device_pts if _device_pts is not None else self._to_dev(np.asarray(points, np.float64))
        data, status = ops.build_las_pf3(pts_d, scale=self.config['las_scale'],
                                         offset=self.config['las_offset'], intensity_mode=C.LAS_INTENSITY_UNIT,
                                         year=today.year, day_of_year=today.timetuple().tm_yday)
        ops.ExportBuffers(status=status).raise_for_flags()
        with open(filename, 'wb') as f:
            f.write(memoryview(self._to_host(data)))

    @_trace.traced("LiDARMotionSimulator.save_lvx")
    def save_lvx(self, results, base_filename):
        """lidar_data.lvx with the LVX v1.1 container of LMC:58-250 around device-quantised records."""
        data = self.build_lvx_bytes(results)
        with open(f"{base_filename}.lvx", 'wb') as f:
            f.write(data.tobytes())
        return True

    def build_lvx_bytes(self, results) -> np.ndarray:
        """The whole LVX v1.1 file image (LMC:58-250), quantised and laid out on the device."""
        scans = results['raw_scans']
        if not scans:
            raise ValueError("No frame data provided")                      # LMC:75-76
        flat, off = FR.flatten_frames([s['points_local'] for s in scans], np.float64)
        ts = np.array([s['timestamp'] for s in scans], np.float64)
        ids = np.array([s['frame_id'] for s in scans], np.int64)
        _, fpos = frame_layout(off)
        data, status = ops.build_lvx_v11(self._to_dev(flat), self._to_dev(off), self._to_dev(fpos), self._to_dev(ts),
                                         self._to_dev(ids), int(np.diff(off).max()), size=int(fpos[-1]))
        bufs = ops.ExportBuffers(status=status)
        bufs.raise_for_flags()
        return self._to_host(data)
