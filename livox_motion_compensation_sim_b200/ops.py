"""Device operators: torch CUDA tensors in, hand-written sm_100a kernels through the C ABI
(include/lmc_b200.h), torch tensors out.  torch is only the allocator / stream provider.

No fallback: inputs must be CUDA tensors and liblmc_b200.so must load, otherwise these raise."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import torch

from . import _capi as C
from . import _trace


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream          # the CURRENT device's stream: ops run inside _on_tensor_device


def _on_tensor_device(fn):
    """Run the operator on the device its tensors live on, whatever the caller's current device is: the C ABI
    launches on the calling thread's current device and stream, so the guard switches to the tensors' GPU (and
    its current stream) for the duration of the call and refuses arguments spread over several devices."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        def visit(v):
            nonlocal dev
            if isinstance(v, torch.Tensor) and v.is_cuda:
                if dev is None:
                    dev = v.device
                elif v.device != dev:
                    raise ValueError(f"{fn.__name__}: tensors on different devices ({dev} and {v.device})")
            elif isinstance(v, (ExportSpec, ExportBuffers)):
                for x in vars(v).values():
                    visit(x)
        for v in args:
            visit(v)
        for v in kwargs.values():
            visit(v)
        if dev is None:
            return fn(*args, **kwargs)                      # no CUDA tensor: the operator's own checks raise
        with torch.cuda.device(dev), _trace.span("lmc." + fn.__name__):
            return fn(*args, **kwargs)
    return wrapper


def _req(t: Optional[torch.Tensor], dtype, name: str, shape_tail=None) -> int:
    if t is None:
        return 0
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name}: expected a CUDA tensor (this path has no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")
    if shape_tail is not None and tuple(t.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"{name}: expected shape (n,{','.join(map(str, shape_tail))}), got {tuple(t.shape)}")
    return t.data_ptr()


@dataclass
class ExportBuffers:
    """Integer-quantised export buffers produced by the fused epilogues."""
    lvx14: Optional[torch.Tensor] = None          # (N,14) uint8   <iiiBB records
    las_x: Optional[torch.Tensor] = None          # (N) int32
    las_y: Optional[torch.Tensor] = None
    las_z: Optional[torch.Tensor] = None
    las_intensity: Optional[torch.Tensor] = None  # (N) uint16
    status: Optional[torch.Tensor] = None         # (1) int32 bitmask of C.FLAG_*

    def flags(self) -> int:
        return 0 if self.status is None else int(self.status.item())

    def raise_for_flags(self) -> None:
        """Mirror the reference's failure modes: int(nan) -> ValueError (LMC:257),
        struct.pack / laspy overflow -> OverflowError."""
        f = self.flags()
        if f & C.FLAG_NAN:
            raise ValueError("cannot convert float NaN to integer")
        if f & C.FLAG_OVERFLOW:
            raise OverflowError("quantised value out of range for the export format")


@dataclass
class ExportSpec:
    lvx: bool = False
    lvx_mode: int = C.LVX_TYPE2_OF_INPUT
    tag: Optional[torch.Tensor] = None
    las: bool = False
    las_scale: Sequence[float] = (0.01, 0.01, 0.01)      # laspy header default (LMC:953)
    las_offset: Sequence[float] = (0.0, 0.0, 0.0)
    las_intensity_mode: int = C.LAS_INTENSITY_UNIT
    into: Optional[ExportBuffers] = None                 # reuse caller buffers (merged cloud shards)
    peer_out: Sequence[int] = ()                         # peer-mapped device pointers of the other ranks' `out` copies
    peer_lvx14: Sequence[int] = ()                       # ... and of their lvx14 copies (fused merged-cloud assembly)
    mc_out: int = 0                                      # NVSwitch multicast address of `out` (0 = per-peer stores)
    mc_lvx14: int = 0                                    # ... and of lvx14; both or neither


def _make_export(spec: Optional[ExportSpec], n: int, device):
    if spec is None or not (spec.lvx or spec.las or spec.peer_out):
        return None, None
    b = spec.into if spec.into is not None else ExportBuffers()
    if spec.lvx and b.lvx14 is None:
        b.lvx14 = torch.empty((n, 14), dtype=torch.uint8, device=device)
    if spec.las and b.las_x is None:
        b.las_x = torch.empty(n, dtype=torch.int32, device=device)
        b.las_y = torch.empty(n, dtype=torch.int32, device=device)
        b.las_z = torch.empty(n, dtype=torch.int32, device=device)
        b.las_intensity = torch.empty(n, dtype=torch.uint16, device=device)
    if b.status is None:
        b.status = torch.zeros(1, dtype=torch.int32, device=device)
    ex = C.LmcExport()
    ex.lvx14 = _req(b.lvx14, torch.uint8, "lvx14", (14,)) if spec.lvx else 0
    ex.lvx_mode = int(spec.lvx_mode)
    ex.tag = _req(spec.tag, torch.uint8, "tag")
    if spec.las:
        ex.las_x = _req(b.las_x, torch.int32, "las_x")
        ex.las_y = _req(b.las_y, torch.int32, "las_y")
        ex.las_z = _req(b.las_z, torch.int32, "las_z")
        ex.las_intensity = _req(b.las_intensity, torch.uint16, "las_intensity")
    ex.las_intensity_mode = int(spec.las_intensity_mode)
    for c in range(3):
        ex.las_scale[c] = float(spec.las_scale[c])
        ex.las_offset[c] = float(spec.las_offset[c])
    ex.status = b.status.data_ptr()
    npeer = max(len(spec.peer_out), len(spec.peer_lvx14))
    if npeer > C.MAX_PEERS:
        raise ValueError(f"at most {C.MAX_PEERS} peers")
    ex.n_peers = npeer
    for r in range(npeer):
        ex.peer_out[r] = int(spec.peer_out[r]) if r < len(spec.peer_out) else None
        ex.peer_lvx14[r] = int(spec.peer_lvx14[r]) if (spec.lvx and r < len(spec.peer_lvx14)) else None
    ex.mc_out = int(spec.mc_out) or None
    ex.mc_lvx14 = int(spec.mc_lvx14) or None
    return ex, b


def _layout(pts: torch.Tensor):
    if pts.dtype == torch.float64:
        return True
    if pts.dtype == torch.float32:
        return False
    raise TypeError(f"points must be float64 (parity layout) or float32 (throughput layout), got {pts.dtype}")


def _range(n, p_range):
    if p_range is None:
        return 0, n
    return int(p_range[0]), int(p_range[1])


@_on_tensor_device
def pose_lookup_hold_next(traj_t: torch.Tensor, traj_Rt: torch.Tensor, frame_t: torch.Tensor):
    """(a1) LMC:802-812 on the device. Returns (pose_Rt (F,12) f64, pose_idx (F) int32)."""
    F = frame_t.shape[0]
    pose = torch.empty((F, 12), dtype=torch.float64, device=frame_t.device)
    idx = torch.empty(F, dtype=torch.int32, device=frame_t.device)
    C.check(C.lib().lmc_pose_lookup_hold_next(
        _req(traj_t, torch.float64, "traj_t"), traj_t.shape[0], _req(traj_Rt, torch.float64, "traj_Rt", (12,)),
        _req(frame_t, torch.float64, "frame_t"), F, pose.data_ptr(), idx.data_ptr(), _stream_ptr()))
    return pose, idx


def _point_op(name, pts, frame_off, args, out, export, p_range, want_out, per_frame=None):
    """The body of the aligned-cloud operators: lmc_<name>_f64 / _f32 (pts, *args(f64), out, n_points, n_frames, p_begin,
    p_end, ex, stream), with out and the export buffers allocated here.  args(f64) checks and returns the operator's own
    arguments between pts and out (timestamps follow the layout); per_frame = (name, tensor) needs one row per frame."""
    f64 = _layout(pts)
    n, F = pts.shape[0], frame_off.shape[0] - 1
    if per_frame is not None and per_frame[1].shape[0] != F:
        raise ValueError(f"{per_frame[0]} must have one row per frame")
    if out is None and want_out:
        out = torch.empty_like(pts)
    ex, bufs = _make_export(export, n, pts.device)
    b, e = _range(n, p_range)
    fn = getattr(C.lib(), f"lmc_{name}_{'f64' if f64 else 'f32'}")
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), *args(f64), _req(out, pts.dtype, "out", (4,)), n, F, b, e,
               None if ex is None else C.ctypes.byref(ex), _stream_ptr()))
    return out, bufs


def _slerp_args(f64, ts, frame_off, frame_start, sample_ts, seg):
    """The Mode C arguments of deskew_slerp, deskew_slerp_local and distort_slerp: ts ... n_samples."""
    return (_req(ts, torch.int64 if f64 else torch.uint32, "ts"), _req(frame_off, torch.int64, "frame_off"),
            _req(frame_start, torch.int64, "frame_start"), _req(sample_ts, torch.int64, "sample_ts"),
            _req(seg, torch.float64, "seg", (22,)), sample_ts.shape[0])


@_on_tensor_device
def align_rigid(pts: torch.Tensor, frame_off: torch.Tensor, pose_Rt: torch.Tensor, *, out: Optional[torch.Tensor] = None,
                export: Optional[ExportSpec] = None, p_range=None, want_out: bool = True):
    """(a2)+(a3) LMC:772-776 over all frames, frame-major (LMC:888). Returns (aligned, ExportBuffers|None)."""
    return _point_op("align_rigid", pts, frame_off,
                     lambda f64: (_req(frame_off, torch.int64, "frame_off"), _req(pose_Rt, torch.float64, "pose_Rt", (12,))),
                     out, export, p_range, want_out, per_frame=("pose_Rt", pose_Rt))


@_on_tensor_device
def deskew_gyro(pts: torch.Tensor, ts: torch.Tensor, frame_off: torch.Tensor, frame_start: torch.Tensor,
                imu_ts: torch.Tensor, imu_gyro: torch.Tensor, *, out: Optional[torch.Tensor] = None,
                export: Optional[ExportSpec] = None, p_range=None, want_out: bool = True):
    """(a6)-(a8) CS:1435-1536. f64 points take int64 ns timestamps, f32 points uint32 ns offsets."""
    return _point_op("deskew_gyro", pts, frame_off,
                     lambda f64: (_req(ts, torch.int64 if f64 else torch.uint32, "ts"), _req(frame_off, torch.int64, "frame_off"),
                                  _req(frame_start, torch.int64, "frame_start"), _req(imu_ts, torch.int64, "imu_ts"),
                                  _req(imu_gyro, torch.float64, "imu_gyro", (3,)), imu_ts.shape[0]),
                     out, export, p_range, want_out)


@_on_tensor_device
def deskew_slerp(pts: torch.Tensor, ts: Optional[torch.Tensor], frame_off: torch.Tensor, frame_start: Optional[torch.Tensor],
                 sample_ts: torch.Tensor, seg: torch.Tensor, *, hold_idx: Optional[torch.Tensor] = None,
                 out: Optional[torch.Tensor] = None, export: Optional[ExportSpec] = None, p_range=None, want_out: bool = True):
    """Mode C: per-point bracket search + SLERP + lerp (+ optional hold-next = Mode A)."""
    return _point_op("deskew_slerp", pts, frame_off,
                     lambda f64: (*_slerp_args(f64, ts, frame_off, frame_start, sample_ts, seg), _req(hold_idx, torch.int32, "hold_idx")),
                     out, export, p_range, want_out)


@_on_tensor_device
def slerp_pose_at(sample_ts: torch.Tensor, seg: torch.Tensor, query_ts: torch.Tensor) -> torch.Tensor:
    """Mode C's pose at each int64 ns query time (same bracket, end clamps and alpha as deskew_slerp): (n, 12) f64 rows
    [R row-major | pos], the pose_Rt layout of align_rigid -- align_rigid with them is Mode A at the interpolated pose."""
    n = query_ts.shape[0]
    pose = torch.empty((n, 12), dtype=torch.float64, device=query_ts.device)
    C.check(C.lib().lmc_slerp_pose_at(_req(sample_ts, torch.int64, "sample_ts"), _req(seg, torch.float64, "seg", (22,)), sample_ts.shape[0],
                                      _req(query_ts, torch.int64, "query_ts"), n, pose.data_ptr(), _stream_ptr()))
    return pose


@_on_tensor_device
def deskew_slerp_local(pts: torch.Tensor, ts: torch.Tensor, frame_off: torch.Tensor, frame_start: Optional[torch.Tensor],
                       sample_ts: torch.Tensor, seg: torch.Tensor, ref_pose: torch.Tensor, *, out: Optional[torch.Tensor] = None,
                       export: Optional[ExportSpec] = None, p_range=None, want_out: bool = True):
    """Sensor-frame deskew: every point of frame f in the sensor frame of ref_pose[f] ((F, 12) f64, normally
    slerp_pose_at of the frame's start or end time), rotation and translation removed.  Arguments as deskew_slerp (no
    hold_idx); the world position is kept in f64 registers, so the f32 layout loses nothing at map-scale positions."""
    return _point_op("deskew_slerp_local", pts, frame_off,
                     lambda f64: (*_slerp_args(f64, ts, frame_off, frame_start, sample_ts, seg),
                                  _req(ref_pose, torch.float64, "ref_pose", (12,))),
                     out, export, p_range, want_out, per_frame=("ref_pose", ref_pose))


@_on_tensor_device
def distort_slerp(pts: torch.Tensor, ts: torch.Tensor, frame_off: torch.Tensor, frame_start: Optional[torch.Tensor],
                  sample_ts: torch.Tensor, seg: torch.Tensor, *, out: Optional[torch.Tensor] = None,
                  export: Optional[ExportSpec] = None, p_range=None, want_out: bool = True):
    """Distortion, the exact inverse of deskew_slerp: every WORLD point into the sensor frame of Mode C's pose at the
    point's own time, R(t)^T (W - x(t)) -- what a sensor moving along the sample table records of a static world.
    Arguments as deskew_slerp_local (no ref_pose); deskew_slerp of the result gives the world points back."""
    return _point_op("distort_slerp", pts, frame_off,
                     lambda f64: _slerp_args(f64, ts, frame_off, frame_start, sample_ts, seg),
                     out, export, p_range, want_out)


@_on_tensor_device
def quantize(pts: torch.Tensor, export: ExportSpec) -> ExportBuffers:
    """(a4)/(a5)/(a9)/(a10) stand-alone quantisers over an (N,4) point array."""
    f64 = _layout(pts)
    n = pts.shape[0]
    ex, bufs = _make_export(export, n, pts.device)
    if ex is None:
        raise ValueError("quantize: export spec selects no output")
    fn = C.lib().lmc_quantize_f64 if f64 else C.lib().lmc_quantize_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), n, C.ctypes.byref(ex), _stream_ptr()))
    return bufs


@_on_tensor_device
def build_slerp_table(sample_quat_xyzw: torch.Tensor, sample_pos: torch.Tensor, sample_ts: torch.Tensor,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The (S,22) pose-segment table of deskew_slerp built on the device from (S,4) quaternions (x y z w),
    (S,3) positions and int64 ns sample times -- the device twin of frames.slerp_segment_table."""
    S = sample_quat_xyzw.shape[0]
    if out is None:
        out = torch.empty((S, 22), dtype=torch.float64, device=sample_quat_xyzw.device)
    C.check(C.lib().lmc_build_slerp_table(_req(sample_quat_xyzw, torch.float64, "sample_quat", (4,)), _req(sample_pos, torch.float64, "sample_pos", (3,)),
                                          _req(sample_ts, torch.int64, "sample_ts"), S, _req(out, torch.float64, "seg", (22,)), _stream_ptr()))
    return out


@_on_tensor_device
def transform_homog(pts: torch.Tensor, T, order: int = C.HOMOG_BATCH, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(N3) CS:214-233: one 4x4 homogeneous matrix T (host array) over (n,4) points; order = _capi.HOMOG_BATCH
    (the reference call on n >= 2 points) or HOMOG_SINGLE (the call on one point, CS:2136-2138)."""
    import numpy as np
    f64 = _layout(pts)
    Th = np.ascontiguousarray(np.asarray(T, np.float64).reshape(4, 4))
    if out is None:
        out = torch.empty_like(pts)
    fn = C.lib().lmc_transform_homog_f64 if f64 else C.lib().lmc_transform_homog_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), Th.ctypes.data, int(order), _req(out, pts.dtype, "out", (4,)), pts.shape[0], _stream_ptr()))
    return out


@_on_tensor_device
def build_lvx_v11(pts: torch.Tensor, frame_off: torch.Tensor, frame_pos: torch.Tensor, frame_time: torch.Tensor,
                  frame_id: torch.Tensor, max_frame_points: int, size: Optional[int] = None):
    """(N1) LMC:58-250 on the device: RAW points -> the complete LVX v1.1 file image (uint8 tensor).
    frame_pos (int64[F+1], byte offsets incl. the 88-byte preamble) comes from lvx.frame_layout(); size = its last entry.
    Returns (file bytes tensor, status flags tensor)."""
    f64 = _layout(pts)
    F = frame_off.shape[0] - 1
    if size is None:
        size = int(frame_pos[-1].item())                    # (a host sync: pass the file size when the layout was made on the host)
    out = torch.empty(size, dtype=torch.uint8, device=pts.device)
    status = torch.zeros(1, dtype=torch.int32, device=pts.device)
    fn = C.lib().lmc_lvx_v11_build_f64 if f64 else C.lib().lmc_lvx_v11_build_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), _req(frame_off, torch.int64, "frame_off"), _req(frame_pos, torch.int64, "frame_pos"),
               _req(frame_time, torch.float64, "frame_time"), _req(frame_id, torch.int64, "frame_id"), out.data_ptr(),
               pts.shape[0], F, int(max_frame_points), status.data_ptr(), _stream_ptr()))
    return out, status


def _file_range_buffer(n_bytes: int, file_pos0: int, device) -> torch.Tensor:
    """uint8 buffer for file bytes [file_pos0, file_pos0 + n_bytes) whose address is congruent to file_pos0 modulo 16:
    the writer kernels assemble every byte range at the FILE's 16-byte phase (odd record starts in the LAS file stay odd)."""
    pad = file_pos0 % 16
    return torch.empty(pad + n_bytes, dtype=torch.uint8, device=device)[pad:]


@_on_tensor_device
def build_lvx_v11_range(pts: torch.Tensor, frame_off: torch.Tensor, frame_pos: torch.Tensor, frame_time: torch.Tensor,
                        frame_id: torch.Tensor, f_begin: int, f_end: int, file_pos0: int, n_bytes: int, max_frame_points: int):
    """(N1, SURVEY 8e) a rank's shard of the LVX v1.1 file: frames [f_begin, f_end) of the GLOBAL arrays.  The returned
    uint8 tensor holds file bytes [file_pos0, file_pos0 + n_bytes) -- file_pos0 = 0 for the rank owning frame 0 (its range
    starts with the 88-byte preamble), frame_pos[f_begin] otherwise; n_bytes = frame_pos[f_end] - file_pos0."""
    f64 = _layout(pts)
    F = frame_off.shape[0] - 1
    out = _file_range_buffer(max(int(n_bytes), 0), int(file_pos0), pts.device)
    status = torch.zeros(1, dtype=torch.int32, device=pts.device)
    fn = C.lib().lmc_lvx_v11_build_range_f64 if f64 else C.lib().lmc_lvx_v11_build_range_f32
    if n_bytes > 0:
        C.check(fn(_req(pts, pts.dtype, "pts", (4,)), _req(frame_off, torch.int64, "frame_off"), _req(frame_pos, torch.int64, "frame_pos"),
                   _req(frame_time, torch.float64, "frame_time"), _req(frame_id, torch.int64, "frame_id"), out.data_ptr(), int(file_pos0),
                   pts.shape[0], F, int(f_begin), int(f_end), int(max_frame_points), status.data_ptr(), _stream_ptr()))
    return out, status


@_on_tensor_device
def las_pf3_records(pts: torch.Tensor, p_begin: int, p_end: int, file_pos0: int, *, scale=(0.01, 0.01, 0.01), offset=(0.0, 0.0, 0.0),
                    intensity_mode: int = C.LAS_INTENSITY_UNIT, gps_time: Optional[torch.Tensor] = None):
    """(N2, SURVEY 8e) a rank's shard of the LAS 1.2 / PF3 file: the records of points [p_begin, p_end) of the GLOBAL
    cloud `pts`.  Returns (uint8 tensor = file bytes [file_pos0, 227 + 34 p_end), int32[6] shard extremes, status);
    file_pos0 = 0 for the rank that also holds the header (filled in later by las_pf3_header), 227 + 34 p_begin otherwise."""
    f64 = _layout(pts)
    n = pts.shape[0]
    size = C.LAS_HEADER_BYTES + C.LAS_RECORD_BYTES * int(p_end) - int(file_pos0)
    out = _file_range_buffer(size, int(file_pos0), pts.device)
    mm = torch.empty(6, dtype=torch.int32, device=pts.device)
    status = torch.zeros(1, dtype=torch.int32, device=pts.device)
    sc = (C.ctypes.c_double * 3)(*[float(v) for v in scale])
    of = (C.ctypes.c_double * 3)(*[float(v) for v in offset])
    fn = C.lib().lmc_las_pf3_records_f64 if f64 else C.lib().lmc_las_pf3_records_f32
    if size == 0:                                           # an empty shard: no bytes (its buffer has no address), neutral extremes
        mm[0::2], mm[1::2] = 2 ** 31 - 1, -2 ** 31
        return out, mm, status
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), _req(gps_time, torch.float64, "gps_time"), n, int(p_begin), int(p_end), sc, of,
               int(intensity_mode), out.data_ptr(), int(file_pos0), mm.data_ptr(), status.data_ptr(), _stream_ptr()))
    return out, mm, status


@_on_tensor_device
def las_pf3_header(header_out: torch.Tensor, minmax: torch.Tensor, n_points: int, *, scale=(0.01, 0.01, 0.01), offset=(0.0, 0.0, 0.0),
                   year: int = 2026, day_of_year: int = 1) -> None:
    """(N2, SURVEY 8e) the 227-byte LAS header of an n_points-record file from the (all-reduced) integer extremes,
    written into header_out[:227] (the first bytes of the header-owning rank's shard)."""
    sc = (C.ctypes.c_double * 3)(*[float(v) for v in scale])
    of = (C.ctypes.c_double * 3)(*[float(v) for v in offset])
    C.check(C.lib().lmc_las_pf3_header(int(n_points), sc, of, int(year), int(day_of_year), _req(minmax, torch.int32, "minmax"),
                                       _req(header_out, torch.uint8, "header_out"), _stream_ptr()))


@_on_tensor_device
def build_lvx_cs(pts: torch.Tensor, tag: Optional[torch.Tensor], frame_off: torch.Tensor, frame_ts: torch.Tensor,
                 prefix: bytes, fmt: int, max_frame_points: int):
    """(N1) CS:245-374 on the device: COMPENSATED points [x y z intensity] (+ tag bytes) -> the complete LVX2 / LVX3
    (fmt = _capi.LVXCS_LVX2) or legacy LVX (LVXCS_LEGACY) file image.  prefix = the file's leading bytes
    (lvx.lvx_cs_prefix); frame_ts int64 ns >= 0.  Returns (file bytes tensor, status flags tensor)."""
    f64 = _layout(pts)
    n, F = pts.shape[0], frame_off.shape[0] - 1
    if len(prefix) > C.LVXCS_PREFIX_MAX:
        raise ValueError("prefix too long")
    size = len(prefix) + C.LVXCS_FRAME_BYTES[int(fmt)] * F + 14 * n
    out = torch.empty(size, dtype=torch.uint8, device=pts.device)
    status = torch.zeros(1, dtype=torch.int32, device=pts.device)
    pre = (C.ctypes.c_uint8 * max(len(prefix), 1)).from_buffer_copy(bytes(prefix) or b"\0")
    fn = C.lib().lmc_lvx_cs_build_f64 if f64 else C.lib().lmc_lvx_cs_build_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), _req(tag, torch.uint8, "tag"), _req(frame_off, torch.int64, "frame_off"),
               _req(frame_ts, torch.int64, "frame_ts"), pre, len(prefix), int(fmt), out.data_ptr(), n, F, int(max_frame_points),
               status.data_ptr(), _stream_ptr()))
    return out, status


def _pcd_format(pts: torch.Tensor):
    """LMC:946-947 for every row of pts -> (text, tile_off, status): lmc_pcd_ascii_size_* (line lengths need no digits: four
    compares per number), one host read of the total, lmc_pcd_ascii_write_* into the exactly sized buffer."""
    f64 = _layout(pts)
    n = pts.shape[0]
    tiles = (n + C.PCD_TILE - 1) // C.PCD_TILE
    tile_off = torch.empty(tiles + 1, dtype=torch.int64, device=pts.device)
    status = torch.zeros(1, dtype=torch.int32, device=pts.device)
    L = C.lib()
    ptr = _req(pts, pts.dtype, "pts", (4,))
    C.check((L.lmc_pcd_ascii_size_f64 if f64 else L.lmc_pcd_ascii_size_f32)(ptr, n, tile_off.data_ptr(), _stream_ptr()))
    total = int(tile_off[-1].item())                       # the one host sync: the text buffer has to be sized
    out = torch.empty(total, dtype=torch.uint8, device=pts.device)
    C.check((L.lmc_pcd_ascii_write_f64 if f64 else L.lmc_pcd_ascii_write_f32)(ptr, n, tile_off.data_ptr(), out.data_ptr(), status.data_ptr(), _stream_ptr()))
    return out, tile_off, status


@_on_tensor_device
def pcd_ascii_body(pts: torch.Tensor):
    """(N2) LMC:946-947 on the device: one '%.6f %.6f %.6f %.6f\\n' line per row, byte-identical to the
    reference's f-string formatting.  Returns (uint8 text tensor, status flags tensor)."""
    out, _, status = _pcd_format(pts)
    return out, status


@_on_tensor_device
def pcd_ascii_frames(pts: torch.Tensor, frame_off: torch.Tensor):
    """(N2) the '%.6f' bodies of EVERY per-frame PCD file in one formatting pass: pts is the frame-major buffer,
    frame_off int64[F+1] its CSR offsets (device).  Returns (uint8 text tensor, int64[F+1] device byte offsets,
    status): frame f's file body (LMC:946-947 over that frame's rows) is text[byte_off[f]:byte_off[f+1]], and the
    whole text is the body of the merged file (np.vstack order, LMC:888 / 897)."""
    f64 = _layout(pts)
    n = pts.shape[0]
    out, tile_off, status = _pcd_format(pts)
    nq = frame_off.shape[0]
    byte_off = torch.empty(nq, dtype=torch.int64, device=pts.device)
    L = C.lib()
    C.check((L.lmc_pcd_ascii_row_offsets_f64 if f64 else L.lmc_pcd_ascii_row_offsets_f32)(
        _req(pts, pts.dtype, "pts", (4,)), n, tile_off.data_ptr(), _req(frame_off, torch.int64, "frame_off"), nq, byte_off.data_ptr(), _stream_ptr()))
    return out, byte_off, status


@_on_tensor_device
def text_rows(rows: torch.Tensor, cols, decimals, sep: str = " "):
    """(N2) CS:1643-1716 on the device: one line per row of a 2-D f64 / f32 tensor, column cols[k] printed as
    '%.{decimals[k]}f', joined by sep, '\\n' terminated -- byte-identical to the reference's f-strings /
    np.savetxt / pandas float_format.  Returns (uint8 text tensor, status flags tensor)."""
    if rows.dim() != 2 or rows.dtype not in (torch.float64, torch.float32):
        raise TypeError("rows: expected a 2-D float64 / float32 CUDA tensor")
    f64 = rows.dtype == torch.float64
    n, stride = rows.shape
    k = len(cols)
    if k != len(decimals) or not 1 <= k <= C.TEXT_MAX_COLS:
        raise ValueError(f"1..{C.TEXT_MAX_COLS} columns, one decimals entry each")
    ca = (C.ctypes.c_int32 * k)(*[int(c) for c in cols])
    da = (C.ctypes.c_int32 * k)(*[int(v) for v in decimals])
    tiles = (n + C.PCD_TILE - 1) // C.PCD_TILE
    tile_off = torch.empty(tiles + 1, dtype=torch.int64, device=rows.device)
    L = C.lib()
    fs, fw = (L.lmc_text_rows_size_f64, L.lmc_text_rows_write_f64) if f64 else (L.lmc_text_rows_size_f32, L.lmc_text_rows_write_f32)
    ptr = _req(rows, rows.dtype, "rows")
    C.check(fs(ptr, n, stride, k, ca, da, ord(sep), tile_off.data_ptr(), _stream_ptr()))
    size = int(tile_off[-1].item())
    out = torch.empty(size, dtype=torch.uint8, device=rows.device)
    status = torch.zeros(1, dtype=torch.int32, device=rows.device)
    C.check(fw(ptr, n, stride, k, ca, da, ord(sep), tile_off.data_ptr(), out.data_ptr(), status.data_ptr(), _stream_ptr()))
    return out, status


@_on_tensor_device
def build_las_pf3(pts: torch.Tensor, *, scale=(0.01, 0.01, 0.01), offset=(0.0, 0.0, 0.0), intensity_mode: int = C.LAS_INTENSITY_UNIT,
                  gps_time: Optional[torch.Tensor] = None, year: int = 2026, day_of_year: int = 1):
    """(N2) A complete LAS 1.2 / PF3 file image on the device (parity unpinned: laspy absent; LAS 1.2 spec).
    Returns (uint8 file tensor, status flags tensor)."""
    f64 = _layout(pts)
    n = pts.shape[0]
    out = torch.empty(C.LAS_HEADER_BYTES + C.LAS_RECORD_BYTES * n, dtype=torch.uint8, device=pts.device)
    mm = torch.empty(6, dtype=torch.int32, device=pts.device)
    status = torch.zeros(1, dtype=torch.int32, device=pts.device)
    sc = (C.ctypes.c_double * 3)(*[float(v) for v in scale])
    of = (C.ctypes.c_double * 3)(*[float(v) for v in offset])
    fn = C.lib().lmc_las_pf3_build_f64 if f64 else C.lib().lmc_las_pf3_build_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)), _req(gps_time, torch.float64, "gps_time"), n, sc, of, int(intensity_mode),
               int(year), int(day_of_year), out.data_ptr(), mm.data_ptr(), status.data_ptr(), _stream_ptr()))
    return out, status


def _grid3(v, name):
    import numpy as np
    a = np.broadcast_to(np.asarray(v, np.float64), (3,))
    if not np.isfinite(a).all() or (name == "leaf" and not (a > 0).all()):
        raise ValueError(f"{name} must be three finite values{' > 0' if name == 'leaf' else ''} (or one, broadcast)")
    return (C.ctypes.c_double * 3)(*[float(x) for x in a])


@_on_tensor_device
def voxel_downsample(pts: torch.Tensor, leaf, origin=(0.0, 0.0, 0.0), *, point_voxel: bool = False):
    """Voxel-grid map of an (N,4) cloud on the device: the centroid and the point count of every occupied voxel of the
    grid with cell size `leaf` (three values or one) anchored at `origin`, voxels ranked by their first point (a
    frame-major cloud's map grows frame by frame).  Exact integer sums: the result is bit-identical from run to run and
    under any permutation of the input.  A point with a non-finite value, a key beyond 2^20 cells from the origin on an
    axis or |intensity| >= 256 belongs to no voxel and sets C.FLAG_NAN / C.FLAG_OVERFLOW in status.
    Returns (centroids (V,4) in pts' dtype, counts int32[V], point_voxel int32[N] (voxel rank, -1 dropped) or None,
    status (1) int32)."""
    f64 = _layout(pts)
    n, dev = pts.shape[0], pts.device
    L, O = _grid3(leaf, "leaf"), _grid3(origin, "origin")
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    pv = torch.empty(n, dtype=torch.int32, device=dev) if point_voxel else None
    if n == 0:
        return torch.empty((0, 4), dtype=pts.dtype, device=dev), torch.empty(0, dtype=torch.int32, device=dev), pv, status
    lib = C.lib()
    ws = torch.empty(int(lib.lmc_voxel_workspace_bytes(n)), dtype=torch.uint8, device=dev)
    nv = torch.empty(1, dtype=torch.int64, device=dev)
    ptr = _req(pts, pts.dtype, "pts", (4,))
    C.check((lib.lmc_voxel_index_f64 if f64 else lib.lmc_voxel_index_f32)(ptr, n, L, O, ws.data_ptr(), nv.data_ptr(), status.data_ptr(),
                                                                          _stream_ptr()))
    V = int(nv.item())                                      # the one host sync: the outputs are sized by V
    cent = torch.empty((V, 4), dtype=pts.dtype, device=dev)
    counts = torch.empty(V, dtype=torch.int32, device=dev)
    C.check((lib.lmc_voxel_reduce_f64 if f64 else lib.lmc_voxel_reduce_f32)(ptr, n, L, O, ws.data_ptr(), V, cent.data_ptr(), counts.data_ptr(),
                                                                            _req(pv, torch.int32, "point_voxel"), _stream_ptr()))
    return cent, counts, pv, status


@dataclass
class PointMap:
    """A prior point map on the device (build_point_map): the map points sorted by voxel on the voxel map's grid, their
    original rows, CSR voxel offsets and the key -> voxel-rank lookup table (keys int64[cap] | ranks int32[cap], an empty
    slot has key -1)."""
    pts: torch.Tensor                # (M,4) f64, sorted by voxel rank
    index: torch.Tensor              # int64[M] original row
    vox_off: torch.Tensor            # int64[V+1]
    table: torch.Tensor              # uint8 lookup table, lmc_map_workspace_bytes(V) bytes
    leaf: tuple
    origin: tuple

    @property
    def n_voxels(self) -> int:
        return self.vox_off.shape[0] - 1

    @property
    def keys(self) -> torch.Tensor:
        cap = self._cap()
        return self.table[:8 * cap].view(torch.int64)

    @property
    def ranks(self) -> torch.Tensor:
        cap = self._cap()
        b = (8 * cap + 255) // 256 * 256
        return self.table[b:b + 4 * cap].view(torch.int32)

    def _cap(self) -> int:
        c = 64
        while c < 2 * self.n_voxels:
            c <<= 1
        return c

    def _c(self) -> "C.LmcPointMap":
        m = C.LmcPointMap()
        m.pts_m4, m.index, m.vox_off = self.pts.data_ptr() or None, self.index.data_ptr() or None, self.vox_off.data_ptr()
        m.table = self.table.data_ptr()
        m.n_points, m.n_voxels = self.pts.shape[0], self.n_voxels
        for c in range(3):
            m.leaf[c], m.origin[c] = self.leaf[c], self.origin[c]
        return m


@_on_tensor_device
def build_point_map(map_pts: torch.Tensor, leaf, origin=(0.0, 0.0, 0.0)) -> PointMap:
    """Build a prior point map of the (M,4) cloud `map_pts` on the voxel map's grid (`leaf`: three values or one, anchored
    at `origin`; keys limited to 2^20 cells from the origin per axis, so a UTM-scale map needs an origin near the data).
    The voxel ranks and counts come from voxel_downsample, the rows are sorted stably by voxel, and k_map_insert fills
    the lookup table.  ValueError for a NaN / inf map point, OverflowError for one beyond the key range or with
    |intensity| >= 256, as voxel_map."""
    L, O = _grid3(leaf, "leaf"), _grid3(origin, "origin")
    _, counts, pv, status = voxel_downsample(map_pts, leaf, origin, point_voxel=True)
    ExportBuffers(status=status).raise_for_flags()
    dev = map_pts.device
    order = torch.argsort(pv.long(), stable=True)
    pts = map_pts.index_select(0, order).to(torch.float64).contiguous()
    vox_off = torch.zeros(counts.shape[0] + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=vox_off[1:])
    lib = C.lib()
    table = torch.empty(int(lib.lmc_map_workspace_bytes(counts.shape[0])), dtype=torch.uint8, device=dev)
    pm = PointMap(pts, order.contiguous(), vox_off, table, tuple(L), tuple(O))
    m = pm._c()
    C.check(lib.lmc_map_build(C.ctypes.byref(m), _stream_ptr()))
    return pm


def _gate(pmap: PointMap, max_dist) -> float:
    d = float(max_dist)
    if not (d > 0.0 and d < float("inf")) or d > min(pmap.leaf):
        raise ValueError("max_dist must be finite, > 0 and <= min(leaf): the 27 cells around a query must cover its ball")
    return d


@_on_tensor_device
def map_nearest(pts: torch.Tensor, pmap: PointMap, max_dist: float):
    """Exact fixed-radius nearest neighbour of every query row of the (N,4) cloud `pts` in `pmap`: the map point with the
    smallest d2 = (dx dx + dy dy) + dz dz (f64, every operation rounded to nearest) among those with d2 <= max_dist^2;
    equal distances go to the smaller original map row.  max_dist <= min(leaf) is required.  A query with a non-finite
    coordinate (which sets C.FLAG_NAN in status) or outside the key range has no match.
    Returns (index int64[N] original map row or -1, d2 f64[N] (+inf without a match), status (1) int32)."""
    f64 = _layout(pts)
    d = _gate(pmap, max_dist)
    n, dev = pts.shape[0], pts.device
    idx = torch.empty(n, dtype=torch.int64, device=dev)
    d2 = torch.empty(n, dtype=torch.float64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    m = pmap._c()
    fn = C.lib().lmc_map_nearest_f64 if f64 else C.lib().lmc_map_nearest_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)) if n else None, n, C.ctypes.byref(m), d, idx.data_ptr() or None,
               d2.data_ptr() or None, status.data_ptr(), _stream_ptr()))
    return idx, d2, status


@dataclass
class RegStats:
    """Per-frame results of register_frames."""
    inliers: torch.Tensor            # int32[F] inliers of the last iteration
    rms_m: torch.Tensor              # f64[F] rms point-to-point residual of the last iteration (NaN without inliers)
    iterations: torch.Tensor         # int32[F] iterations the frame ran
    flags: torch.Tensor              # int32[F] C.REG_CONVERGED | C.REG_DEGENERATE
    status: torch.Tensor             # (1) int32, C.FLAG_NAN for a non-finite point

    @property
    def converged(self) -> torch.Tensor:
        return (self.flags & C.REG_CONVERGED) != 0

    @property
    def degenerate(self) -> torch.Tensor:
        return (self.flags & C.REG_DEGENERATE) != 0


@_on_tensor_device
def register_frames(pts: torch.Tensor, frame_off: torch.Tensor, pose_Rt: torch.Tensor, pmap: PointMap, max_dist: float,
                    iters: int = 30, tol_t: float = 1e-9, tol_r: float = 1e-12):
    """Refine every frame's pose against the map by point-to-point Gauss-Newton on the device.  pts: sensor-frame clouds
    (raw hold-next scans, or deskew_slerp_local's output), frame-major with CSR frame_off; pose_Rt: the initial (F,12)
    [R | t] table (align_rigid's layout).  Each iteration pairs every point's w = R p + t with its nearest map point
    within max_dist (map_nearest's rule), solves the 6x6 normal equations for [tau; phi] (rotation about the sensor
    position) by Cholesky and applies t += tau, R = Exp(phi) R.  A frame with fewer than 6 inliers or a singular system
    is degenerate and keeps its pose; one whose step is within tol_t (m) and tol_r (rad) is converged and stops.
    No float atomics: two calls give identical bytes.  The result is not invariant under a permutation of the points
    (their order fixes the summation order).  Returns (refined (F,12) f64 pose table, RegStats)."""
    f64 = _layout(pts)
    d = _gate(pmap, max_dist)
    if int(iters) < 1:
        raise ValueError("iters must be >= 1")
    n, F, dev = pts.shape[0], frame_off.shape[0] - 1, pts.device
    if pose_Rt.shape[0] != F:
        raise ValueError("pose_Rt must have one row per frame")
    lib = C.lib()
    ws = torch.empty(max(int(lib.lmc_register_workspace_bytes(n, F)), 1), dtype=torch.uint8, device=dev)
    pose = torch.empty((F, 12), dtype=torch.float64, device=dev)
    st = RegStats(torch.empty(F, dtype=torch.int32, device=dev), torch.empty(F, dtype=torch.float64, device=dev),
                  torch.empty(F, dtype=torch.int32, device=dev), torch.empty(F, dtype=torch.int32, device=dev),
                  torch.zeros(1, dtype=torch.int32, device=dev))
    m = pmap._c()
    fn = lib.lmc_register_frames_f64 if f64 else lib.lmc_register_frames_f32
    C.check(fn(_req(pts, pts.dtype, "pts", (4,)) if n else None, n, _req(frame_off, torch.int64, "frame_off"), F,
               _req(pose_Rt, torch.float64, "pose_Rt", (12,)), C.ctypes.byref(m), d, int(iters), float(tol_t), float(tol_r),
               ws.data_ptr(), pose.data_ptr(), st.inliers.data_ptr(), st.rms_m.data_ptr(), st.iterations.data_ptr(),
               st.flags.data_ptr(), st.status.data_ptr(), _stream_ptr()))
    return pose, st


def _redecide_uncertain(env, pos, Rm, flags, fov_h, fov_v, range_min) -> int:
    """Host re-decision of the points k_scan_mark flagged uncertain (bit 1), with the NumPy calls of LMC:726-745."""
    import numpy as np
    fi, pi = torch.nonzero(flags & 2, as_tuple=True)
    if fi.numel() == 0:
        return 0
    e = env[pi][:, :3].cpu().numpy()
    fi_h = fi.cpu().numpy()
    p = pos.cpu().numpy()[fi_h]
    Rall = Rm.cpu().numpy().reshape(-1, 3, 3)
    rel = e - p
    d2 = np.sum(rel ** 2, axis=1)
    rot = np.empty_like(rel)
    # one matmul per FRAME that has flagged points (torch.nonzero is frame-major, so each frame's points are one slice) --
    # the reference's own expression (LMC:726: R.T @ rel.T over the frame's points), not a Python iteration per point
    starts = np.flatnonzero(np.r_[True, fi_h[1:] != fi_h[:-1]])
    ends = np.r_[starts[1:], len(fi_h)]
    for a, b in zip(starts, ends):
        rot[a:b] = (Rall[fi_h[a]].T @ rel[a:b].T).T
    x, y, z = rot[:, 0], rot[:, 1], rot[:, 2]
    ranges = np.sqrt(d2)
    azimuth = np.arctan2(y, x) * 180 / np.pi
    elevation = np.arcsin(np.clip(z / np.maximum(ranges, 1e-6), -1, 1)) * 180 / np.pi
    vis = (np.abs(azimuth) <= fov_h) & (np.abs(elevation) <= fov_v) & (ranges >= range_min)
    flags[fi, pi] = torch.from_numpy(vis.astype(np.uint8)).to(flags.device)
    return int(fi.numel())


@_on_tensor_device
def scan_frames(env: torch.Tensor, pos: torch.Tensor, Rm: torch.Tensor, *, range_max: float, range_min: float,
                fov_horizontal: float, fov_vertical: float, points_per_frame: int, noise_std: float, noise_fn=None,
                max_flag_bytes: int = 1 << 30, edge_eps_deg: float = 1e-9, motion=None):
    """(N4) LMC:701-770 for every frame at once.  env (M,4) f64, pos (F,3), Rm (F,9) row-major SciPy matrices.
    Returns (raw (N,4) f64 device tensor, frame_off np.int64[F+1]).

    motion = (sample_ts, seg, frame_start, period_ns) (device int64 sample times, the (S,22) table of build_slerp_table,
    host int64[F] frame start times, the frame period in ns) simulates a moving sensor: which points a frame sees is
    still decided at pos[f] / Rm[f], but point j of the m_f kept points of frame f is observed at time
    frame_start[f] + (j * period_ns) // m_f from Mode C's pose there (distort_slerp), and the same noise is added in that
    sensor frame.  Returns (raw, frame_off, point times np.int64[N], env row indices (N) int64 device tensor) then.

    noise_fn(n) must return the (n,3) host array the reference would draw -- by default
    ``np.random.normal(0, noise_std, (n, 3))`` from the GLOBAL legacy NumPy RNG (replayed bit-identically by
    ``frames.legacy_normal``, which leaves the generator where NumPy would), exactly the stream LMC:767
    consumes frame after frame (the legacy generator is a stream: one draw per chunk of frames == the
    reference's per-frame draws).  Frames are processed in chunks so the F x M visibility scratch stays
    below max_flag_bytes; chunks run in frame order, so the noise stream keeps the reference's order.

    Points whose |azimuth| / |elevation| lies within edge_eps_deg of the FOV limit (where a few ulp of device
    atan2 / asin could decide differently from the host libm) are re-decided on the host with the reference's
    own NumPy expression (LMC:726-745), so every visibility decision is the reference's."""
    import numpy as np
    M, F = env.shape[0], pos.shape[0]
    tiles = (M + C.SCAN_TILE - 1) // C.SCAN_TILE
    dev = env.device
    rmax2 = float(range_max ** 2)                                   # LMC:714
    maxp = int(points_per_frame)
    if maxp < 1:                                                    # (the kept counts below would silently be 0)
        raise ValueError(f"points_per_frame must be >= 1, got {points_per_frame}")
    L = C.lib()
    _req(env, torch.float64, "env", (4,)); _req(pos, torch.float64, "pos", (3,)); _req(Rm, torch.float64, "Rm", (9,))
    chunk = max(1, min(F, max_flag_bytes // max(M, 1)))
    outs, kept_all, idx_all, ts_all = [], [], [], []
    if motion is not None:
        s_ts, seg, fstart, period_ns = motion
        fstart = np.asarray(fstart, np.int64)
        if fstart.shape != (F,):
            raise ValueError("motion: frame_start needs one entry per frame")
        _req(s_ts, torch.int64, "sample_ts"); _req(seg, torch.float64, "seg", (22,))
    for f0 in range(0, F, chunk):
        f1 = min(F, f0 + chunk)
        nf = f1 - f0
        p_c, r_c = pos[f0:f1], Rm[f0:f1]
        flags = torch.empty((nf, max(M, 1)), dtype=torch.uint8, device=dev)
        tile_off = torch.empty((nf, tiles + 1), dtype=torch.int32, device=dev)
        cnt = torch.empty(nf + 1, dtype=torch.int32, device=dev)    # n_visible[nf] | n_uncertain
        n_vis = cnt[:nf]
        C.check(L.lmc_scan_mark(env.data_ptr(), M, p_c.data_ptr(), r_c.data_ptr(), nf, rmax2, float(fov_horizontal / 2),
                                float(fov_vertical / 2), float(range_min), float(edge_eps_deg), flags.data_ptr(), tile_off.data_ptr(),
                                n_vis.data_ptr(), cnt[nf:].data_ptr(), _stream_ptr()))
        cnt_h = cnt.cpu().numpy()                                   # the one sync per chunk: the noise draw is sized by these counts
        if cnt_h[nf] > 0:                                           # FOV-edge points: the reference's own arithmetic decides
            _redecide_uncertain(env, p_c, r_c, flags, fov_horizontal / 2, fov_vertical / 2, range_min)
            C.check(L.lmc_scan_recount(flags.data_ptr(), M, nf, tile_off.data_ptr(), n_vis.data_ptr(), _stream_ptr()))
            cnt_h = cnt.cpu().numpy()
        nv = cnt_h[:nf].astype(np.int64)
        step = np.maximum(nv // maxp, 1)
        kept = np.where(nv > maxp, np.minimum((nv + step - 1) // step, maxp), nv)
        off_c = np.zeros(nf + 1, np.int64)
        np.cumsum(kept, out=off_c[1:])
        n_c = int(off_c[-1])
        out = torch.empty((n_c, 4), dtype=torch.float64, device=dev)
        if n_c > 0:
            noise_d = None
            if noise_std > 0:
                if noise_fn is None:
                    # the reference's own draw, np.random.normal(0, noise_std, (n_c, 3)) on the global generator, replayed
                    # bit-identically by lmc_host_legacy_normal (threaded sqrt / log) straight into pinned memory
                    from .frames import legacy_normal
                    stage = torch.empty(3 * n_c, dtype=torch.float64, pin_memory=dev.type == 'cuda')
                    legacy_normal(float(noise_std), 3 * n_c, out=stage.numpy())
                    noise_d = stage.to(dev, non_blocking=True).view(n_c, 3)
                else:
                    noise_d = torch.from_numpy(np.ascontiguousarray(noise_fn(n_c), dtype=np.float64)).to(dev)
            fo = torch.from_numpy(off_c).to(dev)
            if motion is None:
                C.check(L.lmc_scan_emit(env.data_ptr(), M, p_c.data_ptr(), r_c.data_ptr(), nf, rmax2, flags.data_ptr(), tile_off.data_ptr(),
                                        n_vis.data_ptr(), fo.data_ptr(), maxp, _req(noise_d, torch.float64, "noise", (3,)), out.data_ptr(), _stream_ptr()))
            else:
                idx = torch.empty(n_c, dtype=torch.int64, device=dev)
                C.check(L.lmc_scan_emit_index(env.data_ptr(), M, p_c.data_ptr(), r_c.data_ptr(), nf, rmax2, flags.data_ptr(), tile_off.data_ptr(),
                                              n_vis.data_ptr(), fo.data_ptr(), maxp, idx.data_ptr(), _stream_ptr()))
                m = np.diff(off_c)
                fidx = np.repeat(np.arange(nf), m)
                j = np.arange(n_c, dtype=np.int64) - off_c[fidx]
                ts_c = fstart[f0 + fidx] + (j * int(period_ns)) // m[fidx]       # the point-time convention of the deskews
                distort_slerp(env[idx], torch.from_numpy(ts_c).to(dev), fo, None, s_ts, seg, out=out)
                if noise_d is not None:
                    out[:, :3] += noise_d                                        # LMC:768, in the sensor frame of the point's pose
                idx_all.append(idx)
                ts_all.append(ts_c)
        elif motion is not None:
            idx_all.append(torch.empty(0, dtype=torch.int64, device=dev))
            ts_all.append(np.zeros(0, np.int64))
        outs.append(out)
        kept_all.append(kept)
    kept_all = np.concatenate(kept_all) if kept_all else np.zeros(0, np.int64)
    frame_off = np.zeros(F + 1, np.int64)
    np.cumsum(kept_all, out=frame_off[1:])
    raw = outs[0] if len(outs) == 1 else (torch.cat(outs, dim=0) if outs else torch.empty((0, 4), dtype=torch.float64, device=dev))
    if motion is None:
        return raw, frame_off
    env_idx = torch.cat(idx_all) if idx_all else torch.empty(0, dtype=torch.int64, device=dev)
    point_ts = np.concatenate(ts_all) if ts_all else np.zeros(0, np.int64)
    return raw, frame_off, point_ts, env_idx
