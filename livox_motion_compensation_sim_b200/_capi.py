"""ctypes binding of include/lmc_b200.h.  There is no fallback: if liblmc_b200.so is missing or a
call fails, this raises."""
from __future__ import annotations

import ctypes
import os

from ._build import LIB_PATH

OK, ERR_INVALID, ERR_ALIGN, ERR_CUDA = 0, -1, -2, -3
FLAG_NAN, FLAG_OVERFLOW = 1, 2
LVX_TYPE2_OF_INPUT, LVX2_OF_OUTPUT = 0, 1
LVXCS_LVX2, LVXCS_LEGACY = 0, 1
LVXCS_PREFIX_MAX = 96
TEXT_MAX_COLS = 6
HOMOG_BATCH, HOMOG_SINGLE = 0, 1
LVXCS_FRAME_BYTES = {0: 45, 1: 12}
LAS_INTENSITY_UNIT, LAS_INTENSITY_RAW = 0, 1
PATH_DIRECT, PATH_AUTO, PATH_TMA = 0, 1, 2
PCD_TILE = 256
MAX_PEERS = 7
LAS_HEADER_BYTES, LAS_RECORD_BYTES = 227, 34
SCAN_TILE = 256
REG_CONVERGED, REG_DEGENERATE = 1, 2

vp, i64, i32, f64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double


class LmcExport(ctypes.Structure):
    """struct lmc_export (include/lmc_b200.h)"""
    _fields_ = [
        ("lvx14", vp), ("lvx_mode", i32), ("tag", vp),
        ("las_x", vp), ("las_y", vp), ("las_z", vp), ("las_intensity", vp),
        ("las_intensity_mode", i32),
        ("las_scale", ctypes.c_double * 3), ("las_offset", ctypes.c_double * 3),
        ("status", vp),
        ("n_peers", i32), ("peer_out", vp * 7), ("peer_lvx14", vp * 7),
        ("mc_out", vp), ("mc_lvx14", vp),
    ]


class LmcPointMap(ctypes.Structure):
    """struct lmc_point_map (include/lmc_b200.h)"""
    _fields_ = [
        ("pts_m4", vp), ("index", vp), ("vox_off", vp), ("table", vp),
        ("n_points", i64), ("n_voxels", i64),
        ("leaf", ctypes.c_double * 3), ("origin", ctypes.c_double * 3),
    ]


class LmcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liblmc_b200 error {code}: {msg}")
        self.code = code


_SIGNATURES = {
    "lmc_version": ([], ctypes.c_int),
    "lmc_last_error": ([], ctypes.c_char_p),
    "lmc_device_query": ([vp, vp, vp], ctypes.c_int),
    "lmc_set_path": ([i32], ctypes.c_int),
    "lmc_get_path": ([], ctypes.c_int),
    "lmc_pose_lookup_hold_next": ([vp, i64, vp, vp, i32, vp, vp, vp], ctypes.c_int),
    "lmc_align_rigid_f64": ([vp, vp, vp, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_align_rigid_f32": ([vp, vp, vp, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_deskew_gyro_f64": ([vp, vp, vp, vp, vp, vp, i64, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_deskew_gyro_f32": ([vp, vp, vp, vp, vp, vp, i64, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_deskew_slerp_f64": ([vp, vp, vp, vp, vp, vp, i64, vp, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_deskew_slerp_f32": ([vp, vp, vp, vp, vp, vp, i64, vp, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_build_slerp_table": ([vp, vp, vp, i64, vp, vp], ctypes.c_int),
    "lmc_slerp_pose_at": ([vp, vp, i64, vp, i64, vp, vp], ctypes.c_int),
    "lmc_deskew_slerp_local_f64": ([vp, vp, vp, vp, vp, vp, i64, vp, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_deskew_slerp_local_f32": ([vp, vp, vp, vp, vp, vp, i64, vp, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_distort_slerp_f64": ([vp, vp, vp, vp, vp, vp, i64, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_distort_slerp_f32": ([vp, vp, vp, vp, vp, vp, i64, vp, i64, i32, i64, i64, vp, vp], ctypes.c_int),
    "lmc_quantize_f64": ([vp, i64, vp, vp], ctypes.c_int),
    "lmc_quantize_f32": ([vp, i64, vp, vp], ctypes.c_int),
    "lmc_lvx_v11_build_f64": ([vp, vp, vp, vp, vp, vp, i64, i32, i64, vp, vp], ctypes.c_int),
    "lmc_lvx_v11_build_f32": ([vp, vp, vp, vp, vp, vp, i64, i32, i64, vp, vp], ctypes.c_int),
    "lmc_lvx_v11_build_range_f64": ([vp, vp, vp, vp, vp, vp, i64, i64, i32, i32, i32, i64, vp, vp], ctypes.c_int),
    "lmc_lvx_v11_build_range_f32": ([vp, vp, vp, vp, vp, vp, i64, i64, i32, i32, i32, i64, vp, vp], ctypes.c_int),
    "lmc_las_pf3_records_f64": ([vp, vp, i64, i64, i64, vp, vp, i32, vp, i64, vp, vp, vp], ctypes.c_int),
    "lmc_las_pf3_records_f32": ([vp, vp, i64, i64, i64, vp, vp, i32, vp, i64, vp, vp, vp], ctypes.c_int),
    "lmc_las_pf3_header": ([i64, vp, vp, i32, i32, vp, vp, vp], ctypes.c_int),
    "lmc_transform_homog_f64": ([vp, vp, i32, vp, i64, vp], ctypes.c_int),
    "lmc_transform_homog_f32": ([vp, vp, i32, vp, i64, vp], ctypes.c_int),
    "lmc_lvx_cs_build_f64": ([vp, vp, vp, vp, vp, i32, i32, vp, i64, i32, i64, vp, vp], ctypes.c_int),
    "lmc_lvx_cs_build_f32": ([vp, vp, vp, vp, vp, i32, i32, vp, i64, i32, i64, vp, vp], ctypes.c_int),
    "lmc_pcd_ascii_size_f64": ([vp, i64, vp, vp], ctypes.c_int),
    "lmc_pcd_ascii_size_f32": ([vp, i64, vp, vp], ctypes.c_int),
    "lmc_pcd_ascii_write_f64": ([vp, i64, vp, vp, vp, vp], ctypes.c_int),
    "lmc_pcd_ascii_write_f32": ([vp, i64, vp, vp, vp, vp], ctypes.c_int),
    "lmc_pcd_ascii_row_offsets_f64": ([vp, i64, vp, vp, i32, vp, vp], ctypes.c_int),
    "lmc_pcd_ascii_row_offsets_f32": ([vp, i64, vp, vp, i32, vp, vp], ctypes.c_int),
    "lmc_host_gather": ([vp, vp, i64, vp, i32], ctypes.c_int),
    "lmc_host_copy": ([vp, vp, i64, i32], ctypes.c_int),
    "lmc_host_legacy_normal": ([vp, vp, vp, vp, f64, f64, i64, vp, i32], ctypes.c_int),
    "lmc_text_rows_size_f64": ([vp, i64, i32, i32, vp, vp, i32, vp, vp], ctypes.c_int),
    "lmc_text_rows_size_f32": ([vp, i64, i32, i32, vp, vp, i32, vp, vp], ctypes.c_int),
    "lmc_text_rows_write_f64": ([vp, i64, i32, i32, vp, vp, i32, vp, vp, vp, vp], ctypes.c_int),
    "lmc_text_rows_write_f32": ([vp, i64, i32, i32, vp, vp, i32, vp, vp, vp, vp], ctypes.c_int),
    "lmc_las_pf3_build_f64": ([vp, vp, i64, vp, vp, i32, i32, i32, vp, vp, vp, vp], ctypes.c_int),
    "lmc_las_pf3_build_f32": ([vp, vp, i64, vp, vp, i32, i32, i32, vp, vp, vp, vp], ctypes.c_int),
    "lmc_scan_mark": ([vp, i64, vp, vp, i32, f64, f64, f64, f64, f64, vp, vp, vp, vp, vp], ctypes.c_int),
    "lmc_scan_recount": ([vp, i64, i32, vp, vp, vp], ctypes.c_int),
    "lmc_scan_emit": ([vp, i64, vp, vp, i32, f64, vp, vp, vp, vp, i32, vp, vp, vp], ctypes.c_int),
    "lmc_scan_emit_index": ([vp, i64, vp, vp, i32, f64, vp, vp, vp, vp, i32, vp, vp], ctypes.c_int),
    "lmc_voxel_workspace_bytes": ([i64], i64),
    "lmc_voxel_index_f64": ([vp, i64, vp, vp, vp, vp, vp, vp], ctypes.c_int),
    "lmc_voxel_index_f32": ([vp, i64, vp, vp, vp, vp, vp, vp], ctypes.c_int),
    "lmc_voxel_reduce_f64": ([vp, i64, vp, vp, vp, i64, vp, vp, vp, vp], ctypes.c_int),
    "lmc_voxel_reduce_f32": ([vp, i64, vp, vp, vp, i64, vp, vp, vp, vp], ctypes.c_int),
    "lmc_map_workspace_bytes": ([i64], i64),
    "lmc_map_build": ([vp, vp], ctypes.c_int),
    "lmc_map_nearest_f64": ([vp, i64, vp, f64, vp, vp, vp, vp], ctypes.c_int),
    "lmc_map_nearest_f32": ([vp, i64, vp, f64, vp, vp, vp, vp], ctypes.c_int),
    "lmc_register_workspace_bytes": ([i64, i32], i64),
    "lmc_register_frames_f64": ([vp, i64, vp, i32, vp, vp, f64, i32, f64, f64, vp, vp, vp, vp, vp, vp, vp, vp], ctypes.c_int),
    "lmc_register_frames_f32": ([vp, i64, vp, i32, vp, vp, f64, i32, f64, f64, vp, vp, vp, vp, vp, vp, vp, vp], ctypes.c_int),
    "lmc_map_normals": ([vp, f64, i32, vp, vp, vp], ctypes.c_int),
    "lmc_register_plane_workspace_bytes": ([i64, i32], i64),
    "lmc_register_frames_plane_f64": ([vp, i64, vp, i32, vp, vp, vp, f64, f64, i32, f64, f64, vp, vp, vp, vp, vp, vp, vp, vp], ctypes.c_int),
    "lmc_register_frames_plane_f32": ([vp, i64, vp, i32, vp, vp, vp, f64, f64, i32, f64, f64, vp, vp, vp, vp, vp, vp, vp, vp], ctypes.c_int),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib() -> ctypes.CDLL:
    """Load liblmc_b200.so (built in-tree by __graft_entry__.build() / _build.build_library())."""
    global _lib
    if _lib is None:
        path = os.environ.get("LMC_B200_LIB", LIB_PATH)       # experiments: alternative builds of the same ABI
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -m livox_motion_compensation_sim_b200._build` "
                "(nvcc, sm_100a). There is no CPU fallback for this path.")
        L = ctypes.CDLL(path)
        for name, (args, res) in _SIGNATURES.items():
            fn = getattr(L, name)           # AttributeError if the library does not export it
            fn.argtypes, fn.restype = args, res
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != OK:
        raise LmcError(rc, lib().lmc_last_error().decode(errors="replace"))


def set_path(path: int) -> None:
    check(lib().lmc_set_path(int(path)))


def get_path() -> int:
    return int(lib().lmc_get_path())
