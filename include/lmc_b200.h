/*
 * lmc_b200.h -- C ABI of liblmc_b200.so: the B200 (sm_100a) motion-compensation hot path of
 * manishborikar92/livox-motion-compensation-sim.
 *
 * The reference is pure Python and has NO plugin / FFI layer (SURVEY.md section 8b): its boundary
 * for this path is the Python method surface.  Every entry point below therefore cites the
 * reference *method* it replaces; the ctypes binding a maintainer would add on the reference side
 * is shown in INTEGRATION.md.
 *
 *   LMC = lidar_motion_compensation.py        CS = livox_mid70_complete_simulator.py
 *
 * Conventions
 *   - every data pointer is a caller-owned DEVICE pointer (e.g. torch.Tensor.data_ptr()) unless
 *     the parameter name ends in _host; the library never allocates or frees caller-visible memory.
 *     ("Device pointer" = any address the GPU can dereference: the UVA address of a pinned host buffer
 *     works as well -- the kernel then reads / writes it across PCIe, INTEGRATION.md section 8.)
 *     The lmc_host_* functions are the exception: HOST pointers only, no device work, synchronous
 *     (the host side of the boundary: frame-list packing and the scanner's NumPy noise stream)
 *   - point arrays, record arrays and LAS arrays must be 32-byte aligned at index 0
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all calls are
 *     asynchronous and stream-ordered, re-entrant across streams and devices
 *   - return value: LMC_OK or a negative LMC_ERR_*; lmc_last_error() gives a thread-local message.
 *     No exceptions cross the ABI, and there is no CPU fallback: without a usable sm_100 device the
 *     calls fail with LMC_ERR_CUDA.
 *   - frames are CSR rows: frame f owns points [frame_off[f], frame_off[f+1]) of the flat arrays,
 *     frame-major, which is exactly np.vstack order (LMC:888).  Empty frames are zero-length rows.
 *   - [p_begin, p_end) selects the slice of points this call processes (a rank's shard of the
 *     merged cloud); pass 0, n_points for everything.  Results are written at the same global
 *     indices, so frame-sharded ranks fill disjoint slices of one merged buffer.
 */
#ifndef LMC_B200_H
#define LMC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LMC_VERSION           100      /* 0.1.0 */

#define LMC_OK                  0
#define LMC_ERR_INVALID        -1      /* bad argument (NULL, negative size, bad enum)            */
#define LMC_ERR_ALIGN          -2      /* pointer not 32-byte aligned                             */
#define LMC_ERR_CUDA           -3      /* CUDA runtime error / no sm_100 device                   */

/* bits OR-ed into *status by the quantising epilogues (where the reference would raise) */
#define LMC_FLAG_NAN            1u     /* int(nan): ValueError in LMC:257 / CS:368                */
#define LMC_FLAG_OVERFLOW       2u     /* struct.pack('<i') / laspy OverflowError / u8 range      */

/* lvx_mode */
#define LMC_LVX_TYPE2_OF_INPUT  0      /* LMC:252-272 on the RAW sensor-frame input point (LMC:977):
                                          trunc(clip(x*1000, int32 range)), refl=trunc(clip(i*255,0,255)), tag 0 */
#define LMC_LVX2_OF_OUTPUT      1      /* CS:365-374 on the COMPENSATED output point:
                                          trunc(x*1000) (no clip), intensity and tag bytes copied */
/* las_intensity_mode */
#define LMC_LAS_INTENSITY_UNIT  0      /* LMC:961   (i * 65535).astype(uint16)                    */
#define LMC_LAS_INTENSITY_RAW   1      /* CS:1686   i.astype(uint16)                              */

/*
 * Optional fused export epilogues.  Any output pointer may be NULL (that export is skipped); a NULL
 * lmc_export* skips all of them.  All arrays are indexed by global point index.
 */
typedef struct lmc_export {
    uint8_t*  lvx14;              /* (n_points, 14) little-endian <iiiBB records                      */
    int32_t   lvx_mode;           /* LMC_LVX_*                                                        */
    const uint8_t* tag;           /* (n_points) tag byte for LMC_LVX2_OF_OUTPUT, NULL = 0             */
    int32_t*  las_x;              /* (n_points) LAS integer X = rint((x - offset) / scale)            */
    int32_t*  las_y;
    int32_t*  las_z;
    uint16_t* las_intensity;      /* (n_points)                                                       */
    int32_t   las_intensity_mode; /* LMC_LAS_INTENSITY_*                                              */
    double    las_scale[3];       /* laspy header default 0.01 (LMC:953), 0.001 set at CS:1679-1681   */
    double    las_offset[3];      /* 0                                                                */
    uint32_t* status;             /* device u32, OR of LMC_FLAG_*; NULL = not reported                */
    /* Merged-cloud assembly fused into the epilogue (SURVEY 8e): when n_peers > 0 the aligned cloud and
     * the LVX records are ALSO stored, at the same global point indices, into the other ranks' copies of
     * the merged buffers (peer-mapped device pointers, e.g. torch symmetric memory buffer_ptrs) -- the
     * all-gather happens over NVLink while the kernel computes.  A cross-rank barrier after the kernel
     * makes the remote writes visible.  LAS arrays are not mirrored. */
    int32_t   n_peers;            /* 0 .. LMC_MAX_PEERS                                              */
    void*     peer_out[7];        /* same layout as out_n4 (NULL entries are skipped)                 */
    uint8_t*  peer_lvx14[7];      /* same layout as lvx14                                             */
    /* The same assembly through the NVSwitch multicast mapping of the merged buffers (torch symmetric memory
     * `multicast_ptr`): when both are non-NULL (float4 layout, out + type-2 LVX records) every result of a full
     * tile leaves as ONE multimem.st that the switch replicates into every rank's copy -- this rank's included --
     * instead of a local store plus n_peers peer stores.  The peer pointers above must still be given: a
     * shard's ragged first / last tile uses them. */
    void*     mc_out;
    uint8_t*  mc_lvx14;
} lmc_export;
#define LMC_MAX_PEERS 7

int         lmc_version(void);
const char* lmc_last_error(void);
/* sm count / compute capability of the current device; fails unless it is sm_100 */
int         lmc_device_query(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
/* kernel path: 0 = direct (one tile per CTA, 256-bit LDG/STG), 1 = auto (default: persistent TMA
 * bulk-copy pipeline on inputs that fill the GPU, direct otherwise), 2 = TMA pipeline always */
int         lmc_set_path(int32_t path);
int         lmc_get_path(void);

/*
 * (a1) frame pose lookup, replaces the per-frame Python at LMC:802-812:
 *   idx_f = min(np.searchsorted(traj_t, frame_t[f]), n_t - 1)       ("hold-next", no interpolation)
 *   pose_Rt[f] = traj_Rt[idx_f]     (12 doubles: R row-major as SciPy builds it at LMC:774, then t)
 * pose_idx (optional, int32[n_frames]) receives idx_f.
 */
int lmc_pose_lookup_hold_next(const double* traj_t, int64_t n_t, const double* traj_Rt,
                              const double* frame_t, int32_t n_frames,
                              double* pose_Rt, int32_t* pose_idx, void* stream);

/*
 * (a2)+(a3) LiDARMotionSimulator.transform_pointcloud over all frames + merged-cloud assembly,
 * replaces LMC:772-776 called from LMC:826-832 and np.vstack at LMC:886-889.
 *   out[i, :3] = R_f @ pts[i, :3] + t_f ;  out[i, 3] = pts[i, 3]       (f = frame of point i)
 * float64 arithmetic in the reference's operation order: bit-exact for (n,4) f64 input.
 * _f32: same arithmetic on float4 points up-cast to f64 in registers, result rounded to f32.
 * `out` may be NULL when only exports are wanted.
 */
int lmc_align_rigid_f64(const double* pts_n4, const int64_t* frame_off, const double* pose_Rt,
                        double* out_n4, int64_t n_points, int32_t n_frames,
                        int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);
int lmc_align_rigid_f32(const float* pts_n4, const int64_t* frame_off, const double* pose_Rt,
                        float* out_n4, int64_t n_points, int32_t n_frames,
                        int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);

/*
 * (a6)-(a8) MotionCompensator.compensate_point_cloud, replaces CS:1435-1536 (per-point IMU bracket
 * search CS:1482-1516, gyro lerp, Rx(-a)Ry(-b)Rz(-c) CS:1518-1536).  Rotation only.
 *   _f64: pts (n,4) f64 [x y z intensity], ts int64 ns per point
 *   _f32: pts float4, ts_off uint32 ns offset from frame_start[f]
 * imu_ts int64[n_imu] sorted, imu_gyro f64 (n_imu,3).  n_imu == 0: points are copied (CS:1439).
 */
int lmc_deskew_gyro_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off,
                        const int64_t* frame_start, const int64_t* imu_ts, const double* imu_gyro,
                        int64_t n_imu, double* out_n4, int64_t n_points, int32_t n_frames,
                        int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);
int lmc_deskew_gyro_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off,
                        const int64_t* frame_start, const int64_t* imu_ts, const double* imu_gyro,
                        int64_t n_imu, float* out_n4, int64_t n_points, int32_t n_frames,
                        int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);

/*
 * (north_star subsystem 1) the pose-segment table lmc_deskew_slerp_* consume, built on the device from
 * the GPS/IMU pose samples: unit quaternions (x y z w, normalised here), positions and int64 ns times.
 * Row k (22 doubles) = [R_k (9) | pos_k (3) | unit axis of R_k^-1 R_{k+1} (3) | angle |
 * pos_{k+1} - pos_k (3) | 1/(t_{k+1} - t_k) | t_k bits | (t_{k+1} - t_k) bits]; the last row has angle 0.
 * Same definition as the host builder frames.slerp_segment_table (SciPy), which it replaces when the
 * pose stream arrives with the points (1.7 s on the host for a 1 h / 200 Hz stream, microseconds here);
 * the two agree to rounding (tests: table columns and the Mode C output built from either).
 */
int lmc_build_slerp_table(const double* sample_quat_xyzw, const double* sample_pos,
                          const int64_t* sample_ts, int64_t n_samples, double* seg_out, void* stream);

/*
 * Mode C: per-point pose-interp deskew (north_star; sketched without a body at
 * docs/Master Guide.md:339-367; no reference implementation -> parity unpinned).
 *   k = bracket(sample_ts, ts) ; alpha = (ts - t_k) * inv_dt_k      (inv_dt_k = 1/(t_{k+1} - t_k) from seg)
 *   out = SLERP(R_k, R_{k+1}, alpha) p + lerp(pos_k, pos_{k+1}, alpha)
 * seg: (n_samples, 22) f64 per-sample table [R_k(9) pos_k(3) axis_k(3) theta_k dpos_k(3) inv_dt_k
 *      t_k dt_k] -- the last two are raw int64 values (t_k, t_{k+1} - t_k) stored in double slots;
 *      n_samples must be < 2^31
 *      (built by the host wrapper, see livox_motion_compensation_sim_b200/frames.py).
 * hold_idx (optional int32[n_frames]): every point of frame f takes sample hold_idx[f], alpha = 0
 *      -> Mode A expressed in Mode C (bit-identical to lmc_align_rigid_* for frames of >= 2 points).
 *   _f64: ts int64 ns per point (frame_start unused, may be NULL)
 *   _f32: ts_off uint32 ns offsets from frame_start[f]
 */
int lmc_deskew_slerp_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off,
                         const int64_t* frame_start, const int64_t* sample_ts, const double* seg,
                         int64_t n_samples, const int32_t* hold_idx, double* out_n4,
                         int64_t n_points, int32_t n_frames,
                         int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);
int lmc_deskew_slerp_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off,
                         const int64_t* frame_start, const int64_t* sample_ts, const double* seg,
                         int64_t n_samples, const int32_t* hold_idx, float* out_n4,
                         int64_t n_points, int32_t n_frames,
                         int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);

/*
 * Pose at a time: Mode C's pose at each of n_query int64 ns times, with Mode C's bracket, end clamps and alpha
 * (definition: oracle/lmc_oracle_local.c::orc_slerp_pose_at).  pose_out (n_query, 12) f64 is laid out like lmc_align_rigid_*'s
 * pose_Rt: R(t) row-major, then pos(t).  lmc_align_rigid_* with these rows is Mode A at the interpolated pose.
 * 1 <= n_samples < 2^31; seg and pose_out 16-byte aligned.
 */
int lmc_slerp_pose_at(const int64_t* sample_ts, const double* seg, int64_t n_samples,
                      const int64_t* query_ts, int64_t n_query, double* pose_out, void* stream);

/*
 * Sensor-frame deskew: every point of frame f in the sensor frame of the frame's reference pose (R_r, x_r) = ref_pose[f]
 * (normally lmc_slerp_pose_at at the frame's start or end time), rotation and translation removed
 * (definition: oracle/lmc_oracle_local.c::orc_deskew_slerp_local_f64):
 *   w   = R(ts) p + (pos(ts) - x_r)       Mode C's pose at the point's time, the offset formed before the lerp
 *   out = R_r^T w ;  out[3] = p[3]
 * The world position is never rounded to the point layout, so map / UTM-scale positions cost no precision in the f32
 * layout.  Arguments, layouts, shards and exports as lmc_deskew_slerp_* (no hold_idx); ref_pose (n_frames, 12) f64,
 * 16-byte aligned, Mode A's row layout.  LMC_LVX2_OF_OUTPUT records are the second simulator's LVX2 points with
 * translation compensated.  Refused (LMC_ERR_INVALID, nothing written): n_peers > 0 or multicast pointers (a merged
 * cloud of points in per-frame sensor frames means nothing), ref_pose NULL, n_samples < 1 or >= 2^31.
 */
int lmc_deskew_slerp_local_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off,
                               const int64_t* frame_start, const int64_t* sample_ts, const double* seg,
                               int64_t n_samples, const double* ref_pose, double* out_n4,
                               int64_t n_points, int32_t n_frames,
                               int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);
int lmc_deskew_slerp_local_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off,
                               const int64_t* frame_start, const int64_t* sample_ts, const double* seg,
                               int64_t n_samples, const double* ref_pose, float* out_n4,
                               int64_t n_points, int32_t n_frames,
                               int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);

/*
 * Distortion, the exact inverse of Mode C: every world point W into the sensor frame of Mode C's pose at the point's own
 * time -- what a sensor moving along the sample table records of a static world
 * (definition: oracle/lmc_oracle_distort.c::orc_distort_slerp_f64):
 *   (k, alpha) = Mode C's bracket, end clamps and alpha at ts
 *   d   = (W - pos_k) - alpha dpos_k       the offset formed before the lerp: world-scale positions never enter the result
 *   out = rot_{-alpha theta_k}(R_k^T d) ;  out[3] = W[3]        (= R(ts)^T (W - pos(ts)))
 * lmc_deskew_slerp_* of the output gives W back.  Arguments, layouts, shards and exports as lmc_deskew_slerp_local_*
 * (no ref_pose); input world points, output raw sensor-frame points (LMC_LVX_TYPE2_OF_INPUT records are of the world
 * points, LMC_LVX2_OF_OUTPUT records of the raw ones).  Refused (LMC_ERR_INVALID, nothing written): n_peers > 0 or
 * multicast pointers, n_samples < 1 or >= 2^31.
 */
int lmc_distort_slerp_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off,
                          const int64_t* frame_start, const int64_t* sample_ts, const double* seg,
                          int64_t n_samples, double* out_n4,
                          int64_t n_points, int32_t n_frames,
                          int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);
int lmc_distort_slerp_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off,
                          const int64_t* frame_start, const int64_t* sample_ts, const double* seg,
                          int64_t n_samples, float* out_n4,
                          int64_t n_points, int32_t n_frames,
                          int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream);

/*
 * (a4)/(a5)/(a9)/(a10) stand-alone quantisers (no transform): LivoxLVXWriter._write_point_data_type2
 * LMC:252-272, the LVX2 packer CS:365-374 and the LAS integer packing behind LMC:957-961 /
 * CS:1683-1686.  `ex` selects outputs and modes exactly as in the fused calls; for lvx_mode both
 * values read the given points.
 */
int lmc_quantize_f64(const double* pts_n4, int64_t n_points, const lmc_export* ex, void* stream);
int lmc_quantize_f32(const float* pts_n4, int64_t n_points, const lmc_export* ex, void* stream);

/*
 * (SURVEY 8f N3) CoordinateTransformer.transform_points (CS:214-233): one 4x4 homogeneous matrix
 * (T_host: HOST pointer, 16 doubles row-major; the last row is not read) applied to every point,
 * the 4th column passing through.  `order` selects which of the reference's two summation orders is
 * reproduced bit for bit:
 *   LMC_HOMOG_BATCH   the call on an (n >= 2, 3) array: dgemm, fma(T3,1, fma(T2,z, fma(T1,y, T0*x)))
 *   LMC_HOMOG_SINGLE  the call on ONE point, which is how _transform_coordinates (CS:2107-2163) calls
 *                     it for every point of every frame: 4-term gemv, (T0*x + T2*z) + (T1*y + T3)
 */
#define LMC_HOMOG_BATCH  0
#define LMC_HOMOG_SINGLE 1
int lmc_transform_homog_f64(const double* pts_n4, const double* T_host, int32_t order,
                            double* out_n4, int64_t n_points, void* stream);
int lmc_transform_homog_f32(const float* pts_n4, const double* T_host, int32_t order,
                            float* out_n4, int64_t n_points, void* stream);

/*
 * (SURVEY 8f N1) LivoxLVXWriter.write_compatible_lvx, replaces LMC:58-250: the complete LVX v1.1 file
 * image -- 88-byte preamble, per frame a 24-byte header and ceil(n/96) packages of 22-byte header +
 * 96 x 14-byte records (tail zero-padded) -- built on the device from the RAW points (LMC:977), with
 * the record arithmetic of LMC:252-272.  frame_pos[f] = byte offset of frame f in the file
 * (frame_pos[0] = 88, frame_pos[n_frames] = file size = capacity of file_out), frame_time in seconds
 * (package timestamp = int(t * 1e9), LMC:177), frame_id = the reference's frame_id.
 * max_frame_points = max over frames of the point count (sizes the launch grid).
 */
int lmc_lvx_v11_build_f64(const double* pts_n4, const int64_t* frame_off, const int64_t* frame_pos,
                          const double* frame_time, const int64_t* frame_id, uint8_t* file_out,
                          int64_t n_points, int32_t n_frames, int64_t max_frame_points,
                          uint32_t* status, void* stream);
int lmc_lvx_v11_build_f32(const float* pts_n4, const int64_t* frame_off, const int64_t* frame_pos,
                          const double* frame_time, const int64_t* frame_id, uint8_t* file_out,
                          int64_t n_points, int32_t n_frames, int64_t max_frame_points,
                          uint32_t* status, void* stream);

/*
 * The same for frames [f_begin, f_end) only -- a rank's shard of the file (SURVEY 8e: every rank builds and writes its own
 * byte range, nothing is gathered).  shard_out[0] is file byte out_file_pos: 0 for the rank that owns frame 0 (its range
 * then starts with the 88-byte preamble), frame_pos[f_begin] otherwise; the shard holds
 * frame_pos[f_end] - out_file_pos bytes.  All arrays are the GLOBAL ones (frame headers carry absolute file offsets).
 * shard_out must be congruent to out_file_pos modulo 16 (the byte ranges are assembled at the file's 16-byte phase).
 */
int lmc_lvx_v11_build_range_f64(const double* pts_n4, const int64_t* frame_off, const int64_t* frame_pos,
                                const double* frame_time, const int64_t* frame_id, uint8_t* shard_out,
                                int64_t out_file_pos, int64_t n_points, int32_t n_frames, int32_t f_begin,
                                int32_t f_end, int64_t max_frame_points, uint32_t* status, void* stream);
int lmc_lvx_v11_build_range_f32(const float* pts_n4, const int64_t* frame_off, const int64_t* frame_pos,
                                const double* frame_time, const int64_t* frame_id, uint8_t* shard_out,
                                int64_t out_file_pos, int64_t n_points, int32_t n_frames, int32_t f_begin,
                                int32_t f_end, int64_t max_frame_points, uint32_t* status, void* stream);

/*
 * (SURVEY 8f N1, second half) the containers of the complete simulator's LivoxLVXWriter.write_lvx_file
 * (CS:245-374), built on the device from COMPENSATED points [x y z intensity] + optional tag bytes:
 *   LMC_LVXCS_LVX2    _write_lvx2 / _write_lvx3 (CS:269-293): per frame a 24-byte header {u32 index,
 *                     u64 timestamp, u32 count, 8 x 0}, one 21-byte package header (CS:354-363) and the
 *                     unpadded 14-byte records of CS:365-374 (int(v*1000) without clip, u8, u8)
 *   LMC_LVXCS_LEGACY  _write_lvx_legacy (CS:256-267, 308-321): per frame {u64 timestamp, u32 count} and
 *                     14-byte records {f32 x y z, u8 intensity, u8 tag}
 * prefix = the file's leading bytes, a HOST pointer (<= LMC_LVXCS_PREFIX_MAX bytes): file header +
 * private header / device block, which depend only on DeviceInfo and the frame count (CS:272-283,
 * 295-306, 323-341).  File size = prefix_len + H * n_frames + 14 * n_points with H =
 * LMC_LVXCS_LVX2_FRAME_BYTES | LMC_LVXCS_LEGACY_FRAME_BYTES.  frame_ts = the frames' 'timestamp' (ns).
 * Errors the reference raises from struct.pack become status bits: |int(v*1000)| beyond int32 or a
 * finite value beyond f32 range or an intensity outside 0..255 -> LMC_FLAG_OVERFLOW, NaN through
 * int() -> LMC_FLAG_NAN.
 */
#define LMC_LVXCS_LVX2   0
#define LMC_LVXCS_LEGACY 1
#define LMC_LVXCS_PREFIX_MAX 96
#define LMC_LVXCS_LVX2_FRAME_BYTES   45
#define LMC_LVXCS_LEGACY_FRAME_BYTES 12
int lmc_lvx_cs_build_f64(const double* pts_n4, const uint8_t* tag, const int64_t* frame_off,
                         const uint64_t* frame_ts, const uint8_t* prefix_host, int32_t prefix_len,
                         int32_t format, uint8_t* file_out, int64_t n_points, int32_t n_frames,
                         int64_t max_frame_points, uint32_t* status, void* stream);
int lmc_lvx_cs_build_f32(const float* pts_n4, const uint8_t* tag, const int64_t* frame_off,
                         const uint64_t* frame_ts, const uint8_t* prefix_host, int32_t prefix_len,
                         int32_t format, uint8_t* file_out, int64_t n_points, int32_t n_frames,
                         int64_t max_frame_points, uint32_t* status, void* stream);

/*
 * (SURVEY 8f N2) ASCII PCD point data, replaces the per-point Python loop of
 * LiDARMotionSimulator.save_pcd (LMC:946-947): for every row of the (n,4) array the line
 *     "%.6f %.6f %.6f %.6f\n"        (x y z intensity)
 * byte-identical to CPython / C printf (correctly rounded, round-half-even on the exact binary value;
 * "nan", "inf", "-inf" as Python prints them).  Lines have variable length, so it is a two-call
 * protocol: _size fills tile_off (int64[ceil(n / LMC_PCD_TILE) + 1], byte offset of every tile of
 * LMC_PCD_TILE points; the last entry is the total text size), the caller allocates text_out of that
 * size, _write produces the bytes.  |values| >= 9.2e12 set LMC_FLAG_OVERFLOW in *status.
 */
#define LMC_PCD_TILE 256
int lmc_pcd_ascii_size_f64(const double* pts_n4, int64_t n_points, int64_t* tile_off, void* stream);
int lmc_pcd_ascii_size_f32(const float* pts_n4, int64_t n_points, int64_t* tile_off, void* stream);
int lmc_pcd_ascii_write_f64(const double* pts_n4, int64_t n_points, const int64_t* tile_off,
                            uint8_t* text_out, uint32_t* status, void* stream);
int lmc_pcd_ascii_write_f32(const float* pts_n4, int64_t n_points, const int64_t* tile_off,
                            uint8_t* text_out, uint32_t* status, void* stream);

/*
 * Byte offsets of arbitrary rows inside the text _write produces (e.g. the frame boundaries of a frame-major
 * buffer): byte_off[q] = offset of the first byte of row rows[q] (rows[q] = n_points gives the total size).
 * One formatting pass then serves every per-frame file of save_results (LMC:870-884: raw_scans_pcd/frame_%04d.pcd,
 * aligned_scans_pcd/aligned_frame_%04d.pcd) and the merged files (LMC:893-899) as slices of the same text.
 * rows / byte_off are device arrays of n_rows entries; tile_off as filled by _size.
 */
int lmc_pcd_ascii_row_offsets_f64(const double* pts_n4, int64_t n_points, const int64_t* tile_off,
                                  const int64_t* rows, int32_t n_rows, int64_t* byte_off, void* stream);
int lmc_pcd_ascii_row_offsets_f32(const float* pts_n4, int64_t n_points, const int64_t* tile_off,
                                  const int64_t* rows, int32_t n_rows, int64_t* byte_off, void* stream);

/*
 * Host-side staging helpers (HOST pointers, synchronous, no device work).  The reference's interface is lists of
 * small per-frame arrays (results['raw_scans'][i]['points_local'], LMC:818-823; np.vstack at LMC:888): packing
 * them into one pinned frame-major buffer is memory-bound host work, split here over n_threads threads.
 *   lmc_host_gather: source i (src[i], dst_off[i+1] - dst_off[i] bytes) is copied to dst + dst_off[i]; dst_off has
 *                    n_src + 1 non-decreasing entries.
 *   lmc_host_copy:   plain copy of n_bytes.
 */
int lmc_host_gather(const void* const* src, const int64_t* dst_off, int64_t n_src, void* dst, int32_t n_threads);
int lmc_host_copy(void* dst, const void* src, int64_t n_bytes, int32_t n_threads);

/*
 * Host-side replay of np.random.normal(loc, scale, n) on NumPy's legacy global generator (RandomState: MT19937 +
 * polar Box-Muller) -- the stream scan_environment consumes for its range noise (LMC:767, seeded at LMC:288), which
 * a run has to consume exactly to reproduce the reference's raw scans.  mt_key (624 words), *mt_pos (0..624),
 * *has_gauss and *cached_gauss are the four fields of np.random.get_state() and are updated in place, so
 * np.random.set_state() afterwards leaves the generator where NumPy itself would have left it.  The word stream and
 * the rejection loop are sequential; the sqrt / log part is spread over n_threads.  Bit-identical to NumPy (same
 * libm calls; tests/test_host.py).
 */
int lmc_host_legacy_normal(uint32_t* mt_key, int32_t* mt_pos, int32_t* has_gauss, double* cached_gauss,
                           double loc, double scale, int64_t n, double* out, int32_t n_threads);

/*
 * (SURVEY 8f N2) the complete simulator's text exports, replaces the per-row Python loops of
 * DataExporter._export_pcd (CS:1663-1664, '%.6f %.6f %.6f %.0f %.0f\n' over [x y z intensity timestamp]),
 * _export_xyz (CS:1703, np.savetxt '%.6f' x 3) and the body of _export_csv (CS:1711-1712, pandas
 * float_format '%.6f', ',' separated): every row of a (n_rows, row_stride) array becomes
 *     "%.{decimals[0]}f" sep "%.{decimals[1]}f" sep ... "\n"     over the columns col_host[0..n_cols)
 * byte-identical to C printf / CPython (correctly rounded, half-even on the exact binary value).
 * col_host / decimals_host are HOST arrays of n_cols <= LMC_TEXT_MAX_COLS entries, decimals 0..9.  Same two-call
 * protocol and tile size as the PCD writer.  |v| >= 2^64 sets LMC_FLAG_OVERFLOW.
 */
#define LMC_TEXT_MAX_COLS 6
int lmc_text_rows_size_f64(const double* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols,
                           const int32_t* col_host, const int32_t* decimals_host, int32_t sep,
                           int64_t* tile_off, void* stream);
int lmc_text_rows_size_f32(const float* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols,
                           const int32_t* col_host, const int32_t* decimals_host, int32_t sep,
                           int64_t* tile_off, void* stream);
int lmc_text_rows_write_f64(const double* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols,
                            const int32_t* col_host, const int32_t* decimals_host, int32_t sep,
                            const int64_t* tile_off, uint8_t* text_out, uint32_t* status, void* stream);
int lmc_text_rows_write_f32(const float* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols,
                            const int32_t* col_host, const int32_t* decimals_host, int32_t sep,
                            const int64_t* tile_off, uint8_t* text_out, uint32_t* status, void* stream);

/*
 * (SURVEY 8f N2) A complete LAS 1.2 / point-format-3 file image -- what save_las (LMC:950-963) and
 * _export_las (CS:1671-1698) get from laspy -- built on the device: 227-byte public header (min / max
 * reduced on the GPU) + 34-byte records.  PARITY UNPINNED (laspy absent): the file follows the LAS 1.2
 * specification; X/Y/Z = rint((v - offset) / scale), intensity per las_intensity_mode, gps_time from
 * the optional array (CS:1689) else 0, every other field 0.  file_out holds LMC_LAS_HEADER_BYTES +
 * LMC_LAS_RECORD_BYTES * n_points bytes; minmax_scratch is 6 device int32 (any contents).
 */
#define LMC_LAS_HEADER_BYTES 227
#define LMC_LAS_RECORD_BYTES 34
int lmc_las_pf3_build_f64(const double* pts_n4, const double* gps_time, int64_t n_points,
                          const double scale[3], const double offset[3], int32_t las_intensity_mode,
                          int32_t year, int32_t day_of_year, uint8_t* file_out, int32_t* minmax_scratch,
                          uint32_t* status, void* stream);
int lmc_las_pf3_build_f32(const float* pts_n4, const double* gps_time, int64_t n_points,
                          const double scale[3], const double offset[3], int32_t las_intensity_mode,
                          int32_t year, int32_t day_of_year, uint8_t* file_out, int32_t* minmax_scratch,
                          uint32_t* status, void* stream);

/*
 * The same in two parts, for frame-sharded ranks (SURVEY 8e): lmc_las_pf3_records_* writes the records of points
 * [p_begin, p_end) into shard_out, where shard_out[0] is file byte out_file_pos (0 for the rank that also holds the
 * header, LMC_LAS_HEADER_BYTES + LMC_LAS_RECORD_BYTES * p_begin otherwise), and leaves the shard's integer extremes
 * {minX, maxX, minY, maxY, minZ, maxZ} in minmax (6 device int32).  After the ranks have min / max-reduced those six
 * integers, lmc_las_pf3_header builds the 227-byte header of the n_points-record file from them.
 * shard_out must be congruent to out_file_pos modulo 16.
 */
int lmc_las_pf3_records_f64(const double* pts_n4, const double* gps_time, int64_t n_points, int64_t p_begin, int64_t p_end,
                            const double scale[3], const double offset[3], int32_t las_intensity_mode,
                            uint8_t* shard_out, int64_t out_file_pos, int32_t* minmax, uint32_t* status, void* stream);
int lmc_las_pf3_records_f32(const float* pts_n4, const double* gps_time, int64_t n_points, int64_t p_begin, int64_t p_end,
                            const double scale[3], const double offset[3], int32_t las_intensity_mode,
                            uint8_t* shard_out, int64_t out_file_pos, int32_t* minmax, uint32_t* status, void* stream);
int lmc_las_pf3_header(int64_t n_points, const double scale[3], const double offset[3], int32_t year, int32_t day_of_year,
                       const int32_t* minmax, uint8_t* header_out, void* stream);

/*
 * (SURVEY 8f N4) LiDARMotionSimulator.scan_environment, replaces LMC:701-770 for every frame of a run at
 * once: range cull (d2 <= range_max^2), world->sensor rotation R_f^T (env - pos_f), FOV cull, order-
 * preserving compaction, systematic subsample to max_points.  Two calls, because the reference draws its
 * noise from the seeded global NumPy RNG sized by each frame's point count (LMC:765-768):
 *   lmc_scan_mark  -> flags (n_frames x n_env bytes: bit 0 visible, bit 1 UNCERTAIN), tile_off
 *                     (n_frames x (ceil(n_env/LMC_SCAN_TILE)+1) int32 scratch), n_visible[f] and
 *                     *n_uncertain.  A point is uncertain when its |azimuth| or |elevation| lies within
 *                     edge_eps_deg of the FOV limit: device atan2 / asin may differ from the host libm
 *                     by a few ulp there.  When *n_uncertain > 0 the caller re-decides those points with
 *                     the reference's NumPy expression (LMC:735-745), writes 0 / 1 into their flags and
 *                     calls lmc_scan_recount, so every decision is the reference's;
 *   (host: kept[f] = n_visible[f] if <= max_points else min(ceil(n / (n // max_points)), max_points);
 *          frame_off = cumsum(kept); noise = np.random.normal(0, std, (sum kept, 3)) or NULL)
 *   lmc_scan_emit  -> raw_out (sum kept, 4): rotated xyz (+ noise) and the environment intensity,
 *                     frame-major, ready for lmc_align_rigid_f64.
 *   lmc_scan_emit_index -> env_idx_out (sum kept) int64: the environment row of every point lmc_scan_emit would emit,
 *                     in its slot (same compaction and subsample), for a caller that observes the points from other
 *                     poses (lmc_distort_slerp_f64: each point from the pose at its own time).
 * pos_f3 / R_f9: per-frame sensor position and SciPy rotation matrix (row-major) of the sensor pose.
 * n_env <= LMC_SCAN_MAX_ENV: per-frame counts, ranks and tile_off are int32, so all four calls refuse a larger
 * environment with LMC_ERR_INVALID before they write anything.
 */
#define LMC_SCAN_TILE 256
#define LMC_SCAN_MAX_ENV 2147483647LL
int lmc_scan_mark(const double* env_m4, int64_t n_env, const double* pos_f3, const double* R_f9, int32_t n_frames,
                  double range_max_sq, double fov_h_half_deg, double fov_v_half_deg, double range_min,
                  double edge_eps_deg, uint8_t* flags, int32_t* tile_off, int32_t* n_visible,
                  int32_t* n_uncertain, void* stream);
int lmc_scan_recount(const uint8_t* flags, int64_t n_env, int32_t n_frames, int32_t* tile_off,
                     int32_t* n_visible, void* stream);
int lmc_scan_emit(const double* env_m4, int64_t n_env, const double* pos_f3, const double* R_f9, int32_t n_frames,
                  double range_max_sq, const uint8_t* flags, const int32_t* tile_off, const int32_t* n_visible,
                  const int64_t* frame_off, int32_t max_points, const double* noise_n3, double* raw_out_n4,
                  void* stream);
int lmc_scan_emit_index(const double* env_m4, int64_t n_env, const double* pos_f3, const double* R_f9, int32_t n_frames,
                        double range_max_sq, const uint8_t* flags, const int32_t* tile_off, const int32_t* n_visible,
                        const int64_t* frame_off, int32_t max_points, int64_t* env_idx_out, void* stream);

/*
 * Voxel-grid map of an (n,4) cloud [x y z intensity]: one centroid and one point count per occupied voxel
 * (definition: oracle/lmc_oracle_voxel.py).  leaf[3] > 0 and origin[3] are finite HOST values; all arithmetic is f64
 * with explicit rounding, f32 points widened exactly.  Per point and axis:
 *   u = (p - o) / L ; k = floor(u) in [-2^20, 2^20) ; q = min(trunc((u - k) 2^32), 2^32 - 1) ; q_I = rint(I 2^24), |I| < 256
 * A point with a non-finite value is dropped with LMC_FLAG_NAN, one with k out of range or |I| >= 256 with
 * LMC_FLAG_OVERFLOW.  Per voxel, with n points and the int64 sums S of q and q_I:
 *   centroid = o + (k + (S / n) 2^-32) L ; intensity = (S_I / n) 2^-24      (every operation rounded to nearest;
 *                                                                            the f32 layout rounds once at the end)
 * The sums are integers, so the map is bit-identical under any thread schedule and any permutation of the input.
 * Voxels are ranked by their first point (smallest point index): a frame-major cloud's map grows frame by frame.
 * Two calls; the caller owns every buffer and reads V in between:
 *   lmc_voxel_workspace_bytes(n)  bytes of scratch (a hash table of the power of two >= 2n slots, 16 bytes a slot, and
 *                                 52 bytes a point); a negative LMC_ERR_* for n outside 0 .. 2^31 - 1
 *   lmc_voxel_index_*             keys, table, ranks; V -> *n_voxels_dev (device int64), flags OR-ed into *status
 *   lmc_voxel_reduce_*            out_n4 (V,4) centroids in the input's layout, counts int32[V], and, when point_voxel is
 *                                 not NULL, int32[n] rank of every point's voxel (-1 for a dropped point)
 * The same points, leaf, origin and workspace go to both calls.  Refused with LMC_ERR_INVALID before anything is
 * written: n < 0 or n >= 2^31, a leaf that is not finite or <= 0, an origin that is not finite, a NULL required
 * buffer, n_voxels outside 0 .. n.  Points, workspace and outputs must be 32-byte aligned (LMC_ERR_ALIGN).
 */
int64_t lmc_voxel_workspace_bytes(int64_t n_points);
int lmc_voxel_index_f64(const double* pts_n4, int64_t n_points, const double leaf[3], const double origin[3],
                        void* workspace, int64_t* n_voxels_dev, uint32_t* status, void* stream);
int lmc_voxel_index_f32(const float* pts_n4, int64_t n_points, const double leaf[3], const double origin[3],
                        void* workspace, int64_t* n_voxels_dev, uint32_t* status, void* stream);
int lmc_voxel_reduce_f64(const double* pts_n4, int64_t n_points, const double leaf[3], const double origin[3],
                         void* workspace, int64_t n_voxels, double* out_n4, int32_t* counts, int32_t* point_voxel,
                         void* stream);
int lmc_voxel_reduce_f32(const float* pts_n4, int64_t n_points, const double leaf[3], const double origin[3],
                         void* workspace, int64_t n_voxels, float* out_n4, int32_t* counts, int32_t* point_voxel,
                         void* stream);

/*
 * A prior point map on the device, exact fixed-radius nearest neighbours in it, and per-frame pose refinement against
 * it (definition: oracle/lmc_oracle_register.py).  The map is the voxel map's grid (leaf, origin, keys: the same f64
 * expressions) over its points: rows sorted by voxel rank (f64, the original row index beside each), CSR voxel
 * offsets, and a lookup table key -> rank (open addressing, the power of two >= 2V slots).  The caller builds the
 * first three from lmc_voxel_index_* / lmc_voxel_reduce_* (ranks, counts, point_voxel) and a stable sort, then fills
 * the table with lmc_map_build.  Every buffer is device memory and 32-byte aligned (LMC_ERR_ALIGN).
 *
 * Nearest (lmc_map_nearest_*): for a query w, its cell k = floor((w - origin) / leaf) and the 27 cells around it;
 * d = w - m and d2 = (dx dx + dy dy) + dz dz, every operation rounded to nearest (no contraction); accepted when
 * d2 <= r2 with r2 = max_dist^2 rounded once on the host; the result is the minimum over (d2, original index), so equal
 * distances go to the smaller index.  max_dist <= min(leaf), so the 27 cells cover the ball.  A query with a
 * non-finite coordinate or whose cell is outside the key range has no match (index -1, d2 = +inf); a non-finite query
 * sets LMC_FLAG_NAN in *status.
 *
 * Register (lmc_register_frames_*): frame f's points p (sensor frame, rows frame_off[f] .. frame_off[f+1]) and its
 * pose [R | t] (pose_Rt rows, align_rigid's layout).  Each of `iters` iterations, for every frame not yet done:
 * a = R p, w = a + t, its nearest map point q as above, and over the inliers r = w - q the 17 sums n, Sa, S aa^T,
 * Sr, S a x r, S |r|^2; then H = [[n I, -[Sa]x], [[Sa]x, S|a|^2 I - S aa^T]], g = [Sr; S a x r], delta = [tau; phi]
 * = -H^-1 g by Cholesky, t <- t + tau, R <- Exp(phi) R (about the sensor position).  A frame with n < 6 or a Cholesky
 * pivot <= 1e-12 trace(H) is DEGENERATE and keeps its pose from then on; one with |tau| <= tol_t and |phi| <= tol_r
 * (after applying that update) is CONVERGED and stops.  Per frame: inliers (n) and rms_m (sqrt(S|r|^2 / n), NaN for
 * n = 0) of its last iteration, the iterations it ran, flags.  No float atomics: results are bit-identical run to run
 * (they depend on the order of the points, which fixes the summation order).
 *
 * Refused with LMC_ERR_INVALID before anything is written: NULL required buffers, negative sizes, more than 2^31 - 1
 * points or map points, n_voxels outside 0 .. n_map_points, a leaf that is not finite and > 0 or an origin that is not
 * finite, max_dist not finite and > 0 or > min(leaf), iters < 1, tol_t / tol_r not finite and >= 0, n_frames < 1 with
 * points present.
 */
#define LMC_REG_CONVERGED       1
#define LMC_REG_DEGENERATE      2

typedef struct lmc_point_map {
    const double*  pts_m4;        /* (n_points, 4) f64 rows sorted by voxel rank                      */
    const int64_t* index;         /* (n_points) original row of each sorted row                       */
    const int64_t* vox_off;       /* (n_voxels + 1) CSR offsets of the voxels' rows                    */
    void*          table;         /* lmc_map_workspace_bytes(n_voxels) bytes: keys u64[cap] | rank u32 */
    int64_t        n_points;
    int64_t        n_voxels;
    double         leaf[3];       /* host values, as the voxel map                                     */
    double         origin[3];
} lmc_point_map;

int64_t lmc_map_workspace_bytes(int64_t n_voxels);
int lmc_map_build(const lmc_point_map* map, void* stream);          /* fills map->table */
int lmc_map_nearest_f64(const double* pts_n4, int64_t n_points, const lmc_point_map* map, double max_dist,
                        int64_t* index_out, double* d2_out, uint32_t* status, void* stream);
int lmc_map_nearest_f32(const float* pts_n4, int64_t n_points, const lmc_point_map* map, double max_dist,
                        int64_t* index_out, double* d2_out, uint32_t* status, void* stream);
int64_t lmc_register_workspace_bytes(int64_t n_points, int32_t n_frames);
int lmc_register_frames_f64(const double* pts_n4, int64_t n_points, const int64_t* frame_off, int32_t n_frames,
                            const double* pose_Rt, const lmc_point_map* map, double max_dist, int32_t iters, double tol_t,
                            double tol_r, void* workspace, double* pose_out, int32_t* inliers, double* rms_m,
                            int32_t* iterations, int32_t* flags, uint32_t* status, void* stream);
int lmc_register_frames_f32(const float* pts_n4, int64_t n_points, const int64_t* frame_off, int32_t n_frames,
                            const double* pose_Rt, const lmc_point_map* map, double max_dist, int32_t iters, double tol_t,
                            double tol_r, void* workspace, double* pose_out, int32_t* inliers, double* rms_m,
                            int32_t* iterations, int32_t* flags, uint32_t* status, void* stream);

/*
 * Normals of a point map (lmc_map_normals; definition: oracle/lmc_oracle_plane.py), one row per map row in the map's
 * sorted row order.  The neighbours of row p are every map row m with d2 <= r2 (r2 = radius^2 rounded once, d2 as in
 * lmc_map_nearest, the row itself included), visited in a fixed order: the 27 cells in dz, dy, dx order, then the
 * rows of each cell in sorted order.  With d = m - p (formed first, so map-scale coordinates never enter a sum), the
 * sequential sums S d and S dd^T give mu = S d / n and C = S dd^T / n - mu mu^T.  C is diagonalised by cyclic Jacobi
 * rotations in the pair order (0,1), (0,2), (1,2), a rotation skipped when its off-diagonal entry is exactly 0, until
 * a sweep leaves every off-diagonal at 0 (at most 32 sweeps).  Every operation is an IEEE-rounded + - x / sqrt, so
 * the result is bit-identical to its NumPy restatement.  The eigenvalues are sorted ascending (ties in index order) and clamped at 0; the row is
 * (nx, ny, nz, planarity): the unit eigenvector of lambda_min with its largest-magnitude component positive (the first
 * on a tie), and planarity = (lambda_mid - lambda_min) / lambda_max (about 1 on a plane, about 0 on a line or a blob).
 * A row with fewer than min_neighbours neighbours or lambda_max = 0 is (NaN, NaN, NaN, 0).  neighbours (may be NULL):
 * each row's neighbour count.  Refused with LMC_ERR_INVALID before anything is written: everything lmc_map_build
 * refuses, radius not finite and > 0 or > min(leaf), min_neighbours < 3, NULL normals for a map with points.
 *
 * Point-to-plane registration (lmc_register_frames_plane_*): lmc_register_frames_*'s iteration with the residual along
 * the nearest map row's normal.  A point is an inlier when its nearest map row q (within max_dist) has planarity >=
 * min_planarity; then e = (nx rx + ny ry) + nz rz with r = w - q, J = [n; a x n], and the 29 sums n, H = S J J^T,
 * g = S J e, S e^2 give delta = -H^-1 g.  Degenerate, converged, the update and the outputs are as point-to-point;
 * rms_m is the rms plane distance.  A frame that sees planes of one orientation only (ground alone) is DEGENERATE and
 * keeps its pose.  Refused as lmc_register_frames_*, and also for min_planarity outside (0, 1] or NULL normals for a
 * map with points.  The workspace is lmc_register_plane_workspace_bytes(n_points, n_frames).
 */
int lmc_map_normals(const lmc_point_map* map, double radius, int32_t min_neighbours, double* normals_m4, int32_t* neighbours,
                    void* stream);
int64_t lmc_register_plane_workspace_bytes(int64_t n_points, int32_t n_frames);
int lmc_register_frames_plane_f64(const double* pts_n4, int64_t n_points, const int64_t* frame_off, int32_t n_frames,
                                  const double* pose_Rt, const lmc_point_map* map, const double* normals_m4, double max_dist,
                                  double min_planarity, int32_t iters, double tol_t, double tol_r, void* workspace,
                                  double* pose_out, int32_t* inliers, double* rms_m, int32_t* iterations, int32_t* flags,
                                  uint32_t* status, void* stream);
int lmc_register_frames_plane_f32(const float* pts_n4, int64_t n_points, const int64_t* frame_off, int32_t n_frames,
                                  const double* pose_Rt, const lmc_point_map* map, const double* normals_m4, double max_dist,
                                  double min_planarity, int32_t iters, double tol_t, double tol_r, void* workspace,
                                  double* pose_out, int32_t* inliers, double* rms_m, int32_t* iterations, int32_t* flags,
                                  uint32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LMC_B200_H */
