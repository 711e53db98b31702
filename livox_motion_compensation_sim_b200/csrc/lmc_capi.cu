// lmc_capi.cu -- the extern "C" boundary declared in include/lmc_b200.h.
// Plain pointers and sizes in, int status out; no exceptions, no allocation of caller-visible
// memory, no CPU fallback (every call needs an sm_100 device).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>
#include "lmc_device.cuh"

namespace lmc {
cudaError_t launch_direct(bool f64, int mode, const Params& P, cudaStream_t st);
cudaError_t launch_stream(bool f64, int mode, const Params& P, const Plan& pl, int dev, cudaStream_t st);
cudaError_t launch_pose_lookup(const double*, int64_t, const double*, const double*, int32_t, double*, int32_t*, cudaStream_t);
cudaError_t launch_pcd_size(bool f64, const void* pts, int64_t n, int64_t* tile_off, cudaStream_t st);
cudaError_t launch_pcd_write(bool f64, const void* pts, int64_t n, const int64_t* tile_off, uint8_t* out, uint32_t* status, cudaStream_t st);
cudaError_t launch_pcd_row_off(bool f64, const void* pts, int64_t n, const int64_t* tile_off, const int64_t* rows, int32_t n_rows,
                               int64_t* byte_off, cudaStream_t st);
cudaError_t launch_scan_mark(const double* env, int64_t M, const double* pos, const double* R, int32_t F, double rmax2, double fh, double fv,
                             double rmin, double edge_eps, uint8_t* flags, int32_t* tile_off, int32_t* n_visible, int32_t* n_uncertain, cudaStream_t st);
cudaError_t launch_scan_recount(const uint8_t* flags, int64_t M, int32_t F, int32_t* tile_off, int32_t* n_visible, cudaStream_t st);
cudaError_t launch_scan_emit(const double* env, int64_t M, const double* pos, const double* R, int32_t F, double rmax2, const uint8_t* flags,
                             const int32_t* tile_off, const int32_t* n_visible, const int64_t* frame_off, int32_t max_points,
                             const double* noise, double* out, int64_t* idx_out, cudaStream_t st);
cudaError_t launch_las_pf3(bool f64, const LasParams& L, int parts, cudaStream_t st);
cudaError_t launch_lvx_v11(bool f64, const void* pts, const int64_t* frame_off, const int64_t* frame_pos, const double* frame_time,
                           const int64_t* frame_id, uint8_t* out, int32_t n_frames, int32_t f_begin, int32_t f_end, int64_t max_frame_points,
                           uint32_t* status, cudaStream_t st);
cudaError_t launch_slerp_table(const double* quat, const double* pos, const int64_t* ts, int64_t S, double* seg, cudaStream_t st);
cudaError_t launch_slerp_pose_at(const int64_t* sample_ts, const double* seg, int64_t S, const int64_t* query_ts, int64_t n_query,
                                 double* pose, cudaStream_t st);
cudaError_t launch_homog(bool f64, const void* in, const double* T_host, int32_t order, void* out, int64_t n, cudaStream_t st);
cudaError_t launch_text_size(bool f64, const void* rows, int64_t n, int32_t n_cols, int32_t row_stride, const int32_t* col, const int32_t* dec,
                             uint8_t sep, int64_t* tile_off, cudaStream_t st);
cudaError_t launch_text_write(bool f64, const void* rows, int64_t n, int32_t n_cols, int32_t row_stride, const int32_t* col, const int32_t* dec,
                              uint8_t sep, const int64_t* tile_off, uint8_t* out, uint32_t* status, cudaStream_t st);
cudaError_t launch_lvx_cs(bool f64, const void* pts, const uint8_t* tag, const int64_t* frame_off, const uint64_t* frame_ts,
                          const uint8_t* prefix_host, int32_t prefix_len, int32_t format, uint8_t* out, int32_t n_frames,
                          int64_t max_frame_points, uint32_t* status, cudaStream_t st);
size_t voxel_workspace_bytes(int64_t n);
cudaError_t launch_voxel_index(bool f64, const void* pts, int64_t n, const double* leaf, const double* origin, void* ws,
                               int64_t* n_voxels, uint32_t* status, cudaStream_t st);
cudaError_t launch_voxel_reduce(bool f64, const void* pts, int64_t n, const double* leaf, const double* origin, void* ws,
                                int64_t V, void* out, int32_t* counts, int32_t* point_voxel, cudaStream_t st);
size_t map_table_bytes(int64_t V);
size_t register_workspace_bytes(int64_t n, int64_t F);
int64_t register_max_chunks(int64_t n, int64_t F);
cudaError_t launch_map_build(const double* pts, const int64_t* vox_off, int64_t V, const double* leaf, const double* origin,
                             void* table, cudaStream_t st);
cudaError_t launch_map_nearest(bool f64, const void* q, int64_t n, const double* pts, const int64_t* idx, const int64_t* vox_off,
                               const void* table, int64_t V, const double* leaf, const double* origin, double r2,
                               int64_t* idx_out, double* d2_out, uint32_t* status, cudaStream_t st);
cudaError_t launch_register_frames(bool f64, const void* q, int64_t n, const int64_t* frame_off, int64_t F, const double* pose_in,
                                   const double* pts, const int64_t* idx, const int64_t* vox_off, const void* table, int64_t V,
                                   const double* leaf, const double* origin, double r2, int32_t iters, double tol_t, double tol_r,
                                   void* ws, double* pose_out, int32_t* inliers, double* rms, int32_t* iterations, int32_t* flags,
                                   uint32_t* status, cudaStream_t st);
}

namespace {

thread_local char g_err[512] = "";
std::atomic<int> g_path{1};                        // 0 = direct, 1 = auto (TMA pipeline on large inputs), 2 = TMA always

int fail(int code, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    return fail(LMC_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}
bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }
// one point row: 32 bytes (f64) or 16 bytes (float4) -- what the row-at-a-time kernels (text writers) need, so that any
// row slice of a frame-major buffer (a rank's shard) can be passed as it is
bool aligned_row(const void* p, bool f64) { return (reinterpret_cast<uintptr_t>(p) & (f64 ? 31u : 15u)) == 0; }

// The device this thread last checked: sm_100 (the kernels are built for sm_100a only and refuse anything else loudly,
// no fallback path exists), and its SM count, which sizes the persistent grid of the streaming kernels.
struct DeviceRecord { int dev = -1, sm_count = 0; };
thread_local DeviceRecord g_dev;

int check_device() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
    if (dev == g_dev.dev) return LMC_OK;
    int major = 0, sms = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
    if (major != 10) return fail(LMC_ERR_CUDA, "device %d is sm_%d0; liblmc_b200 is built for sm_100a only", dev, major);
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
    g_dev = { dev, sms };
    return LMC_OK;
}

int fill_export(lmc::Params& P, const lmc_export* ex) {
    P.lvx14 = nullptr; P.tag = nullptr; P.las_x = P.las_y = P.las_z = nullptr; P.las_int = nullptr; P.status = nullptr;
    P.lvx_mode = 0; P.las_int_mode = 0; P.n_peers = 0; P.mc_out = nullptr; P.mc_lvx = nullptr;
    for (int r = 0; r < LMC_MAX_PEERS; ++r) { P.peer_out[r] = nullptr; P.peer_lvx[r] = nullptr; }
    for (int c = 0; c < 3; ++c) { P.las_scale[c] = 0.01; P.las_rcp[c] = 1.0 / 0.01; P.las_off[c] = 0.0; }
    if (!ex) return LMC_OK;
    if (ex->lvx_mode != LMC_LVX_TYPE2_OF_INPUT && ex->lvx_mode != LMC_LVX2_OF_OUTPUT) return fail(LMC_ERR_INVALID, "bad lvx_mode %d", ex->lvx_mode);
    if (ex->las_intensity_mode != LMC_LAS_INTENSITY_UNIT && ex->las_intensity_mode != LMC_LAS_INTENSITY_RAW)
        return fail(LMC_ERR_INVALID, "bad las_intensity_mode %d", ex->las_intensity_mode);
    const bool any_xyz = ex->las_x || ex->las_y || ex->las_z;
    if (any_xyz && !(ex->las_x && ex->las_y && ex->las_z)) return fail(LMC_ERR_INVALID, "las_x/las_y/las_z must be given together");
    if (any_xyz) for (int c = 0; c < 3; ++c)
        if (!(ex->las_scale[c] > 0.0)) return fail(LMC_ERR_INVALID, "las_scale[%d] must be > 0", c);
    if (!aligned32(ex->lvx14) || !aligned32(ex->las_x) || !aligned32(ex->las_y) || !aligned32(ex->las_z) || !aligned32(ex->las_intensity))
        return fail(LMC_ERR_ALIGN, "export arrays must be 32-byte aligned");
    P.lvx14 = ex->lvx14; P.lvx_mode = ex->lvx_mode; P.tag = ex->tag;
    P.las_x = ex->las_x; P.las_y = ex->las_y; P.las_z = ex->las_z; P.las_int = ex->las_intensity;
    P.las_int_mode = ex->las_intensity_mode; P.status = ex->status;
    if (ex->n_peers < 0 || ex->n_peers > LMC_MAX_PEERS) return fail(LMC_ERR_INVALID, "n_peers must be 0..%d", LMC_MAX_PEERS);
    P.n_peers = ex->n_peers;
    for (int r = 0; r < ex->n_peers; ++r) {
        if (!aligned32(ex->peer_out[r]) || !aligned32(ex->peer_lvx14[r])) return fail(LMC_ERR_ALIGN, "peer buffers must be 32-byte aligned");
        P.peer_out[r] = ex->peer_out[r]; P.peer_lvx[r] = ex->peer_lvx14[r];
    }
    if ((ex->mc_out != nullptr) != (ex->mc_lvx14 != nullptr)) return fail(LMC_ERR_INVALID, "mc_out and mc_lvx14 must be given together");
    if (ex->mc_out != nullptr) {
        if (!aligned32(ex->mc_out) || !aligned32(ex->mc_lvx14)) return fail(LMC_ERR_ALIGN, "multicast buffers must be 32-byte aligned");
        if (ex->n_peers < 1) return fail(LMC_ERR_INVALID, "multicast merge also needs the peer pointers (ragged edge tiles use them)");
        P.mc_out = ex->mc_out; P.mc_lvx = ex->mc_lvx14;
    }
    for (int c = 0; c < 3; ++c) { P.las_scale[c] = ex->las_scale[c]; P.las_rcp[c] = 1.0 / ex->las_scale[c]; P.las_off[c] = ex->las_offset[c]; }
    return LMC_OK;
}

int run(bool f64, int mode, lmc::Params& P, const lmc_export* ex, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (P.n_points < 0 || P.n_frames < 0) return fail(LMC_ERR_INVALID, "negative size");
    if (P.p_begin < 0 || P.p_end > P.n_points || P.p_begin > P.p_end) return fail(LMC_ERR_INVALID, "bad point range [%lld, %lld) of %lld",
        (long long)P.p_begin, (long long)P.p_end, (long long)P.n_points);
    if (P.p_begin == P.p_end) return LMC_OK;
    if (!P.pts) return fail(LMC_ERR_INVALID, "pts is NULL");
    if (P.out == P.pts) return fail(LMC_ERR_INVALID, "in-place operation is not supported");
    if (!aligned32(P.pts) || !aligned32(P.out)) return fail(LMC_ERR_ALIGN, "point arrays must be 32-byte aligned");
    if (mode != lmc::kQuantOnly && !P.frame_off) return fail(LMC_ERR_INVALID, "frame_off is NULL");
    if (mode != lmc::kQuantOnly && P.n_frames < 1) return fail(LMC_ERR_INVALID, "points without frames");
    rc = fill_export(P, ex);
    if (rc != LMC_OK) return rc;
    if (!P.out && !P.lvx14 && !P.las_x && !P.las_int) return fail(LMC_ERR_INVALID, "no output requested");
    const lmc::Plan pl = lmc::plan_point_launch(f64, mode, P, g_path.load(std::memory_order_relaxed), g_dev.sm_count);
    if (pl.rc != LMC_OK) return fail(pl.rc, "%s", pl.msg);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (pl.stream) {
        const cudaError_t e = lmc::launch_stream(f64, mode, P, pl, g_dev.dev, st);
        return e == cudaSuccess ? LMC_OK : cuda_fail(e, "launch (tma path)");
    }
    const cudaError_t e = lmc::launch_direct(f64, mode, P, st);
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "launch (direct path)");
}

lmc::Params base_params(const void* pts, void* out, int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end) {
    lmc::Params P;
    memset(&P, 0, sizeof P);
    P.pts = pts; P.out = out; P.n_points = n_points; P.n_frames = n_frames; P.p_begin = p_begin; P.p_end = p_end;
    return P;
}

}  // namespace

extern "C" {

int lmc_version(void) { return LMC_VERSION; }
const char* lmc_last_error(void) { return g_err; }

int lmc_device_query(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
    int dev = 0, v = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
    if (sm_count) { e = cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev); if (e != cudaSuccess) return cuda_fail(e, "attr"); *sm_count = v; }
    if (cc_major) { e = cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev); if (e != cudaSuccess) return cuda_fail(e, "attr"); *cc_major = v; }
    if (cc_minor) { e = cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev); if (e != cudaSuccess) return cuda_fail(e, "attr"); *cc_minor = v; }
    return check_device();
}

int lmc_set_path(int32_t path) {
    if (path < 0 || path > 2) return fail(LMC_ERR_INVALID, "path must be 0 (direct), 1 (auto) or 2 (tma)");
    g_path = path;
    return LMC_OK;
}
int lmc_get_path(void) { return g_path.load(std::memory_order_relaxed); }

int lmc_pose_lookup_hold_next(const double* traj_t, int64_t n_t, const double* traj_Rt, const double* frame_t,
                              int32_t n_frames, double* pose_Rt, int32_t* pose_idx, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_frames < 0 || n_t < 1) return fail(LMC_ERR_INVALID, "need n_t >= 1, n_frames >= 0");
    if (!traj_t || !traj_Rt || !frame_t || !pose_Rt) return fail(LMC_ERR_INVALID, "NULL argument");
    if ((reinterpret_cast<uintptr_t>(traj_Rt) | reinterpret_cast<uintptr_t>(pose_Rt)) & 15u) return fail(LMC_ERR_ALIGN, "pose tables must be 16-byte aligned");
    cudaError_t e = lmc::launch_pose_lookup(traj_t, n_t, traj_Rt, frame_t, n_frames, pose_Rt, pose_idx, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_pose_lookup");
}

int lmc_build_slerp_table(const double* sample_quat_xyzw, const double* sample_pos, const int64_t* sample_ts, int64_t n_samples,
                          double* seg_out, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_samples < 0) return fail(LMC_ERR_INVALID, "negative n_samples");
    if (n_samples == 0) return LMC_OK;
    if (!sample_quat_xyzw || !sample_pos || !sample_ts || !seg_out) return fail(LMC_ERR_INVALID, "NULL argument");
    if ((reinterpret_cast<uintptr_t>(sample_quat_xyzw) | reinterpret_cast<uintptr_t>(seg_out)) & 15u) return fail(LMC_ERR_ALIGN, "quaternions and table must be 16-byte aligned");
    cudaError_t e = lmc::launch_slerp_table(sample_quat_xyzw, sample_pos, sample_ts, n_samples, seg_out, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_slerp_table");
}

static int align_rigid(bool f64, const void* pts, const int64_t* frame_off, const double* pose_Rt, void* out,
                       int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    lmc::Params P = base_params(pts, out, n_points, n_frames, p_begin, p_end);
    if (!pose_Rt) return fail(LMC_ERR_INVALID, "pose_Rt is NULL");
    if (reinterpret_cast<uintptr_t>(pose_Rt) & 15u) return fail(LMC_ERR_ALIGN, "pose_Rt must be 16-byte aligned");
    P.frame_off = frame_off; P.pose_Rt = pose_Rt;
    return run(f64, lmc::kRigid, P, ex, stream);
}
int lmc_align_rigid_f64(const double* pts_n4, const int64_t* frame_off, const double* pose_Rt, double* out_n4,
                        int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    return align_rigid(true, pts_n4, frame_off, pose_Rt, out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}
int lmc_align_rigid_f32(const float* pts_n4, const int64_t* frame_off, const double* pose_Rt, float* out_n4,
                        int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    return align_rigid(false, pts_n4, frame_off, pose_Rt, out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}

static int deskew_gyro(bool f64, const void* pts, const void* ts, const int64_t* frame_off, const int64_t* frame_start,
                       const int64_t* imu_ts, const double* imu_gyro, int64_t n_imu, void* out,
                       int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    lmc::Params P = base_params(pts, out, n_points, n_frames, p_begin, p_end);
    if (n_imu < 0) return fail(LMC_ERR_INVALID, "n_imu < 0");
    if (!ts || !frame_start) return fail(LMC_ERR_INVALID, "timestamps / frame_start are NULL");
    if (n_imu > 0 && (!imu_ts || !imu_gyro)) return fail(LMC_ERR_INVALID, "imu tables are NULL");
    if (reinterpret_cast<uintptr_t>(ts) & 15u) return fail(LMC_ERR_ALIGN, "timestamps must be 16-byte aligned");
    P.frame_off = frame_off; P.frame_start = frame_start; P.ts = ts;
    P.samp_ts = imu_ts; P.samp_tab = imu_gyro; P.n_samp = n_imu;
    return run(f64, lmc::kGyro, P, ex, stream);
}
int lmc_deskew_gyro_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off, const int64_t* frame_start,
                        const int64_t* imu_ts, const double* imu_gyro, int64_t n_imu, double* out_n4,
                        int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    return deskew_gyro(true, pts_n4, ts, frame_off, frame_start, imu_ts, imu_gyro, n_imu, out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}
int lmc_deskew_gyro_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off, const int64_t* frame_start,
                        const int64_t* imu_ts, const double* imu_gyro, int64_t n_imu, float* out_n4,
                        int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    return deskew_gyro(false, pts_n4, ts_off, frame_off, frame_start, imu_ts, imu_gyro, n_imu, out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}

// Mode C (kSlerp, with the optional hold_idx), sensor-frame deskew (kSlerpLocal, with ref_pose) and distortion (kSlerpDistort).
// f32 points carry ns offsets from their frame's start, so they need frame_start.
static int slerp_family(bool f64, int mode, const void* pts, const void* ts, const int64_t* frame_off, const int64_t* frame_start,
                        const int64_t* sample_ts, const double* seg, int64_t n_samples, const int32_t* hold_idx, const double* ref_pose,
                        void* out, int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    lmc::Params P = base_params(pts, out, n_points, n_frames, p_begin, p_end);
    if (mode == lmc::kSlerp) {
        if (n_samples < 1 || !sample_ts || !seg) return fail(LMC_ERR_INVALID, "need a non-empty sample table");
    } else {
        if (n_samples < 1 || n_samples >= (1LL << 31) || !sample_ts || !seg)
            return fail(LMC_ERR_INVALID, "need a sample table of 1 .. 2^31 - 1 rows");
        if (mode == lmc::kSlerpLocal && !ref_pose) return fail(LMC_ERR_INVALID, "ref_pose is NULL");
        // (refused here too, not only by the launch plan: an empty point range returns before the plan is made)
        if (ex && (ex->n_peers > 0 || ex->mc_out || ex->mc_lvx14)) return fail(LMC_ERR_INVALID, "%s", lmc::no_merge_reason(mode));
    }
    if (!hold_idx && !ts) return fail(LMC_ERR_INVALID, "timestamps are NULL");
    if (!hold_idx && !f64 && !frame_start) return fail(LMC_ERR_INVALID, "frame_start is NULL");
    if ((reinterpret_cast<uintptr_t>(ts) | reinterpret_cast<uintptr_t>(seg) | reinterpret_cast<uintptr_t>(ref_pose)) & 15u)
        return fail(LMC_ERR_ALIGN, mode == lmc::kSlerpLocal ? "timestamps / seg / ref_pose must be 16-byte aligned" : "timestamps / seg must be 16-byte aligned");
    P.frame_off = frame_off; P.frame_start = frame_start; P.ts = ts; P.pose_Rt = ref_pose;
    P.samp_ts = sample_ts; P.samp_tab = seg; P.n_samp = n_samples; P.hold_idx = hold_idx;
    return run(f64, mode, P, ex, stream);
}
int lmc_deskew_slerp_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off, const int64_t* frame_start,
                         const int64_t* sample_ts, const double* seg, int64_t n_samples, const int32_t* hold_idx,
                         double* out_n4, int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end,
                         const lmc_export* ex, void* stream) {
    return slerp_family(true, lmc::kSlerp, pts_n4, ts, frame_off, frame_start, sample_ts, seg, n_samples, hold_idx, nullptr,
                        out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}
int lmc_deskew_slerp_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off, const int64_t* frame_start,
                         const int64_t* sample_ts, const double* seg, int64_t n_samples, const int32_t* hold_idx,
                         float* out_n4, int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end,
                         const lmc_export* ex, void* stream) {
    return slerp_family(false, lmc::kSlerp, pts_n4, ts_off, frame_off, frame_start, sample_ts, seg, n_samples, hold_idx, nullptr,
                        out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}

int lmc_slerp_pose_at(const int64_t* sample_ts, const double* seg, int64_t n_samples, const int64_t* query_ts, int64_t n_query,
                      double* pose_out, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_samples < 1 || n_samples >= (1LL << 31) || n_query < 0) return fail(LMC_ERR_INVALID, "need 1 <= n_samples < 2^31, n_query >= 0");
    if (n_query == 0) return LMC_OK;
    if (!sample_ts || !seg || !query_ts || !pose_out) return fail(LMC_ERR_INVALID, "NULL argument");
    if ((reinterpret_cast<uintptr_t>(seg) | reinterpret_cast<uintptr_t>(pose_out)) & 15u) return fail(LMC_ERR_ALIGN, "seg / pose_out must be 16-byte aligned");
    cudaError_t e = lmc::launch_slerp_pose_at(sample_ts, seg, n_samples, query_ts, n_query, pose_out, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_slerp_pose_at");
}

int lmc_deskew_slerp_local_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off, const int64_t* frame_start,
                               const int64_t* sample_ts, const double* seg, int64_t n_samples, const double* ref_pose,
                               double* out_n4, int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end,
                               const lmc_export* ex, void* stream) {
    return slerp_family(true, lmc::kSlerpLocal, pts_n4, ts, frame_off, frame_start, sample_ts, seg, n_samples, nullptr, ref_pose,
                        out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}
int lmc_deskew_slerp_local_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off, const int64_t* frame_start,
                               const int64_t* sample_ts, const double* seg, int64_t n_samples, const double* ref_pose,
                               float* out_n4, int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end,
                               const lmc_export* ex, void* stream) {
    return slerp_family(false, lmc::kSlerpLocal, pts_n4, ts_off, frame_off, frame_start, sample_ts, seg, n_samples, nullptr, ref_pose,
                        out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}

int lmc_distort_slerp_f64(const double* pts_n4, const int64_t* ts, const int64_t* frame_off, const int64_t* frame_start,
                          const int64_t* sample_ts, const double* seg, int64_t n_samples, double* out_n4,
                          int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    return slerp_family(true, lmc::kSlerpDistort, pts_n4, ts, frame_off, frame_start, sample_ts, seg, n_samples, nullptr, nullptr,
                        out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}
int lmc_distort_slerp_f32(const float* pts_n4, const uint32_t* ts_off, const int64_t* frame_off, const int64_t* frame_start,
                          const int64_t* sample_ts, const double* seg, int64_t n_samples, float* out_n4,
                          int64_t n_points, int32_t n_frames, int64_t p_begin, int64_t p_end, const lmc_export* ex, void* stream) {
    return slerp_family(false, lmc::kSlerpDistort, pts_n4, ts_off, frame_off, frame_start, sample_ts, seg, n_samples, nullptr, nullptr,
                        out_n4, n_points, n_frames, p_begin, p_end, ex, stream);
}

int lmc_quantize_f64(const double* pts_n4, int64_t n_points, const lmc_export* ex, void* stream) {
    lmc::Params P = base_params(pts_n4, nullptr, n_points, 0, 0, n_points);
    if (!ex) return fail(LMC_ERR_INVALID, "ex is NULL");
    return run(true, lmc::kQuantOnly, P, ex, stream);
}
int lmc_quantize_f32(const float* pts_n4, int64_t n_points, const lmc_export* ex, void* stream) {
    lmc::Params P = base_params(pts_n4, nullptr, n_points, 0, 0, n_points);
    if (!ex) return fail(LMC_ERR_INVALID, "ex is NULL");
    return run(false, lmc::kQuantOnly, P, ex, stream);
}

static int lvx_build(bool f64, const void* pts, const int64_t* frame_off, const int64_t* frame_pos, const double* frame_time,
                     const int64_t* frame_id, uint8_t* file_out, int64_t out_file_pos, int64_t n_points, int32_t n_frames,
                     int32_t f_begin, int32_t f_end, int64_t max_frame_points, uint32_t* status, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_frames < 1 || n_points < 0 || max_frame_points < 0) return fail(LMC_ERR_INVALID, "need n_frames >= 1 (the reference refuses an empty frame list, LMC:75-76)");
    if (f_begin < 0 || f_end > n_frames || f_begin > f_end || out_file_pos < 0) return fail(LMC_ERR_INVALID, "bad frame range [%d, %d) of %d", f_begin, f_end, n_frames);
    if (!frame_off || !frame_pos || !frame_time || !frame_id || !file_out || (n_points > 0 && !pts)) return fail(LMC_ERR_INVALID, "NULL argument");
    // the kernels lay every byte range out at the FILE's 16-byte phase: the shard buffer must sit at the same phase
    if (!aligned32(pts) || ((reinterpret_cast<uintptr_t>(file_out) - (uintptr_t)out_file_pos) & 15u))
        return fail(LMC_ERR_ALIGN, "points must be 32-byte aligned and the file buffer congruent to its file position modulo 16");
    cudaError_t e = lmc::launch_lvx_v11(f64, pts, frame_off, frame_pos, frame_time, frame_id, file_out - out_file_pos, n_frames, f_begin, f_end,
                                        max_frame_points, status, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_lvx_v11");
}
int lmc_lvx_v11_build_range_f64(const double* pts_n4, const int64_t* frame_off, const int64_t* frame_pos, const double* frame_time,
                                const int64_t* frame_id, uint8_t* shard_out, int64_t out_file_pos, int64_t n_points, int32_t n_frames,
                                int32_t f_begin, int32_t f_end, int64_t max_frame_points, uint32_t* status, void* stream) {
    return lvx_build(true, pts_n4, frame_off, frame_pos, frame_time, frame_id, shard_out, out_file_pos, n_points, n_frames, f_begin, f_end, max_frame_points, status, stream);
}
int lmc_lvx_v11_build_range_f32(const float* pts_n4, const int64_t* frame_off, const int64_t* frame_pos, const double* frame_time,
                                const int64_t* frame_id, uint8_t* shard_out, int64_t out_file_pos, int64_t n_points, int32_t n_frames,
                                int32_t f_begin, int32_t f_end, int64_t max_frame_points, uint32_t* status, void* stream) {
    return lvx_build(false, pts_n4, frame_off, frame_pos, frame_time, frame_id, shard_out, out_file_pos, n_points, n_frames, f_begin, f_end, max_frame_points, status, stream);
}
int lmc_lvx_v11_build_f64(const double* pts_n4, const int64_t* frame_off, const int64_t* frame_pos, const double* frame_time,
                          const int64_t* frame_id, uint8_t* file_out, int64_t n_points, int32_t n_frames, int64_t max_frame_points,
                          uint32_t* status, void* stream) {
    return lvx_build(true, pts_n4, frame_off, frame_pos, frame_time, frame_id, file_out, 0, n_points, n_frames, 0, n_frames, max_frame_points, status, stream);
}
int lmc_lvx_v11_build_f32(const float* pts_n4, const int64_t* frame_off, const int64_t* frame_pos, const double* frame_time,
                          const int64_t* frame_id, uint8_t* file_out, int64_t n_points, int32_t n_frames, int64_t max_frame_points,
                          uint32_t* status, void* stream) {
    return lvx_build(false, pts_n4, frame_off, frame_pos, frame_time, frame_id, file_out, 0, n_points, n_frames, 0, n_frames, max_frame_points, status, stream);
}

static int homog(bool f64, const void* pts, const double* T, int32_t order, void* out, int64_t n, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (order != LMC_HOMOG_BATCH && order != LMC_HOMOG_SINGLE) return fail(LMC_ERR_INVALID, "order must be LMC_HOMOG_BATCH or LMC_HOMOG_SINGLE");
    if (n < 0 || !T || (n > 0 && (!pts || !out))) return fail(LMC_ERR_INVALID, "bad argument");
    if (!aligned32(pts) || !aligned32(out)) return fail(LMC_ERR_ALIGN, "point buffers must be 32-byte aligned");
    cudaError_t e = lmc::launch_homog(f64, pts, T, order, out, n, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_homog");
}
int lmc_transform_homog_f64(const double* pts_n4, const double* T_host, int32_t order, double* out_n4, int64_t n_points, void* stream) {
    return homog(true, pts_n4, T_host, order, out_n4, n_points, stream);
}
int lmc_transform_homog_f32(const float* pts_n4, const double* T_host, int32_t order, float* out_n4, int64_t n_points, void* stream) {
    return homog(false, pts_n4, T_host, order, out_n4, n_points, stream);
}

static int lvx_cs_build(bool f64, const void* pts, const uint8_t* tag, const int64_t* frame_off, const uint64_t* frame_ts,
                        const uint8_t* prefix, int32_t prefix_len, int32_t format, uint8_t* file_out, int64_t n_points, int32_t n_frames,
                        int64_t max_frame_points, uint32_t* status, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (format != LMC_LVXCS_LVX2 && format != LMC_LVXCS_LEGACY) return fail(LMC_ERR_INVALID, "format must be LMC_LVXCS_LVX2 or LMC_LVXCS_LEGACY");
    if (n_frames < 0 || n_points < 0 || max_frame_points < 0) return fail(LMC_ERR_INVALID, "negative count");
    if (prefix_len < 0 || prefix_len > LMC_LVXCS_PREFIX_MAX || (prefix_len > 0 && !prefix)) return fail(LMC_ERR_INVALID, "prefix: 0..%d bytes", LMC_LVXCS_PREFIX_MAX);
    if (!file_out || (n_frames > 0 && (!frame_off || !frame_ts)) || (n_points > 0 && !pts)) return fail(LMC_ERR_INVALID, "NULL argument");
    if (!aligned32(pts) || !aligned32(file_out)) return fail(LMC_ERR_ALIGN, "points and file buffer must be 32-byte aligned");
    cudaError_t e = lmc::launch_lvx_cs(f64, pts, tag, frame_off, frame_ts, prefix, prefix_len, format, file_out, n_frames, max_frame_points, status,
                                       static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_lvx_cs");
}
int lmc_lvx_cs_build_f64(const double* pts_n4, const uint8_t* tag, const int64_t* frame_off, const uint64_t* frame_ts, const uint8_t* prefix_host,
                         int32_t prefix_len, int32_t format, uint8_t* file_out, int64_t n_points, int32_t n_frames, int64_t max_frame_points,
                         uint32_t* status, void* stream) {
    return lvx_cs_build(true, pts_n4, tag, frame_off, frame_ts, prefix_host, prefix_len, format, file_out, n_points, n_frames, max_frame_points, status, stream);
}
int lmc_lvx_cs_build_f32(const float* pts_n4, const uint8_t* tag, const int64_t* frame_off, const uint64_t* frame_ts, const uint8_t* prefix_host,
                         int32_t prefix_len, int32_t format, uint8_t* file_out, int64_t n_points, int32_t n_frames, int64_t max_frame_points,
                         uint32_t* status, void* stream) {
    return lvx_cs_build(false, pts_n4, tag, frame_off, frame_ts, prefix_host, prefix_len, format, file_out, n_points, n_frames, max_frame_points, status, stream);
}

static int pcd_size(bool f64, const void* pts, int64_t n, int64_t* tile_off, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n < 0 || !tile_off || (n > 0 && !pts)) return fail(LMC_ERR_INVALID, "bad argument");
    if (!aligned_row(pts, f64)) return fail(LMC_ERR_ALIGN, "points must be aligned to one row (32 bytes f64, 16 bytes float4)");
    cudaError_t e = lmc::launch_pcd_size(f64, pts, n, tile_off, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_pcd_len / k_pcd_scan");
}
static int pcd_write(bool f64, const void* pts, int64_t n, const int64_t* tile_off, uint8_t* out, uint32_t* status, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n < 0 || !tile_off || (n > 0 && (!pts || !out))) return fail(LMC_ERR_INVALID, "bad argument");
    if (!aligned_row(pts, f64) || !aligned32(out)) return fail(LMC_ERR_ALIGN, "points must be aligned to one row and the text buffer to 32 bytes");
    cudaError_t e = lmc::launch_pcd_write(f64, pts, n, tile_off, out, status, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_pcd_write");
}
static int pcd_row_off(bool f64, const void* pts, int64_t n, const int64_t* tile_off, const int64_t* rows, int32_t n_rows, int64_t* byte_off, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n < 0 || n_rows < 0 || !tile_off || (n > 0 && !pts) || (n_rows > 0 && (!rows || !byte_off))) return fail(LMC_ERR_INVALID, "bad argument");
    if (!aligned_row(pts, f64)) return fail(LMC_ERR_ALIGN, "points must be aligned to one row (32 bytes f64, 16 bytes float4)");
    cudaError_t e = lmc::launch_pcd_row_off(f64, pts, n, tile_off, rows, n_rows, byte_off, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_pcd_row_off");
}
static int text_check(const void* rows, int64_t n, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* dec, int32_t sep) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n < 0 || (n > 0 && !rows) || !col || !dec) return fail(LMC_ERR_INVALID, "bad argument");
    if (n_cols < 1 || n_cols > LMC_TEXT_MAX_COLS || row_stride < 1) return fail(LMC_ERR_INVALID, "n_cols must be 1..%d, row_stride >= 1", LMC_TEXT_MAX_COLS);
    if (sep < 1 || sep > 255) return fail(LMC_ERR_INVALID, "separator must be one byte");
    for (int c = 0; c < n_cols; ++c)
        if (col[c] < 0 || col[c] >= row_stride || dec[c] < 0 || dec[c] > 9) return fail(LMC_ERR_INVALID, "column %d: source index must be < row_stride, decimals 0..9", c);
    return LMC_OK;
}
static int text_size(bool f64, const void* rows, int64_t n, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* dec, int32_t sep,
                     int64_t* tile_off, void* stream) {
    int rc = text_check(rows, n, row_stride, n_cols, col, dec, sep);
    if (rc != LMC_OK) return rc;
    if (!tile_off) return fail(LMC_ERR_INVALID, "NULL tile_off");
    cudaError_t e = lmc::launch_text_size(f64, rows, n, n_cols, row_stride, col, dec, (uint8_t)sep, tile_off, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_text_len / k_pcd_scan");
}
static int text_write(bool f64, const void* rows, int64_t n, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* dec, int32_t sep,
                      const int64_t* tile_off, uint8_t* out, uint32_t* status, void* stream) {
    int rc = text_check(rows, n, row_stride, n_cols, col, dec, sep);
    if (rc != LMC_OK) return rc;
    if (!tile_off || (n > 0 && !out)) return fail(LMC_ERR_INVALID, "NULL argument");
    if (!aligned32(out)) return fail(LMC_ERR_ALIGN, "text buffer must be 32-byte aligned");
    cudaError_t e = lmc::launch_text_write(f64, rows, n, n_cols, row_stride, col, dec, (uint8_t)sep, tile_off, out, status, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_text_write");
}
int lmc_text_rows_size_f64(const double* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* decimals, int32_t sep,
                           int64_t* tile_off, void* stream) { return text_size(true, rows, n_rows, row_stride, n_cols, col, decimals, sep, tile_off, stream); }
int lmc_text_rows_size_f32(const float* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* decimals, int32_t sep,
                           int64_t* tile_off, void* stream) { return text_size(false, rows, n_rows, row_stride, n_cols, col, decimals, sep, tile_off, stream); }
int lmc_text_rows_write_f64(const double* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* decimals, int32_t sep,
                            const int64_t* tile_off, uint8_t* text_out, uint32_t* status, void* stream) {
    return text_write(true, rows, n_rows, row_stride, n_cols, col, decimals, sep, tile_off, text_out, status, stream);
}
int lmc_text_rows_write_f32(const float* rows, int64_t n_rows, int32_t row_stride, int32_t n_cols, const int32_t* col, const int32_t* decimals, int32_t sep,
                            const int64_t* tile_off, uint8_t* text_out, uint32_t* status, void* stream) {
    return text_write(false, rows, n_rows, row_stride, n_cols, col, decimals, sep, tile_off, text_out, status, stream);
}
int lmc_pcd_ascii_size_f64(const double* pts_n4, int64_t n_points, int64_t* tile_off, void* stream) { return pcd_size(true, pts_n4, n_points, tile_off, stream); }
int lmc_pcd_ascii_size_f32(const float* pts_n4, int64_t n_points, int64_t* tile_off, void* stream) { return pcd_size(false, pts_n4, n_points, tile_off, stream); }
int lmc_pcd_ascii_write_f64(const double* pts_n4, int64_t n_points, const int64_t* tile_off, uint8_t* text_out, uint32_t* status, void* stream) {
    return pcd_write(true, pts_n4, n_points, tile_off, text_out, status, stream);
}
int lmc_pcd_ascii_write_f32(const float* pts_n4, int64_t n_points, const int64_t* tile_off, uint8_t* text_out, uint32_t* status, void* stream) {
    return pcd_write(false, pts_n4, n_points, tile_off, text_out, status, stream);
}

int lmc_pcd_ascii_row_offsets_f64(const double* pts_n4, int64_t n_points, const int64_t* tile_off, const int64_t* rows, int32_t n_rows,
                                  int64_t* byte_off, void* stream) { return pcd_row_off(true, pts_n4, n_points, tile_off, rows, n_rows, byte_off, stream); }
int lmc_pcd_ascii_row_offsets_f32(const float* pts_n4, int64_t n_points, const int64_t* tile_off, const int64_t* rows, int32_t n_rows,
                                  int64_t* byte_off, void* stream) { return pcd_row_off(false, pts_n4, n_points, tile_off, rows, n_rows, byte_off, stream); }

// ---- voxel-grid map: lmc_voxel_index_* (table, ranks, V) then lmc_voxel_reduce_* (sums, centroids) -------------------
int64_t lmc_voxel_workspace_bytes(int64_t n_points) {
    if (n_points < 0 || n_points >= (1LL << 31)) return fail(LMC_ERR_INVALID, "n_points must be 0 .. 2^31 - 1");
    return (int64_t)lmc::voxel_workspace_bytes(n_points);
}
static int voxel_check(const void* pts, int64_t n, const double* leaf, const double* origin, const void* ws) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n < 0 || n >= (1LL << 31)) return fail(LMC_ERR_INVALID, "n_points must be 0 .. 2^31 - 1");
    if (!leaf || !origin || !ws || (n > 0 && !pts)) return fail(LMC_ERR_INVALID, "NULL argument");
    for (int c = 0; c < 3; ++c) {
        if (!(leaf[c] > 0.0 && leaf[c] <= 1.7976931348623157e308)) return fail(LMC_ERR_INVALID, "leaf[%d] must be finite and > 0", c);
        if (!(origin[c] >= -1.7976931348623157e308 && origin[c] <= 1.7976931348623157e308)) return fail(LMC_ERR_INVALID, "origin[%d] must be finite", c);
    }
    if (!aligned32(pts) || !aligned32(ws)) return fail(LMC_ERR_ALIGN, "points and workspace must be 32-byte aligned");
    return LMC_OK;
}
static int voxel_index(bool f64, const void* pts, int64_t n, const double* leaf, const double* origin, void* ws, int64_t* n_voxels,
                       uint32_t* status, void* stream) {
    int rc = voxel_check(pts, n, leaf, origin, ws);
    if (rc != LMC_OK) return rc;
    if (!n_voxels || !status) return fail(LMC_ERR_INVALID, "NULL n_voxels_dev / status");
    cudaError_t e = lmc::launch_voxel_index(f64, pts, n, leaf, origin, ws, n_voxels, status, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_voxel_insert / k_voxel_count / k_voxel_rank");
}
static int voxel_reduce(bool f64, const void* pts, int64_t n, const double* leaf, const double* origin, void* ws, int64_t V, void* out,
                        int32_t* counts, int32_t* point_voxel, void* stream) {
    int rc = voxel_check(pts, n, leaf, origin, ws);
    if (rc != LMC_OK) return rc;
    if (V < 0 || V > n) return fail(LMC_ERR_INVALID, "n_voxels must be 0 .. n_points");
    if (V > 0 && (!out || !counts)) return fail(LMC_ERR_INVALID, "NULL out_n4 / counts");
    if (!aligned32(out) || !aligned32(counts) || !aligned32(point_voxel)) return fail(LMC_ERR_ALIGN, "outputs must be 32-byte aligned");
    cudaError_t e = lmc::launch_voxel_reduce(f64, pts, n, leaf, origin, ws, V, out, counts, point_voxel, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_voxel_accum / k_voxel_finalize");
}
int lmc_voxel_index_f64(const double* pts_n4, int64_t n_points, const double leaf[3], const double origin[3], void* workspace,
                        int64_t* n_voxels_dev, uint32_t* status, void* stream) {
    return voxel_index(true, pts_n4, n_points, leaf, origin, workspace, n_voxels_dev, status, stream);
}
int lmc_voxel_index_f32(const float* pts_n4, int64_t n_points, const double leaf[3], const double origin[3], void* workspace,
                        int64_t* n_voxels_dev, uint32_t* status, void* stream) {
    return voxel_index(false, pts_n4, n_points, leaf, origin, workspace, n_voxels_dev, status, stream);
}
int lmc_voxel_reduce_f64(const double* pts_n4, int64_t n_points, const double leaf[3], const double origin[3], void* workspace,
                         int64_t n_voxels, double* out_n4, int32_t* counts, int32_t* point_voxel, void* stream) {
    return voxel_reduce(true, pts_n4, n_points, leaf, origin, workspace, n_voxels, out_n4, counts, point_voxel, stream);
}
int lmc_voxel_reduce_f32(const float* pts_n4, int64_t n_points, const double leaf[3], const double origin[3], void* workspace,
                         int64_t n_voxels, float* out_n4, int32_t* counts, int32_t* point_voxel, void* stream) {
    return voxel_reduce(false, pts_n4, n_points, leaf, origin, workspace, n_voxels, out_n4, counts, point_voxel, stream);
}

// ---- point map: lmc_map_build (lookup table), lmc_map_nearest_* (fixed-radius nearest), lmc_register_frames_* -------
static const int64_t kMax31 = (1LL << 31) - 1;
static bool finite_d(double v) { return v >= -1.7976931348623157e308 && v <= 1.7976931348623157e308; }
int64_t lmc_map_workspace_bytes(int64_t n_voxels) {
    if (n_voxels < 0 || n_voxels > kMax31) return fail(LMC_ERR_INVALID, "n_voxels must be 0 .. 2^31 - 1");
    return (int64_t)lmc::map_table_bytes(n_voxels);
}
static int map_check(const lmc_point_map* m) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (!m) return fail(LMC_ERR_INVALID, "NULL map");
    if (m->n_points < 0 || m->n_points > kMax31) return fail(LMC_ERR_INVALID, "map n_points must be 0 .. 2^31 - 1");
    if (m->n_voxels < 0 || m->n_voxels > m->n_points) return fail(LMC_ERR_INVALID, "map n_voxels must be 0 .. n_points");
    if (!m->vox_off || !m->table || (m->n_points > 0 && (!m->pts_m4 || !m->index))) return fail(LMC_ERR_INVALID, "NULL map buffer");
    for (int c = 0; c < 3; ++c) {
        if (!(m->leaf[c] > 0.0 && finite_d(m->leaf[c]))) return fail(LMC_ERR_INVALID, "leaf[%d] must be finite and > 0", c);
        if (!finite_d(m->origin[c])) return fail(LMC_ERR_INVALID, "origin[%d] must be finite", c);
    }
    if (!aligned32(m->pts_m4) || !aligned32(m->index) || !aligned32(m->vox_off) || !aligned32(m->table))
        return fail(LMC_ERR_ALIGN, "map buffers must be 32-byte aligned");
    return LMC_OK;
}
// r2 = max_dist^2 rounded once; max_dist <= min(leaf) keeps the ball inside the 27 cells around the query's
static int gate_check(const lmc_point_map* m, double max_dist, double* r2) {
    if (!(max_dist > 0.0 && finite_d(max_dist))) return fail(LMC_ERR_INVALID, "max_dist must be finite and > 0");
    for (int c = 0; c < 3; ++c)
        if (max_dist > m->leaf[c]) return fail(LMC_ERR_INVALID, "max_dist must be <= min(leaf)");
    *r2 = max_dist * max_dist;
    return LMC_OK;
}
int lmc_map_build(const lmc_point_map* map, void* stream) {
    int rc = map_check(map);
    if (rc != LMC_OK) return rc;
    cudaError_t e = lmc::launch_map_build(map->pts_m4, map->vox_off, map->n_voxels, map->leaf, map->origin, map->table,
                                          static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_map_insert");
}
static int map_nearest(bool f64, const void* pts, int64_t n, const lmc_point_map* m, double max_dist, int64_t* idx_out, double* d2_out,
                       uint32_t* status, void* stream) {
    int rc = map_check(m);
    if (rc != LMC_OK) return rc;
    double r2;
    if ((rc = gate_check(m, max_dist, &r2)) != LMC_OK) return rc;
    if (n < 0 || n > kMax31) return fail(LMC_ERR_INVALID, "n_points must be 0 .. 2^31 - 1");
    if (!status || (n > 0 && (!pts || !idx_out || !d2_out))) return fail(LMC_ERR_INVALID, "NULL argument");
    if (!aligned32(pts) || !aligned32(idx_out) || !aligned32(d2_out)) return fail(LMC_ERR_ALIGN, "points and outputs must be 32-byte aligned");
    cudaError_t e = lmc::launch_map_nearest(f64, pts, n, m->pts_m4, m->index, m->vox_off, m->table, m->n_voxels, m->leaf, m->origin, r2,
                                            idx_out, d2_out, status, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_map_nearest");
}
int lmc_map_nearest_f64(const double* pts_n4, int64_t n_points, const lmc_point_map* map, double max_dist, int64_t* index_out,
                        double* d2_out, uint32_t* status, void* stream) {
    return map_nearest(true, pts_n4, n_points, map, max_dist, index_out, d2_out, status, stream);
}
int lmc_map_nearest_f32(const float* pts_n4, int64_t n_points, const lmc_point_map* map, double max_dist, int64_t* index_out,
                        double* d2_out, uint32_t* status, void* stream) {
    return map_nearest(false, pts_n4, n_points, map, max_dist, index_out, d2_out, status, stream);
}
int64_t lmc_register_workspace_bytes(int64_t n_points, int32_t n_frames) {
    if (n_points < 0 || n_points > kMax31 || n_frames < 0) return fail(LMC_ERR_INVALID, "n_points must be 0 .. 2^31 - 1, n_frames >= 0");
    if (lmc::register_max_chunks(n_points, n_frames) > kMax31) return fail(LMC_ERR_INVALID, "more than 2^31 - 1 point chunks");
    return (int64_t)lmc::register_workspace_bytes(n_points, n_frames);
}
static int register_frames(bool f64, const void* pts, int64_t n, const int64_t* frame_off, int32_t F, const double* pose_in,
                           const lmc_point_map* m, double max_dist, int32_t iters, double tol_t, double tol_r, void* ws, double* pose_out,
                           int32_t* inliers, double* rms, int32_t* iterations, int32_t* flags, uint32_t* status, void* stream) {
    int rc = map_check(m);
    if (rc != LMC_OK) return rc;
    double r2;
    if ((rc = gate_check(m, max_dist, &r2)) != LMC_OK) return rc;
    if (n < 0 || n > kMax31 || F < 0) return fail(LMC_ERR_INVALID, "n_points must be 0 .. 2^31 - 1, n_frames >= 0");
    if (n > 0 && F < 1) return fail(LMC_ERR_INVALID, "points without frames");
    if (lmc::register_max_chunks(n, F) > kMax31) return fail(LMC_ERR_INVALID, "more than 2^31 - 1 point chunks");
    if (iters < 1) return fail(LMC_ERR_INVALID, "iters must be >= 1");
    if (!(tol_t >= 0.0 && finite_d(tol_t) && tol_r >= 0.0 && finite_d(tol_r))) return fail(LMC_ERR_INVALID, "tol_t / tol_r must be finite and >= 0");
    if (!frame_off || !ws || !status || (n > 0 && !pts) ||
        (F > 0 && (!pose_in || !pose_out || !inliers || !rms || !iterations || !flags)))
        return fail(LMC_ERR_INVALID, "NULL argument");
    if (!aligned32(pts) || !aligned32(frame_off) || !aligned32(pose_in) || !aligned32(ws) || !aligned32(pose_out) || !aligned32(inliers) ||
        !aligned32(rms) || !aligned32(iterations) || !aligned32(flags))
        return fail(LMC_ERR_ALIGN, "buffers must be 32-byte aligned");
    cudaError_t e = lmc::launch_register_frames(f64, pts, n, frame_off, F, pose_in, m->pts_m4, m->index, m->vox_off, m->table, m->n_voxels,
                                                m->leaf, m->origin, r2, iters, tol_t, tol_r, ws, pose_out, inliers, rms, iterations, flags,
                                                status, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_reg_accum / k_reg_solve");
}
int lmc_register_frames_f64(const double* pts_n4, int64_t n_points, const int64_t* frame_off, int32_t n_frames, const double* pose_Rt,
                            const lmc_point_map* map, double max_dist, int32_t iters, double tol_t, double tol_r, void* workspace,
                            double* pose_out, int32_t* inliers, double* rms_m, int32_t* iterations, int32_t* flags, uint32_t* status,
                            void* stream) {
    return register_frames(true, pts_n4, n_points, frame_off, n_frames, pose_Rt, map, max_dist, iters, tol_t, tol_r, workspace, pose_out,
                           inliers, rms_m, iterations, flags, status, stream);
}
int lmc_register_frames_f32(const float* pts_n4, int64_t n_points, const int64_t* frame_off, int32_t n_frames, const double* pose_Rt,
                            const lmc_point_map* map, double max_dist, int32_t iters, double tol_t, double tol_r, void* workspace,
                            double* pose_out, int32_t* inliers, double* rms_m, int32_t* iterations, int32_t* flags, uint32_t* status,
                            void* stream) {
    return register_frames(false, pts_n4, n_points, frame_off, n_frames, pose_Rt, map, max_dist, iters, tol_t, tol_r, workspace, pose_out,
                           inliers, rms_m, iterations, flags, status, stream);
}

// ---- host-side staging helpers (no device work): the reference hands over / expects lists of small per-frame
// arrays; packing them into the pinned staging buffer (and unpacking results) is memory-bound host work that one
// Python thread does at 8 GB/s.  These split the byte range over n_threads std::threads.
static void run_threads(int n_threads, int64_t total, const std::function<void(int64_t, int64_t)>& body) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 64) n_threads = 64;
    const int64_t min_chunk = 1 << 20;                                       // not worth a thread below 1 MiB
    int64_t want = (total + min_chunk - 1) / min_chunk;
    if (want < 1) want = 1;
    if (want < n_threads) n_threads = (int)want;
    if (n_threads == 1) { body(0, total); return; }
    std::vector<std::thread> th;
    th.reserve(n_threads - 1);
    const int64_t per = ((total + n_threads - 1) / n_threads + 63) & ~int64_t(63);
    for (int t = 1; t < n_threads; ++t) {
        const int64_t b = per * t, e = b + per < total ? b + per : total;
        if (b < e) th.emplace_back(body, b, e);
    }
    body(0, per < total ? per : total);
    for (auto& x : th) x.join();
}
int lmc_host_gather(const void* const* src, const int64_t* dst_off, int64_t n_src, void* dst, int32_t n_threads) {
    if (n_src < 0 || (n_src > 0 && (!src || !dst_off || !dst))) return fail(LMC_ERR_INVALID, "bad argument");
    if (n_src == 0) return LMC_OK;
    for (int64_t i = 0; i < n_src; ++i) {
        if (dst_off[i + 1] < dst_off[i]) return fail(LMC_ERR_INVALID, "dst_off must be non-decreasing");
        if (dst_off[i + 1] > dst_off[i] && !src[i]) return fail(LMC_ERR_INVALID, "NULL source %lld", (long long)i);
    }
    const int64_t base = dst_off[0], total = dst_off[n_src] - base;
    run_threads(n_threads, total, [&](int64_t b, int64_t e) {
        // first source whose byte range reaches past b
        int64_t lo = 0, hi = n_src;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (dst_off[mid + 1] - base <= b) lo = mid + 1; else hi = mid; }
        for (int64_t i = lo; i < n_src && dst_off[i] - base < e; ++i) {
            const int64_t s0 = dst_off[i] - base, s1 = dst_off[i + 1] - base;
            const int64_t c0 = s0 > b ? s0 : b, c1 = s1 < e ? s1 : e;
            if (c1 > c0) memcpy(static_cast<char*>(dst) + base + c0, static_cast<const char*>(src[i]) + (c0 - s0), (size_t)(c1 - c0));
        }
    });
    return LMC_OK;
}
int lmc_host_copy(void* dst, const void* src, int64_t n_bytes, int32_t n_threads) {
    if (n_bytes < 0 || (n_bytes > 0 && (!dst || !src))) return fail(LMC_ERR_INVALID, "bad argument");
    run_threads(n_threads, n_bytes, [&](int64_t b, int64_t e) { memcpy(static_cast<char*>(dst) + b, static_cast<const char*>(src) + b, (size_t)(e - b)); });
    return LMC_OK;
}

// parts: 1 records of [p_begin, p_end) into out (out[0] = file byte out_file_pos), 2 header into out[0..227), 3 both
static int las_build(bool f64, const void* pts, const double* gps_time, int64_t n, const double* scale, const double* offset,
                     int32_t mode, int32_t year, int32_t day, uint8_t* out, int32_t* mm, uint32_t* status, void* stream,
                     int parts = 3, int64_t p_begin = 0, int64_t p_end = -1, int64_t out_file_pos = 0) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (p_end < 0) p_end = n;
    if (n < 0 || n > 0xffffffffLL) return fail(LMC_ERR_INVALID, "LAS 1.2 holds at most 2^32 - 1 point records");
    if (p_begin < 0 || p_end > n || p_begin > p_end || out_file_pos < 0) return fail(LMC_ERR_INVALID, "bad point range");
    if (!out || !mm || !scale || !offset || ((parts & 1) && p_end > p_begin && !pts)) return fail(LMC_ERR_INVALID, "NULL argument");
    if (mode != LMC_LAS_INTENSITY_UNIT && mode != LMC_LAS_INTENSITY_RAW) return fail(LMC_ERR_INVALID, "bad las_intensity_mode");
    if (!aligned32(pts) || ((reinterpret_cast<uintptr_t>(out) - (uintptr_t)out_file_pos) & 15u))
        return fail(LMC_ERR_ALIGN, "points must be 32-byte aligned and the file buffer congruent to its file position modulo 16");
    lmc::LasParams L;
    memset(&L, 0, sizeof L);
    L.pts = pts; L.gps_time = gps_time; L.out = out - out_file_pos; L.minmax = mm; L.status = status; L.n = (parts == 2) ? n : p_end; L.p_begin = p_begin;
    for (int c = 0; c < 3; ++c) {
        if (!(scale[c] > 0.0)) return fail(LMC_ERR_INVALID, "scale[%d] must be > 0", c);
        L.scale[c] = scale[c]; L.rcp[c] = 1.0 / scale[c]; L.off[c] = offset[c];
    }
    L.intensity_mode = mode; L.year = (uint16_t)year; L.day = (uint16_t)day;
    cudaError_t e = lmc::launch_las_pf3(f64, L, parts, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_las_records / k_las_header");
}
int lmc_las_pf3_records_f64(const double* pts_n4, const double* gps_time, int64_t n_points, int64_t p_begin, int64_t p_end,
                            const double scale[3], const double offset[3], int32_t las_intensity_mode, uint8_t* shard_out,
                            int64_t out_file_pos, int32_t* minmax, uint32_t* status, void* stream) {
    return las_build(true, pts_n4, gps_time, n_points, scale, offset, las_intensity_mode, 0, 0, shard_out, minmax, status, stream, 1, p_begin, p_end, out_file_pos);
}
int lmc_las_pf3_records_f32(const float* pts_n4, const double* gps_time, int64_t n_points, int64_t p_begin, int64_t p_end,
                            const double scale[3], const double offset[3], int32_t las_intensity_mode, uint8_t* shard_out,
                            int64_t out_file_pos, int32_t* minmax, uint32_t* status, void* stream) {
    return las_build(false, pts_n4, gps_time, n_points, scale, offset, las_intensity_mode, 0, 0, shard_out, minmax, status, stream, 1, p_begin, p_end, out_file_pos);
}
int lmc_las_pf3_header(int64_t n_points, const double scale[3], const double offset[3], int32_t year, int32_t day_of_year,
                       const int32_t* minmax, uint8_t* header_out, void* stream) {
    return las_build(false, nullptr, nullptr, n_points, scale, offset, LMC_LAS_INTENSITY_UNIT, year, day_of_year, header_out,
                     const_cast<int32_t*>(minmax), nullptr, stream, 2);
}
int lmc_las_pf3_build_f64(const double* pts_n4, const double* gps_time, int64_t n_points, const double scale[3], const double offset[3],
                          int32_t las_intensity_mode, int32_t year, int32_t day_of_year, uint8_t* file_out, int32_t* minmax_scratch,
                          uint32_t* status, void* stream) {
    return las_build(true, pts_n4, gps_time, n_points, scale, offset, las_intensity_mode, year, day_of_year, file_out, minmax_scratch, status, stream);
}
int lmc_las_pf3_build_f32(const float* pts_n4, const double* gps_time, int64_t n_points, const double scale[3], const double offset[3],
                          int32_t las_intensity_mode, int32_t year, int32_t day_of_year, uint8_t* file_out, int32_t* minmax_scratch,
                          uint32_t* status, void* stream) {
    return las_build(false, pts_n4, gps_time, n_points, scale, offset, las_intensity_mode, year, day_of_year, file_out, minmax_scratch, status, stream);
}

int lmc_scan_mark(const double* env_m4, int64_t n_env, const double* pos_f3, const double* R_f9, int32_t n_frames,
                  double range_max_sq, double fov_h_half_deg, double fov_v_half_deg, double range_min, double edge_eps_deg,
                  uint8_t* flags, int32_t* tile_off, int32_t* n_visible, int32_t* n_uncertain, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_env < 0 || n_frames < 0 || !(edge_eps_deg >= 0.0)) return fail(LMC_ERR_INVALID, "negative size / edge_eps");
    if (n_env > LMC_SCAN_MAX_ENV) return fail(LMC_ERR_INVALID, "n_env above LMC_SCAN_MAX_ENV");
    if (n_frames == 0) return LMC_OK;
    if (!pos_f3 || !R_f9 || !tile_off || !n_visible || (n_env > 0 && (!env_m4 || !flags))) return fail(LMC_ERR_INVALID, "NULL argument");
    if (!aligned32(env_m4)) return fail(LMC_ERR_ALIGN, "environment must be 32-byte aligned");
    cudaError_t e = lmc::launch_scan_mark(env_m4, n_env, pos_f3, R_f9, n_frames, range_max_sq, fov_h_half_deg, fov_v_half_deg, range_min,
                                          edge_eps_deg, flags, tile_off, n_visible, n_uncertain, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_scan_mark / k_scan_offsets");
}
int lmc_scan_recount(const uint8_t* flags, int64_t n_env, int32_t n_frames, int32_t* tile_off, int32_t* n_visible, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_env < 0 || n_frames < 0) return fail(LMC_ERR_INVALID, "negative size");
    if (n_env > LMC_SCAN_MAX_ENV) return fail(LMC_ERR_INVALID, "n_env above LMC_SCAN_MAX_ENV");
    if (n_frames == 0) return LMC_OK;
    if (!tile_off || !n_visible || (n_env > 0 && !flags)) return fail(LMC_ERR_INVALID, "NULL argument");
    cudaError_t e = lmc::launch_scan_recount(flags, n_env, n_frames, tile_off, n_visible, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_scan_count / k_scan_offsets");
}
int lmc_scan_emit(const double* env_m4, int64_t n_env, const double* pos_f3, const double* R_f9, int32_t n_frames,
                  double range_max_sq, const uint8_t* flags, const int32_t* tile_off, const int32_t* n_visible,
                  const int64_t* frame_off, int32_t max_points, const double* noise_n3, double* raw_out_n4, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_env < 0 || n_frames < 0 || max_points < 1) return fail(LMC_ERR_INVALID, "bad size / max_points");
    if (n_env > LMC_SCAN_MAX_ENV) return fail(LMC_ERR_INVALID, "n_env above LMC_SCAN_MAX_ENV");
    if (n_frames == 0 || n_env == 0) return LMC_OK;
    if (!env_m4 || !pos_f3 || !R_f9 || !flags || !tile_off || !n_visible || !frame_off || !raw_out_n4) return fail(LMC_ERR_INVALID, "NULL argument");
    if (!aligned32(env_m4) || !aligned32(raw_out_n4)) return fail(LMC_ERR_ALIGN, "environment / output must be 32-byte aligned");
    cudaError_t e = lmc::launch_scan_emit(env_m4, n_env, pos_f3, R_f9, n_frames, range_max_sq, flags, tile_off, n_visible, frame_off, max_points,
                                          noise_n3, raw_out_n4, nullptr, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_scan_emit");
}
int lmc_scan_emit_index(const double* env_m4, int64_t n_env, const double* pos_f3, const double* R_f9, int32_t n_frames,
                        double range_max_sq, const uint8_t* flags, const int32_t* tile_off, const int32_t* n_visible,
                        const int64_t* frame_off, int32_t max_points, int64_t* env_idx_out, void* stream) {
    int rc = check_device();
    if (rc != LMC_OK) return rc;
    if (n_env < 0 || n_frames < 0 || max_points < 1) return fail(LMC_ERR_INVALID, "bad size / max_points");
    if (n_env > LMC_SCAN_MAX_ENV) return fail(LMC_ERR_INVALID, "n_env above LMC_SCAN_MAX_ENV");
    if (n_frames == 0 || n_env == 0) return LMC_OK;
    if (!env_m4 || !pos_f3 || !R_f9 || !flags || !tile_off || !n_visible || !frame_off || !env_idx_out) return fail(LMC_ERR_INVALID, "NULL argument");
    cudaError_t e = lmc::launch_scan_emit(env_m4, n_env, pos_f3, R_f9, n_frames, range_max_sq, flags, tile_off, n_visible, frame_off, max_points,
                                          nullptr, nullptr, env_idx_out, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? LMC_OK : cuda_fail(e, "k_scan_emit (index)");
}

}  // extern "C"
