/*
 * lmc_oracle.c -- CPU restatement of the reference's motion-compensation hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library, and only as the checker / CPU baseline.  The product
 * (livox_motion_compensation_sim_b200) never imports, links or executes it.
 *
 * Parity status: PINNED for Mode A, the LVX / LVX2 quantisers and Mode B -- every
 * function below is checked bit-for-bit against outputs of the real reference
 * (imported from /root/reference in the build container, see
 * tests/golden/make_golden.py) on the committed fixtures in tests/golden/.
 * PARITY UNPINNED for (i) the LAS scale/offset quantiser, whose arithmetic lives in
 * the un-vendored, un-pinned third-party `laspy` (call sites
 * lidar_motion_compensation.py:950-963 and livox_mid70_complete_simulator.py:1671-1698)
 * and is restated here from the LAS 1.2 spec + laspy 2.x behaviour, and (ii) the ROTATION
 * half of Mode C (pose-interp deskew): the reference has no per-point SLERP anywhere.  Its
 * bracket search + position lerp ARE pinned: with identity orientations Mode C equals the
 * reference's own IMUSimulator._interpolate_trajectory (CS:1248-1275, np.interp), golden
 * tests/golden/modec_lerp.npz.
 *
 * Reference citations use LMC = lidar_motion_compensation.py and
 * CS = livox_mid70_complete_simulator.py.
 *
 * Floating-point discipline: compile with -ffp-contract=off; every fused
 * multiply-add below is an explicit fma() so the operation order is exactly the one
 * NumPy/OpenBLAS executes for the reference's expressions (established empirically
 * against the reference, see DESIGN.md "Bit-exact op order").
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define ORC_FLAG_NAN       1u  /* int(nan): the reference raises ValueError          */
#define ORC_FLAG_OVERFLOW  2u  /* struct.pack('<i') / laspy OverflowError territory  */

/* ------------------------------------------------------------------------------------
 * (a1) frame pose lookup -- LMC:804-806
 *   pose_idx = np.searchsorted(trajectory['time'], t)   (side='left')
 *   pose_idx = min(pose_idx, len-1); pose_idx = max(pose_idx, 0)
 * "hold-next": first GPS/IMU sample at or after the frame time, no interpolation.
 * ---------------------------------------------------------------------------------- */
void orc_pose_lookup_hold_next(const double* traj_t, int64_t n_t,
                               const double* frame_t, int64_t n_frames, int32_t* idx_out)
{
    for (int64_t f = 0; f < n_frames; ++f) {
        double t = frame_t[f];
        int64_t lo = 0, hi = n_t;              /* lower_bound: first i with traj_t[i] >= t */
        while (lo < hi) {
            int64_t mid = lo + ((hi - lo) >> 1);
            if (traj_t[mid] < t) lo = mid + 1; else hi = mid;
        }
        if (lo > n_t - 1) lo = n_t - 1;
        if (lo < 0) lo = 0;
        idx_out[f] = (int32_t)lo;
    }
}

/* One row of R @ p in the order OpenBLAS dgemm executes it for (3x3)@(3xN), N >= 2:
 * products accumulated k = 0,1,2 with FMA. */
static inline double row_gemm(const double* r, double x, double y, double z)
{
    return fma(r[2], z, fma(r[1], y, r[0] * x));
}
/* Same row when NumPy routes the product through gemv (N == 1, and every
 * (3,3)@(3,) product in CS): the y product is formed first. */
static inline double row_gemv(const double* r, double x, double y, double z)
{
    return fma(r[2], z, fma(r[0], x, r[1] * y));
}

/* ------------------------------------------------------------------------------------
 * (a2)+(a3) transform_pointcloud over all frames, written frame-major at the CSR
 * offsets (== np.vstack order, LMC:888) -- LMC:772-776
 *   transformed = (R_matrix @ points[:, :3].T).T + translation
 *   return np.column_stack([transformed, points[:, 3]])
 * pose_Rt[f] = 9 doubles of R (row-major, from SciPy on the host) + 3 of translation.
 * ---------------------------------------------------------------------------------- */
void orc_align_rigid_f64(const double* pts, const int64_t* frame_off, const double* pose_Rt,
                         double* out, int64_t n_frames)
{
    for (int64_t f = 0; f < n_frames; ++f) {
        const double* R = pose_Rt + 12 * f;
        const double* t = R + 9;
        int64_t b = frame_off[f], e = frame_off[f + 1];
        int single = (e - b) == 1;
        for (int64_t i = b; i < e; ++i) {
            double x = pts[4 * i], y = pts[4 * i + 1], z = pts[4 * i + 2];
            for (int r = 0; r < 3; ++r) {
                double d = single ? row_gemv(R + 3 * r, x, y, z) : row_gemm(R + 3 * r, x, y, z);
                out[4 * i + r] = d + t[r];
            }
            out[4 * i + 3] = pts[4 * i + 3];
        }
    }
}

/* ------------------------------------------------------------------------------------
 * (a4) LVX data-type-2 point record -- LMC:252-272
 *   x_mm = int(np.clip(point[0] * 1000, -2147483648, 2147483647))   (trunc toward 0)
 *   reflectivity = int(np.clip(point[3] * 255, 0, 255)); tag = 0
 * 14 bytes little-endian <iiiBB.  Applied to RAW sensor-frame points (LMC:977).
 * Returns OR of ORC_FLAG_* (NaN makes the reference raise; we emit 0 and flag).
 * ---------------------------------------------------------------------------------- */
static inline double clipd(double v, double lo, double hi)
{
    /* np.clip == minimum(maximum(v, lo), hi); NaN propagates */
    if (v != v) return v;
    return v < lo ? lo : (v > hi ? hi : v);
}
static inline void put_i32(uint8_t* p, int32_t v) { memcpy(p, &v, 4); }

uint32_t orc_quantize_lvx_type2(const double* pts, int64_t n, uint8_t* out14)
{
    uint32_t flags = 0;
    for (int64_t i = 0; i < n; ++i) {
        uint8_t* o = out14 + 14 * i;
        for (int c = 0; c < 3; ++c) {
            double v = clipd(pts[4 * i + c] * 1000.0, -2147483648.0, 2147483647.0);
            int32_t q = 0;
            if (v != v) flags |= ORC_FLAG_NAN; else q = (int32_t)v;   /* C cast truncates */
            put_i32(o + 4 * c, q);
        }
        double r = clipd(pts[4 * i + 3] * 255.0, 0.0, 255.0);
        uint8_t rq = 0;
        if (r != r) flags |= ORC_FLAG_NAN; else rq = (uint8_t)(int32_t)r;
        o[12] = rq;
        o[13] = 0;
    }
    return flags;
}

/* ------------------------------------------------------------------------------------
 * (a9) LVX2 point record -- CS:365-374
 *   x_mm = int(point.x * 1000)   (trunc, NO clip; struct.pack('<iii') raises if the
 *   value does not fit int32 -> ORC_FLAG_OVERFLOW, value saturated here)
 *   <B intensity, <B tag          (copied)
 * Applied to COMPENSATED points.  pts is (n,4) f64 with integer-valued intensity.
 * ---------------------------------------------------------------------------------- */
uint32_t orc_quantize_lvx2(const double* pts, const uint8_t* tag, int64_t n, uint8_t* out14)
{
    uint32_t flags = 0;
    for (int64_t i = 0; i < n; ++i) {
        uint8_t* o = out14 + 14 * i;
        for (int c = 0; c < 3; ++c) {
            double v = pts[4 * i + c] * 1000.0;
            int32_t q = 0;
            if (v != v) flags |= ORC_FLAG_NAN;
            else {
                double tv = trunc(v);
                if (tv > 2147483647.0)       { flags |= ORC_FLAG_OVERFLOW; q = INT32_MAX; }
                else if (tv < -2147483648.0) { flags |= ORC_FLAG_OVERFLOW; q = INT32_MIN; }
                else q = (int32_t)tv;
            }
            put_i32(o + 4 * c, q);
        }
        double it = pts[4 * i + 3];
        uint8_t iq = 0;
        if (it != it) flags |= ORC_FLAG_NAN;
        else if (it < 0.0 || it > 255.0) { flags |= ORC_FLAG_OVERFLOW; iq = it < 0.0 ? 0 : 255; }
        else iq = (uint8_t)(int32_t)it;
        o[12] = iq;
        o[13] = tag ? tag[i] : 0;
    }
    return flags;
}

/* ------------------------------------------------------------------------------------
 * (a5)/(a10) LAS 1.2 PF3 integer packing -- call sites LMC:950-963, CS:1671-1698.
 * PARITY UNPINNED: the arithmetic is inside laspy (absent, version un-pinned).
 * Restated from laspy 2.x: X = np.round((x - offset) / scale) stored as int32
 * (np.round == round-half-even); OverflowError if it does not fit.
 * intensity_mode 0: LMC:961  (points[:,3] * 65535).astype(np.uint16)   trunc + wrap
 * intensity_mode 1: CS:1686  points[:,3].astype(np.uint16)
 * ---------------------------------------------------------------------------------- */
uint32_t orc_quantize_las(const double* pts, int64_t n, const double* scale, const double* offset,
                          int32_t intensity_mode, int32_t* X, int32_t* Y, int32_t* Z,
                          uint16_t* inten)
{
    uint32_t flags = 0;
    int32_t* dst[3] = { X, Y, Z };
    for (int64_t i = 0; i < n; ++i) {
        for (int c = 0; c < 3; ++c) {
            double v = nearbyint((pts[4 * i + c] - offset[c]) / scale[c]);  /* RN-even */
            int32_t q = 0;
            if (v != v) flags |= ORC_FLAG_NAN;
            else if (v > 2147483647.0)  { flags |= ORC_FLAG_OVERFLOW; q = INT32_MAX; }
            else if (v < -2147483648.0) { flags |= ORC_FLAG_OVERFLOW; q = INT32_MIN; }
            else q = (int32_t)v;
            dst[c][i] = q;
        }
        double it = pts[4 * i + 3];
        if (intensity_mode == 0) it = it * 65535.0;
        uint16_t iq = 0;
        if (it != it) flags |= ORC_FLAG_NAN;
        else if (it >= 9.2e18 || it <= -9.2e18) flags |= ORC_FLAG_OVERFLOW;
        else iq = (uint16_t)(int64_t)it;        /* x86 astype(uint16): cvttsd2si then wrap */
        inten[i] = iq;
    }
    return flags;
}

/* ------------------------------------------------------------------------------------
 * (a7) _interpolate_imu_data bracket -- CS:1482-1516.
 * before = last sample with ts <= target, after = first sample with ts > target
 * (the list is sorted).  Returns k = index of `before` (-1 if none).
 * ---------------------------------------------------------------------------------- */
static inline int64_t bracket_right(const int64_t* ts, int64_t n, int64_t target)
{
    int64_t lo = 0, hi = n;                   /* upper_bound: first i with ts[i] > target */
    while (lo < hi) {
        int64_t mid = lo + ((hi - lo) >> 1);
        if (ts[mid] <= target) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

/* (a8) _create_rotation_matrix -- CS:1518-1536:  Rx(-rx) @ Ry(-ry) @ Rz(-rz), each
 * 3x3 product through dgemm (k = 0,1,2 FMA chain). */
static void mm3(const double* A, const double* B, double* C)
{
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c)
            C[3 * r + c] = fma(A[3 * r + 2], B[6 + c], fma(A[3 * r + 1], B[3 + c], A[3 * r] * B[c]));
}
static void gyro_rotation(const double* ang, double* M)
{
    double rx = ang[0], ry = ang[1], rz = ang[2];
    double Rx[9] = { 1, 0, 0,   0, cos(-rx), -sin(-rx),   0, sin(-rx), cos(-rx) };
    double Ry[9] = { cos(-ry), 0, sin(-ry),   0, 1, 0,   -sin(-ry), 0, cos(-ry) };
    double Rz[9] = { cos(-rz), -sin(-rz), 0,   sin(-rz), cos(-rz), 0,   0, 0, 1 };
    double T[9];
    mm3(Rx, Ry, T);
    mm3(T, Rz, M);
}

/* ------------------------------------------------------------------------------------
 * (a6) MotionCompensator.compensate_point_cloud -- CS:1435-1480 (+ a7, a8)
 * per point:  s = interpolate(imu, ts); dt = (ts - frame_start) * 1e-9;
 *             ang = gyro(s) * dt;  p' = (Rx(-ax) @ Ry(-ay) @ Rz(-az)) @ p
 * Rotation only; intensity (column 3) copied.  n_imu == 0 -> points unchanged
 * (CS:1439-1440).  pts (n,4) f64, ts int64[n] ns, frame_off CSR, frame_start int64[F].
 * ---------------------------------------------------------------------------------- */
void orc_deskew_gyro_f64(const double* pts, const int64_t* ts, const int64_t* frame_off,
                         const int64_t* frame_start, int64_t n_frames,
                         const int64_t* imu_ts, const double* imu_gyro, int64_t n_imu,
                         double* out)
{
    for (int64_t f = 0; f < n_frames; ++f) {
        for (int64_t i = frame_off[f]; i < frame_off[f + 1]; ++i) {
            const double* p = pts + 4 * i;
            double* o = out + 4 * i;
            if (n_imu == 0) { memcpy(o, p, 32); continue; }
            int64_t k = bracket_right(imu_ts, n_imu, ts[i]);
            double g[3];
            if (k < 0) {                       /* no `before`: return after (sample 0) */
                for (int c = 0; c < 3; ++c) g[c] = imu_gyro[c];
            } else if (k >= n_imu - 1) {       /* no `after`: return before (last)     */
                for (int c = 0; c < 3; ++c) g[c] = imu_gyro[3 * (n_imu - 1) + c];
            } else {
                int64_t tb = imu_ts[k], ta = imu_ts[k + 1];
                /* Python int / int true division (correctly rounded; operands < 2^53) */
                double alpha = (double)(ts[i] - tb) / (double)(ta - tb);
                for (int c = 0; c < 3; ++c) {
                    double gb = imu_gyro[3 * k + c], ga = imu_gyro[3 * (k + 1) + c];
                    g[c] = gb + alpha * (ga - gb);            /* CS:1507-1509, no FMA */
                }
            }
            double dt = (double)(ts[i] - frame_start[f]) * 1e-9;       /* CS:1454 */
            double ang[3] = { g[0] * dt, g[1] * dt, g[2] * dt };       /* CS:1457-1458 */
            double M[9];
            gyro_rotation(ang, M);
            for (int r = 0; r < 3; ++r) o[r] = row_gemv(M + 3 * r, p[0], p[1], p[2]);  /* CS:1465 */
            o[3] = p[3];
        }
    }
}

/* ------------------------------------------------------------------------------------
 * Mode C: per-point pose-interp deskew (north_star: binary search + SLERP + lerp).
 * PARITY UNPINNED for the rotation -- no reference implementation exists (docs/Master
 * Guide.md:339-367 is a body-less sketch); bracket + position lerp pinned by the reference's
 * np.interp trajectory interpolation (CS:1248-1275, golden modec_lerp.npz).  Definition
 * (validated against scipy Slerp + lerp in oracle/lmc_oracle.py::slerp_deskew_scipy):
 *   k = bracket_right(sample_ts, ts)  (same bracket rule as a7, clamped at both ends)
 *   alpha = (ts - t_k) * inv_dt_k,  inv_dt_k = 1.0 / (double)(t_{k+1} - t_k) from the table
 *           (a per-segment reciprocal instead of a per-point division: <= 1 ulp from the quotient)
 *   R(ts) = R_k * exp(alpha * rotvec(R_k^-1 R_{k+1}))      == scipy Slerp
 *   pos(ts) = pos_k + alpha * (pos_{k+1} - pos_k)
 *   out = R(ts) p + pos(ts)
 * seg is the per-segment table, SEG_STRIDE doubles per sample k:
 *   [0..8] R_k row-major, [9..11] pos_k, [12..14] unit axis n_k, [15] theta_k,
 *   [16..18] dpos_k = pos_{k+1}-pos_k, [19] inv_dt_k, [20],[21] t_k / dt_k as raw int64 bits (unused
 *   here: the device kernel verifies its bracket guess against them).  Last sample: theta = dpos = inv_dt = 0.
 * hold_idx != NULL: every point of frame f uses sample hold_idx[f] with alpha = 0
 * (Mode A expressed in Mode C: must equal orc_align_rigid_f64 bit-for-bit for n_f >= 2).
 * ---------------------------------------------------------------------------------- */
#define ORC_SEG_STRIDE 22

void orc_deskew_slerp_f64(const double* pts, const int64_t* ts, const int64_t* frame_off,
                          int64_t n_frames, const int64_t* sample_ts, const double* seg,
                          int64_t n_samples, const int32_t* hold_idx, double* out)
{
    for (int64_t f = 0; f < n_frames; ++f) {
        for (int64_t i = frame_off[f]; i < frame_off[f + 1]; ++i) {
            const double* p = pts + 4 * i;
            double* o = out + 4 * i;
            int64_t k; double alpha = 0.0;
            if (hold_idx) k = hold_idx[f];
            else {
                k = bracket_right(sample_ts, n_samples, ts[i]);
                if (k < 0) k = 0;
                else if (k >= n_samples - 1) k = n_samples - 1;
                else alpha = (double)(ts[i] - sample_ts[k]) * seg[ORC_SEG_STRIDE * k + 19];
            }
            const double* s = seg + ORC_SEG_STRIDE * k;
            double th = alpha * s[15];
            double sn = sin(th), v = 1.0 - cos(th);
            double nx = s[12], ny = s[13], nz = s[14];
            double x = p[0], y = p[1], z = p[2];
            /* c1 = n x p ; c2 = n x c1 ; p1 = p + sin*c1 + (1-cos)*c2   (Rodrigues) */
            double c1x = fma(ny, z, -(nz * y)), c1y = fma(nz, x, -(nx * z)), c1z = fma(nx, y, -(ny * x));
            double c2x = fma(ny, c1z, -(nz * c1y)), c2y = fma(nz, c1x, -(nx * c1z)), c2z = fma(nx, c1y, -(ny * c1x));
            double x1 = fma(v, c2x, fma(sn, c1x, x));
            double y1 = fma(v, c2y, fma(sn, c1y, y));
            double z1 = fma(v, c2z, fma(sn, c1z, z));
            for (int r = 0; r < 3; ++r) {
                double t = fma(alpha, s[16 + r], s[9 + r]);
                o[r] = row_gemm(s + 3 * r, x1, y1, z1) + t;
            }
            o[3] = p[3];
        }
    }
}

/* ------------------------------------------------------------------------------------
 * (N4) scan_environment without the noise -- LMC:701-770
 *   d2 = sum((env - pos)**2, axis=1) ; range mask d2 <= range_max**2
 *   rotated = (R.T @ (env - pos).T).T            (dgemm, k = 0,1,2 FMA chain from +0.0, also for one column)
 *   az = arctan2(y, x) * 180 / pi ; el = arcsin(clip(z / max(sqrt(d2), 1e-6), -1, 1)) * 180 / pi
 *   visible = |az| <= fov_h/2 & |el| <= fov_v/2 & range >= range_min   (env order kept)
 *   n_visible > max_points: step = n_visible // max_points; keep indices arange(0, n, step)[:max]
 * Writes the kept points (rotated xyz + intensity) to out (capacity >= M rows) and returns their
 * count; the caller adds np.random.normal noise exactly as LMC:765-768 does.
 * ---------------------------------------------------------------------------------- */
int64_t orc_scan_frame(const double* env, int64_t M, const double* pos, const double* R,
                       double rmax2, double fov_h_half, double fov_v_half, double range_min,
                       int64_t max_points, double* out)
{
    const double pi = 3.141592653589793;
    int64_t nvis = 0;
    for (int64_t i = 0; i < M; ++i) {
        double dx = env[4 * i] - pos[0], dy = env[4 * i + 1] - pos[1], dz = env[4 * i + 2] - pos[2];
        double d2 = (dx * dx + dy * dy) + dz * dz;
        if (!(d2 <= rmax2)) continue;
        /* from +0.0 like dgemm: three -0.0 products sum to +0.0 */
        double x = fma(R[6 + 0], dz, fma(R[3 + 0], dy, fma(R[0], dx, 0.0)));
        double y = fma(R[6 + 1], dz, fma(R[3 + 1], dy, fma(R[1], dx, 0.0)));
        double z = fma(R[6 + 2], dz, fma(R[3 + 2], dy, fma(R[2], dx, 0.0)));
        double rng = sqrt(d2);
        double az = atan2(y, x) * 180.0 / pi;
        double sr = rng > 1e-6 ? rng : 1e-6;
        double q = z / sr; q = q < -1.0 ? -1.0 : (q > 1.0 ? 1.0 : q);
        double el = asin(q) * 180.0 / pi;
        if (!(fabs(az) <= fov_h_half && fabs(el) <= fov_v_half && rng >= range_min)) continue;
        out[4 * nvis] = x; out[4 * nvis + 1] = y; out[4 * nvis + 2] = z; out[4 * nvis + 3] = env[4 * i + 3];
        ++nvis;
    }
    if (nvis > max_points) {
        int64_t step = nvis / max_points, kept = 0;
        for (int64_t j = 0; j < nvis && kept < max_points; j += step, ++kept)
            memmove(out + 4 * kept, out + 4 * j, 32);
        nvis = kept;
    }
    return nvis;
}

int orc_version(void) { return 1; }
