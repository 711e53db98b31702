/*
 * lmc_oracle_local.c -- CPU definition of the pose at a time and of sensor-frame deskew.
 *
 * TEST INFRASTRUCTURE ONLY, like lmc_oracle.c (whose Mode C this extends): only tests/ and the profiles may load it, as
 * the checker.  The product never imports, links or executes it.
 *
 * PARITY UNPINNED for the rotation, as Mode C's: the reference has no per-point SLERP.  The bracket and the position lerp
 * are Mode C's, which golden tests/golden/modec_lerp.npz pins.
 *
 * Floating-point discipline as lmc_oracle.c: compile with -ffp-contract=off, every fused multiply-add an explicit fma().
 */
#include <math.h>
#include <stdint.h>

#define ORC_SEG_STRIDE 22        /* lmc_oracle.c: the Mode C per-sample table */

/* lmc_oracle.c::bracket_right: last sample with ts <= target (-1 if none) */
static inline int64_t bracket_right(const int64_t* ts, int64_t n, int64_t target)
{
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = lo + ((hi - lo) >> 1);
        if (ts[mid] <= target) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}
/* lmc_oracle.c::row_gemm: one row of R @ p in OpenBLAS dgemm order */
static inline double row_gemm(const double* r, double x, double y, double z)
{
    return fma(r[2], z, fma(r[1], y, r[0] * x));
}

/* ------------------------------------------------------------------------------------
 * Pose at a time and sensor-frame deskew: Mode C's bracket, clamps and alpha exactly as in
 * orc_deskew_slerp_f64 (no hold-next), and its Rodrigues step
 *   rot(v) = R_k (v + sin(th) n x v + (1 - cos(th)) n x (n x v)),  th = alpha * theta_k, n = n_k
 * (validated against scipy Slerp + np.interp in oracle/lmc_oracle_local.py::slerp_deskew_local_scipy).
 * ---------------------------------------------------------------------------------- */
static int64_t slerp_bracket(const int64_t* sample_ts, const double* seg, int64_t n_samples, int64_t t, double* alpha)
{
    int64_t k = bracket_right(sample_ts, n_samples, t);
    *alpha = 0.0;
    if (k < 0) k = 0;
    else if (k >= n_samples - 1) k = n_samples - 1;
    else *alpha = (double)(t - sample_ts[k]) * seg[ORC_SEG_STRIDE * k + 19];
    return k;
}
/* the Rodrigues step of orc_deskew_slerp_f64 (before R_k) */
static void slerp_rodrigues(const double* s, double alpha, double x, double y, double z, double* p1)
{
    double th = alpha * s[15];
    double sn = sin(th), v = 1.0 - cos(th);
    double nx = s[12], ny = s[13], nz = s[14];
    double c1x = fma(ny, z, -(nz * y)), c1y = fma(nz, x, -(nx * z)), c1z = fma(nx, y, -(ny * x));
    double c2x = fma(ny, c1z, -(nz * c1y)), c2y = fma(nz, c1x, -(nx * c1z)), c2z = fma(nx, c1y, -(ny * c1x));
    p1[0] = fma(v, c2x, fma(sn, c1x, x));
    p1[1] = fma(v, c2y, fma(sn, c1y, y));
    p1[2] = fma(v, c2z, fma(sn, c1z, z));
}

/* pose_out[q] (12 doubles, the layout of orc_align_rigid_f64's pose_Rt): column j of R(t) = rot(e_j),
 * pos(t)_r = fma(alpha, dpos_k[r], pos_k[r]).  orc_align_rigid_f64 with these rows is Mode A at the
 * interpolated pose. */
void orc_slerp_pose_at(const int64_t* sample_ts, const double* seg, int64_t n_samples,
                       const int64_t* query_ts, int64_t n_query, double* pose_out)
{
    for (int64_t q = 0; q < n_query; ++q) {
        double alpha;
        int64_t k = slerp_bracket(sample_ts, seg, n_samples, query_ts[q], &alpha);
        const double* s = seg + ORC_SEG_STRIDE * k;
        double* o = pose_out + 12 * q;
        for (int j = 0; j < 3; ++j) {
            double p1[3];
            slerp_rodrigues(s, alpha, j == 0, j == 1, j == 2, p1);
            for (int r = 0; r < 3; ++r) o[3 * r + j] = row_gemm(s + 3 * r, p1[0], p1[1], p1[2]);
        }
        for (int r = 0; r < 3; ++r) o[9 + r] = fma(alpha, s[16 + r], s[9 + r]);
    }
}

/* Every point of frame f in the sensor frame of (Rr, xr) = ref_pose[f] (12 doubles, R row-major | x):
 *   d_r   = fma(alpha, dpos_k[r], pos_k[r] - xr[r])     (the offset before the lerp: no UTM magnitudes in the result)
 *   w_r   = row_gemm(R_k row r, rot step of p) + d_r
 *   out_c = fma(Rr[2][c], w_2, fma(Rr[1][c], w_1, Rr[0][c] * w_0))      (Rr^T w);  out_3 = p_3 */
void orc_deskew_slerp_local_f64(const double* pts, const int64_t* ts, const int64_t* frame_off,
                                int64_t n_frames, const int64_t* sample_ts, const double* seg,
                                int64_t n_samples, const double* ref_pose, double* out)
{
    for (int64_t f = 0; f < n_frames; ++f) {
        const double* Rr = ref_pose + 12 * f;
        const double* xr = Rr + 9;
        for (int64_t i = frame_off[f]; i < frame_off[f + 1]; ++i) {
            const double* p = pts + 4 * i;
            double* o = out + 4 * i;
            double alpha;
            int64_t k = slerp_bracket(sample_ts, seg, n_samples, ts[i], &alpha);
            const double* s = seg + ORC_SEG_STRIDE * k;
            double p1[3], w[3];
            slerp_rodrigues(s, alpha, p[0], p[1], p[2], p1);
            for (int r = 0; r < 3; ++r) {
                double d = fma(alpha, s[16 + r], s[9 + r] - xr[r]);
                w[r] = row_gemm(s + 3 * r, p1[0], p1[1], p1[2]) + d;
            }
            for (int c = 0; c < 3; ++c) o[c] = fma(Rr[6 + c], w[2], fma(Rr[3 + c], w[1], Rr[c] * w[0]));
            o[3] = p[3];
        }
    }
}
