/*
 * lmc_oracle_distort.c -- CPU definition of distortion, the inverse of Mode C: a world point into the sensor frame of Mode C's
 * pose at the point's own time.
 *
 * TEST INFRASTRUCTURE ONLY, like lmc_oracle.c and lmc_oracle_local.c: only tests/ and the profiles may load it, as the
 * checker.  The product never imports, links or executes it.
 *
 * PARITY UNPINNED for the rotation, as Mode C's: the reference has no per-point SLERP.  Bracket, clamps, alpha and the
 * Rodrigues step are Mode C's, restated here exactly as lmc_oracle_local.c states them.
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

/* lmc_oracle_local.c::slerp_bracket: Mode C's bracket, end clamps and alpha (no hold-next) */
static int64_t slerp_bracket(const int64_t* sample_ts, const double* seg, int64_t n_samples, int64_t t, double* alpha)
{
    int64_t k = bracket_right(sample_ts, n_samples, t);
    *alpha = 0.0;
    if (k < 0) k = 0;
    else if (k >= n_samples - 1) k = n_samples - 1;
    else *alpha = (double)(t - sample_ts[k]) * seg[ORC_SEG_STRIDE * k + 19];
    return k;
}

/* lmc_oracle_local.c::slerp_rodrigues: v + sin(th) n x v + (1 - cos(th)) n x (n x v), th = alpha * theta_k, n = n_k */
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

/* Every world point W at its time ts[i] into the sensor frame of Mode C's pose there, R(t)^T (W - x(t))
 * (validated against scipy Slerp + np.interp in oracle/lmc_oracle_distort.py::distort_slerp_scipy):
 *   d_r   = fma(-alpha, dpos_k[r], W_r - pos_k[r])      (the offset before the lerp: no UTM magnitudes in the result)
 *   v_c   = fma(R_k[2][c], d_2, fma(R_k[1][c], d_1, R_k[0][c] * d_0))      (R_k^T d)
 *   out   = rot step of v by -alpha * theta_k about n_k;  out_3 = W_3
 * orc_deskew_slerp_f64 of the result gives W back (to rounding). */
void orc_distort_slerp_f64(const double* pts, const int64_t* ts, int64_t n_points, const int64_t* sample_ts,
                           const double* seg, int64_t n_samples, double* out)
{
    for (int64_t i = 0; i < n_points; ++i) {
        const double* W = pts + 4 * i;
        double* o = out + 4 * i;
        double alpha;
        int64_t k = slerp_bracket(sample_ts, seg, n_samples, ts[i], &alpha);
        const double* s = seg + ORC_SEG_STRIDE * k;
        double d[3], v[3], p1[3];
        for (int r = 0; r < 3; ++r) d[r] = fma(-alpha, s[16 + r], W[r] - s[9 + r]);
        for (int c = 0; c < 3; ++c) v[c] = fma(s[6 + c], d[2], fma(s[3 + c], d[1], s[c] * d[0]));
        slerp_rodrigues(s, -alpha, v[0], v[1], v[2], p1);
        o[0] = p1[0]; o[1] = p1[1]; o[2] = p1[2];
        o[3] = W[3];
    }
}
