// lmc_device.cuh -- device-side building blocks shared by every kernel of liblmc_b200.so
//
// All floating-point arithmetic that must reproduce the reference bit-for-bit is written with
// explicit __dmul_rn/__dadd_rn/__fma_rn so nvcc can neither contract nor re-associate it; the
// operation orders are the ones NumPy/OpenBLAS execute for the reference's expressions and are
// the same as oracle/lmc_oracle.c (see DESIGN.md "Bit-exact op order").
//
//   LMC = lidar_motion_compensation.py        CS = livox_mid70_complete_simulator.py
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "lmc_plan.h"

namespace lmc {

constexpr int kMaxBnd    = 30;        // frame boundaries cached per tile (more -> per-point global search)
constexpr int kSegStride = 22;        // doubles per Mode C sample row

struct Pt { double x, y, z, w; };

// LAS 1.2 / PF3 file builder (lmc_las.cu)
struct LasParams {
    const void*   pts;
    const double* gps_time;      // optional (CS:1689 gps_time = ts * 1e-9), NULL -> 0.0
    uint8_t*      out;
    int32_t*      minmax;        // device scratch: {minX, maxX, minY, maxY, minZ, maxZ}, pre-set to {MAX, MIN, ...}
    uint32_t*     status;
    int64_t       n;             // records of points [p_begin, n)
    int64_t       p_begin;
    double        scale[3], rcp[3], off[3];
    int32_t       intensity_mode;
    uint16_t      year, day;
};


// frames intersecting one tile of points, staged in shared memory
struct TileMeta {
    int64_t edge[kMaxBnd + 2];    // frame_off[f_lo .. f_lo + nb + 1]
    int64_t fstart[kMaxBnd + 2];  // frame_start[f_lo .. f_lo + nb] (Mode B/C), staged with the edges
    int32_t f_lo;                 // frame of the tile's first point
    int32_t nb;                   // frame boundaries inside the tile
    int32_t overflow;             // more than kMaxBnd boundaries: per-point global search
    int32_t pad;
};

// ------------------------------------------------------------------------------------------
// 256-bit global accesses (sm_100: LDG.E.256 / STG.E.256).  Points are streamed exactly once, so
// loads bypass L1 allocation; a thread's pair of consecutive points is one (f32) or two (f64)
// fully-used 32-byte sectors.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldg256(const double* p, double& a, double& b, double& c, double& d) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void stg256(double* p, double a, double b, double c, double d) {
    asm volatile("st.global.L1::no_allocate.v4.f64 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
__device__ __forceinline__ void ldg256(const float* p, float (&v)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ void stg256(float* p, const float (&v)[8]) {
    asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

__device__ __forceinline__ void lds_f64x2(uint32_t addr, double& a, double& b) {
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(a), "=d"(b) : "r"(addr));
}

// ------------------------------------------------------------------------------------------
// shared -> global TMA bulk stores (cp.async.bulk, SASS UBLKCP.G.S).  Output that is assembled in shared
// memory (packed 14-byte records, file images, text) leaves as ONE asynchronous bulk copy per contiguous
// run instead of an LDS.128 + STG.128 round trip through registers per 16 bytes: fewer instructions, full-line
// writes, and the issuing thread moves on while the copy drains.  The data was written through the generic
// proxy, so every writer executes fence.proxy.async before the barrier that precedes the copy.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {      // 16-byte aligned, size % 16 == 0
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit()      { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0()  { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0()       { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Bytes [b0, b1) of a CTA's shared-memory image -> g[b0, b1), where the image was assembled at the destination's
// 16-byte phase (g + k and img + k are congruent mod 16): aligned body as one bulk store by thread 0, ragged ends
// byte-wise.  Contains the CTA barrier that completes the image; returns once the copy has finished reading it.
__device__ __forceinline__ void cta_image_out(uint8_t* g, const uint8_t* img, int b0, int b1, int tid, int n_threads) {
    fence_async_smem();
    __syncthreads();
    int a0 = (b0 + 15) & ~15; if (a0 > b1) a0 = b1;
    int a1 = b1 & ~15;        if (a1 < a0) a1 = a0;
    const bool body = tid == 0 && a1 > a0;
    if (body) { bulk_s2g(g + a0, img + a0, (uint32_t)(a1 - a0)); bulk_commit(); }
    for (int k = b0 + tid; k < a0; k += n_threads) g[k] = img[k];
    for (int k = a1 + tid; k < b1; k += n_threads) g[k] = img[k];
    if (body) bulk_wait_read0();
}

// A file writer's CTA walks its points as j = tid + k * T: load all K rows first (K independent 16/32-byte loads in flight per
// thread instead of one round trip per loop iteration), then quantise.  Rows at or beyond npts are not touched.
template <bool F64> struct RawRow;
template <> struct RawRow<false> { float4 v;        __device__ __forceinline__ Pt pt() const { return Pt{ (double)v.x, (double)v.y, (double)v.z, (double)v.w }; } };
template <> struct RawRow<true>  { double x, y, z, w; __device__ __forceinline__ Pt pt() const { return Pt{ x, y, z, w }; } };
template <bool F64, int K, int T>
__device__ __forceinline__ void load_rows_strided(const void* __restrict__ pts, int64_t first, int tid, int npts, RawRow<F64> (&r)[K]) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int j = tid + k * T;
        if (j < npts) {
            if constexpr (F64) ldg256(reinterpret_cast<const double*>(pts) + 4 * (first + j), r[k].x, r[k].y, r[k].z, r[k].w);
            else r[k].v = __ldg(reinterpret_cast<const float4*>(pts) + (first + j));
        }
    }
}

// ------------------------------------------------------------------------------------------
// Reference operation orders
// ------------------------------------------------------------------------------------------
// sum_k a_k*b_k as OpenBLAS dgemm runs it for the reference's (3x3)@(3xN), N >= 2  (LMC:775)
__device__ __forceinline__ double dot_gemm(double a0, double b0, double a1, double b1, double a2, double b2) {
    return __fma_rn(a2, b2, __fma_rn(a1, b1, __dmul_rn(a0, b0)));
}
// the same through gemv: NumPy takes this route for a 3x1 right-hand side (single-point frame at
// LMC:775) and for every (3,3)@(3,) product (CS:1465)
__device__ __forceinline__ double dot_gemv(double a0, double b0, double a1, double b1, double a2, double b2) {
    return __fma_rn(a2, b2, __fma_rn(a0, b0, __dmul_rn(a1, b1)));
}

// (a2) R p + t with R,t = 12 doubles
__device__ __forceinline__ void rigid_apply(const double (&M)[12], bool single, const Pt& p, Pt& o) {
    if (single) {
        o.x = __dadd_rn(dot_gemv(M[0], p.x, M[1], p.y, M[2], p.z), M[9]);
        o.y = __dadd_rn(dot_gemv(M[3], p.x, M[4], p.y, M[5], p.z), M[10]);
        o.z = __dadd_rn(dot_gemv(M[6], p.x, M[7], p.y, M[8], p.z), M[11]);
    } else {
        o.x = __dadd_rn(dot_gemm(M[0], p.x, M[1], p.y, M[2], p.z), M[9]);
        o.y = __dadd_rn(dot_gemm(M[3], p.x, M[4], p.y, M[5], p.z), M[10]);
        o.z = __dadd_rn(dot_gemm(M[6], p.x, M[7], p.y, M[8], p.z), M[11]);
    }
    o.w = p.w;
}

// sin(x) and 1 - cos(x).  Deskew angles are tiny (gyro * 0.1 s, or one 5 ms pose segment), so Taylor
// polynomials without range reduction are exact to < 1 ulp; |x| > 0.5 takes the library path.
__constant__ double kSinC[7] = { -7.6471637318198164759e-13 /* -1/15! */, 1.6059043836821614599e-10, -2.5052108385441718775e-08,
                                 2.7557319223985890653e-06, -1.9841269841269841270e-04, 8.3333333333333333333e-03,
                                 -1.6666666666666666667e-01 /* -1/3! */ };
__constant__ double kCosC[8] = { -4.7794773323873852974e-14 /* -1/16! */, 1.1470745597729724714e-11, -2.0876756987868098979e-09,
                                 2.7557319223985890653e-07, -2.4801587301587301587e-05, 1.3888888888888888889e-03,
                                 -4.1666666666666666667e-02, 0.5 /* 1/2! */ };
// Branch-free polynomial parts.  kSmallAngle covers what deskew actually sees (one 5 ms pose segment,
// gyro * 0.1 s): |x| <= 0.125 needs only degree 11 / 12 (next terms 1e-20, 3e-22 relative); up to 0.5 the
// degree 15 / 16 version is used.  Which one is taken depends on x alone, so the straight-line fast paths
// (which require every angle <= kSmallAngle) and the general path always agree bit-for-bit.
constexpr double kSmallAngle = 0.125;
__device__ __forceinline__ void sin_vercos_small(double x, double& s, double& v) {      // |x| <= kSmallAngle
    const double u = x * x;
    double ps = kSinC[2], pc = kCosC[2];
#pragma unroll
    for (int i = 3; i < 7; ++i) ps = fma(ps, u, kSinC[i]);
#pragma unroll
    for (int i = 3; i < 8; ++i) pc = fma(pc, u, kCosC[i]);
    s = fma(x * u, ps, x);
    v = u * pc;
}
// Gyro deskew angles are rate * (<= 0.1 s): below 2^-4 rad for anything a vehicle does (0.6 rad/s).  Degree 9 / 8
// is then exact to half an ulp (next terms 2e-20 / 3e-19), and cos comes out of one FMA instead of 1 - v:
// 8 FP64 operations per angle instead of 13.  Mode B picks this tier per POINT (all three angles below
// kTinyAngle), in the fast and the general path alike, so a point's result does not depend on which path
// evaluated it.
constexpr double kTinyAngle = 0.0625;
constexpr uint32_t kTinyHi = 0x3FB00000u, kSmallHi = 0x3FC00000u;      // high words of 2^-4 and of kSmallAngle = 2^-3
__device__ __forceinline__ void sin_cos_tiny(double x, double& s, double& c) {          // |x| < kTinyAngle
    const double u = x * x;
    const double ps = fma(fma(fma(kSinC[3], u, kSinC[4]), u, kSinC[5]), u, kSinC[6]);
    const double pc = fma(fma(fma(-kCosC[4], u, -kCosC[5]), u, -kCosC[6]), u, -kCosC[7]);
    s = fma(x * u, ps, x);
    c = fma(u, pc, 1.0);
}
__device__ __forceinline__ void sin_vercos_mid(double x, double& s, double& v) {        // |x| <= 0.5
    const double u = x * x;
    double ps = kSinC[0], pc = kCosC[0];
#pragma unroll
    for (int i = 1; i < 7; ++i) ps = fma(ps, u, kSinC[i]);
#pragma unroll
    for (int i = 1; i < 8; ++i) pc = fma(pc, u, kCosC[i]);
    s = fma(x * u, ps, x);
    v = u * pc;
}
__device__ __forceinline__ void sin_vercos(double x, double& s, double& v) {
    if (fabs(x) <= kSmallAngle) {
        sin_vercos_small(x, s, v);
    } else if (fabs(x) <= 0.5) {
        sin_vercos_mid(x, s, v);
    } else {
        double c;
        sincos(x, &s, &c);
        v = 1.0 - c;
    }
}

// (a8) CS:1518-1536  Rx(-rx) @ Ry(-ry) @ Rz(-rz), both 3x3 products in dgemm order, then
// (CS:1465) M @ p in gemv order.  The structural zeros/ones of the factors are kept as literal
// operands so signed zeros and non-finite inputs behave exactly like the reference's dgemm.
__device__ __forceinline__ void gyro_rotate(double ax, double ay, double az, const Pt& p, Pt& o) {
    double sa, ca, sb, cb, sc, cc;
    if (fmax(fmax(fabs(ax), fabs(ay)), fabs(az)) < kTinyAngle) {
        sin_cos_tiny(-ax, sa, ca);
        sin_cos_tiny(-ay, sb, cb);
        sin_cos_tiny(-az, sc, cc);
    } else {
        double va, vb, vc;
        sin_vercos(-ax, sa, va);
        sin_vercos(-ay, sb, vb);
        sin_vercos(-az, sc, vc);
        ca = 1.0 - va; cb = 1.0 - vb; cc = 1.0 - vc;
    }
    const double Rx[9] = { 1.0, 0.0, 0.0,   0.0, ca, -sa,   0.0, sa, ca };
    const double Ry[9] = { cb, 0.0, sb,   0.0, 1.0, 0.0,   -sb, 0.0, cb };
    const double Rz[9] = { cc, -sc, 0.0,   sc, cc, 0.0,   0.0, 0.0, 1.0 };
    double T[9], M[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c)
            T[3 * r + c] = dot_gemm(Rx[3 * r], Ry[c], Rx[3 * r + 1], Ry[3 + c], Rx[3 * r + 2], Ry[6 + c]);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c)
            M[3 * r + c] = dot_gemm(T[3 * r], Rz[c], T[3 * r + 1], Rz[3 + c], T[3 * r + 2], Rz[6 + c]);
    o.x = dot_gemv(M[0], p.x, M[1], p.y, M[2], p.z);
    o.y = dot_gemv(M[3], p.x, M[4], p.y, M[5], p.z);
    o.z = dot_gemv(M[6], p.x, M[7], p.y, M[8], p.z);
    o.w = p.w;
}

// The same rotation for |angles| <= kSmallAngle with the structural zeros / ones of Rx, Ry, Rz folded
// away: every surviving operation is the one the dgemm chain of gyro_rotate() performs on non-zero
// operands (x*0 terms and "+0" additions dropped), so results agree bit-for-bit except possibly in the
// sign of an exact zero.  14 FP64 ops for the matrix instead of 54, branch-free.
template <bool TINY>
__device__ __forceinline__ void gyro_rotate_small(double ax, double ay, double az, const Pt& p, Pt& o) {
    double sa, ca, sb, cb, sc, cc;
    if constexpr (TINY) {                                                // every |angle| < kTinyAngle
        sin_cos_tiny(-ax, sa, ca);
        sin_cos_tiny(-ay, sb, cb);
        sin_cos_tiny(-az, sc, cc);
    } else {
        double va, vb, vc;
        sin_vercos_small(-ax, sa, va);
        sin_vercos_small(-ay, sb, vb);
        sin_vercos_small(-az, sc, vc);
        ca = 1.0 - va; cb = 1.0 - vb; cc = 1.0 - vc;
    }
    const double t10 = __dmul_rn(sa, sb), t20 = -__dmul_rn(ca, sb);         // (Rx Ry)[1][0], [2][0]
    const double m00 = __dmul_rn(cb, cc), m01 = -__dmul_rn(cb, sc), m02 = sb;
    const double m10 = __fma_rn(ca, sc, __dmul_rn(t10, cc)), m11 = __fma_rn(ca, cc, -__dmul_rn(t10, sc)), m12 = -__dmul_rn(sa, cb);
    const double m20 = __fma_rn(sa, sc, __dmul_rn(t20, cc)), m21 = __fma_rn(sa, cc, -__dmul_rn(t20, sc)), m22 = __dmul_rn(ca, cb);
    o.x = dot_gemv(m00, p.x, m01, p.y, m02, p.z);
    o.y = dot_gemv(m10, p.x, m11, p.y, m12, p.z);
    o.z = dot_gemv(m20, p.x, m21, p.y, m22, p.z);
    o.w = p.w;
}

// Mode C's Rodrigues step: p rotated by alpha * theta_k about the unit axis n_k (before R_k is applied); the same operations
// as slerp_apply's first half (kept separate there: routing Mode C through this function perturbs its register allocation)
template <bool SMALL>
__device__ __forceinline__ void slerp_rotate(const double (&s)[kSegStride], double alpha, double px, double py, double pz,
                                             double& x1, double& y1, double& z1) {
    const double th = __dmul_rn(alpha, s[15]);
    double sn, v;
    if (SMALL) sin_vercos_small(th, sn, v); else sin_vercos(th, sn, v);
    const double nx = s[12], ny = s[13], nz = s[14];
    const double c1x = __fma_rn(ny, pz, -__dmul_rn(nz, py));
    const double c1y = __fma_rn(nz, px, -__dmul_rn(nx, pz));
    const double c1z = __fma_rn(nx, py, -__dmul_rn(ny, px));
    const double c2x = __fma_rn(ny, c1z, -__dmul_rn(nz, c1y));
    const double c2y = __fma_rn(nz, c1x, -__dmul_rn(nx, c1z));
    const double c2z = __fma_rn(nx, c1y, -__dmul_rn(ny, c1x));
    x1 = __fma_rn(v, c2x, __fma_rn(sn, c1x, px));
    y1 = __fma_rn(v, c2y, __fma_rn(sn, c1y, py));
    z1 = __fma_rn(v, c2z, __fma_rn(sn, c1z, pz));
}

// Mode C per-point evaluation (definition: oracle/lmc_oracle.c::orc_deskew_slerp_f64)
template <bool SMALL = false>
__device__ __forceinline__ void slerp_apply(const double (&s)[kSegStride], double alpha, const Pt& p, Pt& o) {
    const double th = __dmul_rn(alpha, s[15]);
    double sn, v;
    if (SMALL) sin_vercos_small(th, sn, v); else sin_vercos(th, sn, v);
    const double nx = s[12], ny = s[13], nz = s[14];
    const double c1x = __fma_rn(ny, p.z, -__dmul_rn(nz, p.y));
    const double c1y = __fma_rn(nz, p.x, -__dmul_rn(nx, p.z));
    const double c1z = __fma_rn(nx, p.y, -__dmul_rn(ny, p.x));
    const double c2x = __fma_rn(ny, c1z, -__dmul_rn(nz, c1y));
    const double c2y = __fma_rn(nz, c1x, -__dmul_rn(nx, c1z));
    const double c2z = __fma_rn(nx, c1y, -__dmul_rn(ny, c1x));
    const double x1 = __fma_rn(v, c2x, __fma_rn(sn, c1x, p.x));
    const double y1 = __fma_rn(v, c2y, __fma_rn(sn, c1y, p.y));
    const double z1 = __fma_rn(v, c2z, __fma_rn(sn, c1z, p.z));
    o.x = __dadd_rn(dot_gemm(s[0], x1, s[1], y1, s[2], z1), __fma_rn(alpha, s[16], s[9]));
    o.y = __dadd_rn(dot_gemm(s[3], x1, s[4], y1, s[5], z1), __fma_rn(alpha, s[17], s[10]));
    o.z = __dadd_rn(dot_gemm(s[6], x1, s[7], y1, s[8], z1), __fma_rn(alpha, s[18], s[11]));
    o.w = p.w;
}

// Sensor-frame deskew (definition: oracle/lmc_oracle_local.c::orc_deskew_slerp_local_f64): Mode C's world point, formed as an
// offset from the reference position x_r before the lerp (world-scale magnitudes never enter the result), then R_r^T.
// ref = the frame's reference pose, R_r row-major | x_r.
template <bool SMALL = false>
__device__ __forceinline__ void slerp_local_apply(const double (&s)[kSegStride], double alpha, const double (&ref)[12], const Pt& p, Pt& o) {
    double x1, y1, z1;
    slerp_rotate<SMALL>(s, alpha, p.x, p.y, p.z, x1, y1, z1);
    const double w0 = __dadd_rn(dot_gemm(s[0], x1, s[1], y1, s[2], z1), __fma_rn(alpha, s[16], __dsub_rn(s[9], ref[9])));
    const double w1 = __dadd_rn(dot_gemm(s[3], x1, s[4], y1, s[5], z1), __fma_rn(alpha, s[17], __dsub_rn(s[10], ref[10])));
    const double w2 = __dadd_rn(dot_gemm(s[6], x1, s[7], y1, s[8], z1), __fma_rn(alpha, s[18], __dsub_rn(s[11], ref[11])));
    o.x = dot_gemm(ref[0], w0, ref[3], w1, ref[6], w2);
    o.y = dot_gemm(ref[1], w0, ref[4], w1, ref[7], w2);
    o.z = dot_gemm(ref[2], w0, ref[5], w1, ref[8], w2);
    o.w = p.w;
}
// Distortion, the inverse of Mode C (definition: oracle/lmc_oracle_distort.c::orc_distort_slerp_f64): the world point into the
// sensor frame of Mode C's pose at the point's time, R(t)^T (W - x(t)).  The offset from pos_k is formed before the lerp
// (world-scale magnitudes never enter the result), R_k^T is applied, then the Rodrigues step by -alpha * theta_k.
template <bool SMALL = false>
__device__ __forceinline__ void distort_apply(const double (&s)[kSegStride], double alpha, const Pt& p, Pt& o) {
    const double d0 = __fma_rn(-alpha, s[16], __dsub_rn(p.x, s[9]));
    const double d1 = __fma_rn(-alpha, s[17], __dsub_rn(p.y, s[10]));
    const double d2 = __fma_rn(-alpha, s[18], __dsub_rn(p.z, s[11]));
    const double v0 = dot_gemm(s[0], d0, s[3], d1, s[6], d2);
    const double v1 = dot_gemm(s[1], d0, s[4], d1, s[7], d2);
    const double v2 = dot_gemm(s[2], d0, s[5], d1, s[8], d2);
    slerp_rotate<SMALL>(s, -alpha, v0, v1, v2, o.x, o.y, o.z);
    o.w = p.w;
}
__device__ __forceinline__ void load_pose12(const double* src, double (&m)[12]) {
    const double2* pr = reinterpret_cast<const double2*>(src);
#pragma unroll
    for (int q = 0; q < 6; ++q) { const double2 v = __ldg(pr + q); m[2 * q] = v.x; m[2 * q + 1] = v.y; }
}

// ------------------------------------------------------------------------------------------
// Quantisers.  cvt.rzi.s32.f64 saturates, which IS np.clip to the int32 range followed by
// truncation, so the clip costs nothing; NaN (where the reference raises) sets a status bit and
// quantises to 0, as in the oracle.  The conversion alone does not give 0 for NaN on sm_100
// (a NaN coordinate or intensity left a non-zero record field), so the 0 is selected explicitly.
// The NaN test is made on the INPUT value (v*1000 is NaN iff v is): testing the product instead
// made ptxas keep -- and spill -- every product until a deferred compare.
// ------------------------------------------------------------------------------------------
// ZERO_NAN = false leaves the NaN fields to the caller, which zeroes them off its hot path (the lean streaming epilogue:
// one test per point pair instead of a select per field)
// (a4) LMC:257-259   int(np.clip(v * 1000, -2147483648, 2147483647))
template <bool ZERO_NAN = true>
__device__ __forceinline__ int32_t q_mm_clip(double v, uint32_t& fl) {
    if (v != v) fl |= LMC_FLAG_NAN;
    const int32_t q = __double2int_rz(__dmul_rn(v, 1000.0));   // +-big -> INT_MAX / INT_MIN
    return ZERO_NAN && v != v ? 0 : q;
}
// (a4) LMC:266       int(np.clip(i * 255, 0, 255))
template <bool ZERO_NAN = true>
__device__ __forceinline__ uint32_t q_refl(double w, uint32_t& fl) {
    if (w != w) fl |= LMC_FLAG_NAN;
    const uint32_t r = min(__double2uint_rz(__dmul_rn(w, 255.0)), 255u);   // negative -> 0 (saturating)
    return ZERO_NAN && w != w ? 0u : r;
}
// (a9) CS:368-370    int(v * 1000)  -- no clip; '<iii' packing raises outside int32
__device__ __forceinline__ int32_t q_mm_noclip(double v, uint32_t& fl) {
    const double m = __dmul_rn(v, 1000.0);
    if (v != v) fl |= LMC_FLAG_NAN;
    if (m >= 2147483648.0 || m <= -2147483649.0) fl |= LMC_FLAG_OVERFLOW;
    return v != v ? 0 : __double2int_rz(m);
}
// (a9) CS:373        struct.pack('<B', point.intensity)
__device__ __forceinline__ uint32_t q_u8_copy(double w, uint32_t& fl) {
    if (w != w) fl |= LMC_FLAG_NAN;
    if (w < 0.0 || w > 255.0) fl |= LMC_FLAG_OVERFLOW;
    return w != w ? 0u : min(__double2uint_rz(w), 255u);
}
// (a5)/(a10) laspy: np.round((v - offset) / scale) -> int32   (parity unpinned, see header).
// The quotient is formed with the host-rounded reciprocal and two Markstein corrections
// (q += fma(-s, q, a) * rcp), which yields the correctly rounded a / s -- identical to the IEEE
// division the restatement uses, at 5 FP64 ops instead of a ~25-instruction division sequence.
// exact route (rare: within 2^-20 of a tie, NaN, inf, |q| >= 2^31 - 1): {X, flags}
__device__ __forceinline__ int2 q_las_exact_body(double v, double scale, double rcp, double off) {
    const double a = __dsub_rn(v, off);
    double q = __dmul_rn(a, rcp);
    uint32_t fl = 0;
    if (fabs(q) < 1.0e300) {                        // finite, far from overflow: refine
        q = __fma_rn(__fma_rn(-scale, q, a), rcp, q);
        q = __fma_rn(__fma_rn(-scale, q, a), rcp, q);
    }
    if (v != v) fl |= LMC_FLAG_NAN;
    if (q >= 2147483647.5 || q < -2147483648.5) fl |= LMC_FLAG_OVERFLOW;
    return make_int2(v != v ? 0 : __double2int_rn(q), (int)fl);  // round-half-even, saturates
}
static __device__ __noinline__ int2 q_las_exact(double v, double scale, double rcp, double off) { return q_las_exact_body(v, scale, rcp, off); }
// OOL: the exact route as a call (Mode A + LAS: +1.6 %) or inline (Mode C + LAS, which is register-starved: the call's register
// shuffling costs it 4-6 %) -- same-box A/B, profiles/r02_ab_las.log
template <bool OOL = true>
__device__ __forceinline__ int32_t q_las(double v, double scale, double rcp, double off, uint32_t& fl) {
    // Only the INTEGER np.round(a / scale) is wanted.  q = a * RN(1/scale) is within 2 ulp of the correctly rounded quotient, i.e.
    // within 2^-21 of it for |q| < 2^31; unless q lies that close to a tie k + 0.5 both round to the same integer, and the two
    // Markstein corrections of the exact route are not needed.  d = q - rint(q) is exact; the two range tests run on high words
    // (integer ALU): NaN / inf / |q| >= 2^31 - 1 and everything within 2^-20 of a tie take the exact route.
    const double q = __dmul_rn(__dsub_rn(v, off), rcp);
    const int32_t X = __double2int_rn(q);
    const double d = __dsub_rn(q, (double)X);
    const uint32_t hq = (uint32_t)__double2hiint(q) & 0x7fffffffu, hd = (uint32_t)__double2hiint(d) & 0x7fffffffu;
    if (hq < 0x41DFFFFFu && hd < 0x3FDFFFFEu) return X;
    const int2 r = OOL ? q_las_exact(v, scale, rcp, off) : q_las_exact_body(v, scale, rcp, off);
    fl |= (uint32_t)r.y;
    return r.x;
}
// LMC:961 (w*65535).astype(uint16) | CS:1686 w.astype(uint16): truncate, wrap modulo 2^16
__device__ __forceinline__ uint32_t q_las_intensity(double w, int mode, uint32_t& fl) {
    const double m = mode == LMC_LAS_INTENSITY_UNIT ? __dmul_rn(w, 65535.0) : w;
    if (w != w) fl |= LMC_FLAG_NAN;
    if (m >= 9.2e18 || m <= -9.2e18) { fl |= LMC_FLAG_OVERFLOW; return 0; }
    return w != w ? 0u : (uint32_t)(__double2ll_rz(m) & 0xffff);
}

// ------------------------------------------------------------------------------------------
// Searches over sorted int64 tables (frame_off, imu_ts, sample_ts)
// ------------------------------------------------------------------------------------------
// Warp-cooperative count of elements <= key (== np.searchsorted(a, key, side='right')); key is
// warp-uniform and all 32 lanes must call.  32-ary search: one probe load + ballot per round.
__device__ __forceinline__ int64_t warp_count_le(const int64_t* __restrict__ a, int64_t n, int64_t key, int lane) {
    int64_t lo = 0, hi = n;                       // answer in [lo, hi]
    while (hi - lo > 32) {
        const int64_t len = hi - lo;
        const int64_t pos = lo + (len * (lane + 1)) / 33;          // 32 probes strictly inside (lo, hi)
        const bool le = __ldg(a + pos) <= key;
        const unsigned m = __ballot_sync(0xffffffffu, le);
        const int c = __popc(m);                                    // probes are sorted: true-prefix
        const int64_t nlo = c > 0 ? lo + (len * c) / 33 + 1 : lo;
        const int64_t nhi = c < 32 ? lo + (len * (c + 1)) / 33 : hi;
        lo = nlo; hi = nhi;
    }
    const int64_t idx = lo + lane;
    const bool le = idx < hi && __ldg(a + idx) <= key;
    return lo + __popc(__ballot_sync(0xffffffffu, le));
}

// per-thread binary search restricted to [lo, hi]: count of a[i] <= key
__device__ __forceinline__ int64_t count_le_in(const int64_t* __restrict__ a, int64_t lo, int64_t hi, int64_t key) {
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(a + mid) <= key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Sample-table bracket for one timestamp: k = (count of ts <= t) - 1 in [-1, S-1], i.e. the
// `before` sample of CS:1482-1494.  Guess-and-verify: a table sampled at a (nearly) constant rate
// is hit directly by k ~ (t - t0) * rate, the verification loads (ts[k], ts[k+1]) are the ones the
// interpolation weight needs anyway, and any table that defeats the guess falls back to a binary
// search -- the result is always the exact bracket.
struct Bracket { int64_t k, tb, ta; };            // tb = ts[k], ta = ts[k+1] where they exist
__device__ __forceinline__ Bracket bracket_of(const int64_t* __restrict__ ts, int64_t S, int64_t t, int64_t t0, double rate) {
    Bracket b;
    int64_t k = __double2ll_rz(__dmul_rn((double)(t - t0), rate));
    k = k < 0 ? 0 : (k > S - 1 ? S - 1 : k);
    int64_t tk = __ldg(ts + k);
    if (tk <= t) {                                 // walk right to the last sample <= t
        int steps = 0;
        b.ta = 0;
        while (k + 1 < S) {
            const int64_t tn = __ldg(ts + k + 1);
            if (tn > t) { b.ta = tn; break; }
            k += 1; tk = tn;
            if (++steps == 4) {                    // the guess was far off: finish with a binary search
                k = count_le_in(ts, k + 1, S, t) - 1;
                tk = __ldg(ts + k);
                if (k + 1 < S) b.ta = __ldg(ts + k + 1);
                break;
            }
        }
        b.k = k; b.tb = tk;
    } else {                                       // walk left to the first sample <= t
        int steps = 0;
        b.ta = tk;
        while (true) {
            if (k == 0) { k = -1; tk = 0; break; }
            k -= 1;
            const int64_t tp = __ldg(ts + k);
            if (tp <= t) { tk = tp; break; }
            b.ta = tp;
            if (++steps == 4) {
                k = count_le_in(ts, 0, k, t) - 1;
                tk = k >= 0 ? __ldg(ts + k) : 0;
                b.ta = __ldg(ts + k + 1);
                break;
            }
        }
        b.k = k; b.tb = tk;
    }
    return b;
}

// frame of point p (global index) + whether that frame holds exactly one point
__device__ __forceinline__ int32_t frame_of(const Params& P, const TileMeta& tm, int64_t p, bool& single) {
    if (!tm.overflow) {
        int lo;
        if (tm.nb <= 1) lo = (tm.nb == 1 && tm.edge[1] <= p) ? 1 : 0;    // a tile rarely holds more than one boundary
        else {
            lo = 0; int hi = tm.nb;                 // count of edge[1..nb] <= p
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (tm.edge[1 + mid] <= p) lo = mid + 1; else hi = mid; }
        }
        single = (tm.edge[lo + 1] - tm.edge[lo]) == 1;
        return tm.f_lo + lo;
    }
    const int64_t f = count_le_in(P.frame_off, 0, (int64_t)P.n_frames + 1, p) - 1;
    single = (__ldg(P.frame_off + f + 1) - __ldg(P.frame_off + f)) == 1;
    return (int32_t)f;
}

// One warp fills TileMeta for points [first, last].  hint >= 0 is a frame known to start at or
// before `first` (the previous tile's last frame when a CTA walks consecutive tiles): the frame of
// `first` is then usually found in the next 32 offsets with a single load.
__device__ __forceinline__ void tile_meta(const Params& P, int64_t first, int64_t last, TileMeta& tm, int lane, int64_t hint = -1) {
    const int64_t F = P.n_frames;
    int64_t f_lo = -1;
    if (hint >= 0) {
        const int64_t j = hint + 1 + lane;
        const int64_t v = j <= F ? __ldg(P.frame_off + j) : INT64_MAX;
        const int c = __popc(__ballot_sync(0xffffffffu, v <= first));
        if (c < 32) f_lo = hint + c;
    }
    if (f_lo < 0) f_lo = warp_count_le(P.frame_off, F + 1, first, lane) - 1;   // count >= 1 since frame_off[0] = 0
    int nb = 0; bool done = false; int overflow = 0;
    if (lane == 0) tm.edge[0] = __ldg(P.frame_off + f_lo);
    for (int64_t j0 = f_lo + 1; !done; j0 += 32) {
        const int64_t j = j0 + lane;
        const int64_t v = j <= F ? __ldg(P.frame_off + j) : INT64_MAX;
        const unsigned m = __ballot_sync(0xffffffffu, v <= last);       // true-prefix (sorted)
        const int c = __popc(m);
        if (lane <= c && nb + lane < kMaxBnd + 1) tm.edge[1 + nb + lane] = v;   // boundaries + closing edge
        nb += c;
        done = c < 32;
        if (nb > kMaxBnd) { overflow = 1; done = true; }
    }
    if (P.frame_start != nullptr && !overflow)
        for (int j = lane; j <= nb; j += 32) tm.fstart[j] = __ldg(P.frame_start + f_lo + j);
    if (lane == 0) { tm.f_lo = (int32_t)f_lo; tm.nb = nb; tm.overflow = overflow; }
}
// frame_start of frame f, from the staged copy when the tile has one
__device__ __forceinline__ int64_t frame_start_of(const Params& P, const TileMeta& tm, int32_t f) {
    return tm.overflow ? __ldg(P.frame_start + f) : tm.fstart[f - tm.f_lo];
}

// ------------------------------------------------------------------------------------------
// General per-point evaluation: every corner case (clamps, ragged brackets, big angles, one-point
// frames).  Self-contained (fetches its own pose / sample row), so the out-of-line copy used by
// the rare fall-backs does not force the callers' cached tables out of registers.
//   f / single: frame of the point and whether it is a one-point frame (frame_of)
//   fs: the frame's start time (Mode B/C); tsraw: int64 ns (f64 layout) or uint32 ns offset from fs
// ------------------------------------------------------------------------------------------
template <bool F64, int MODE>
__device__ __forceinline__ Pt point_eval(const Params& P, int32_t f, bool single, int64_t fs, int64_t tsraw, const Pt& in,
                                         int64_t t0, double rate) {
    Pt out = in;
    if constexpr (MODE == kRigid) {
        double M[12];
        const double2* pr = reinterpret_cast<const double2*>(P.pose_Rt + 12 * (int64_t)f);
#pragma unroll
        for (int q = 0; q < 6; ++q) { const double2 v = __ldg(pr + q); M[2 * q] = v.x; M[2 * q + 1] = v.y; }
        rigid_apply(M, single, in, out);
    } else if constexpr (MODE == kGyro) {
        // (a6)/(a7): per-point bracket in imu_ts, gyro lerp, small-angle rotation
        const int64_t S = P.n_samp;
        if (S == 0) return out;                                        // CS:1439-1440: no IMU data -> unchanged
        const int64_t t = F64 ? tsraw : tsraw + fs;
        const Bracket b = bracket_of(P.samp_ts, S, t, t0, rate);
        double g0, g1, g2;
        if (b.k < 0 || b.k >= S - 1) {                                // CS:1495-1496: clamp to the existing end sample
            const double* g = P.samp_tab + 3 * (b.k < 0 ? 0 : S - 1);
            g0 = __ldg(g); g1 = __ldg(g + 1); g2 = __ldg(g + 2);
        } else {
            const double alpha = __ddiv_rn((double)(t - b.tb), (double)(b.ta - b.tb));         // CS:1503 (true division)
            const double* gb = P.samp_tab + 3 * b.k;
            const double b0 = __ldg(gb), b1 = __ldg(gb + 1), b2 = __ldg(gb + 2);
            const double a0 = __ldg(gb + 3), a1 = __ldg(gb + 4), a2 = __ldg(gb + 5);
            g0 = __dadd_rn(b0, __dmul_rn(alpha, __dsub_rn(a0, b0)));                           // CS:1507-1509
            g1 = __dadd_rn(b1, __dmul_rn(alpha, __dsub_rn(a1, b1)));
            g2 = __dadd_rn(b2, __dmul_rn(alpha, __dsub_rn(a2, b2)));
        }
        const double dt = __dmul_rn((double)(t - fs), 1e-9);                                   // CS:1454
        gyro_rotate(__dmul_rn(g0, dt), __dmul_rn(g1, dt), __dmul_rn(g2, dt), in, out);
    } else if constexpr (kSlerpFamily<MODE>) {
        const int64_t S = P.n_samp;
        int64_t k; double alpha = 0.0;
        if (MODE == kSlerp && P.hold_idx != nullptr) k = __ldg(P.hold_idx + f);
        else {
            const int64_t t = F64 ? tsraw : tsraw + fs;
            const Bracket b = bracket_of(P.samp_ts, S, t, t0, rate);
            k = b.k;
            if (k < 0) k = 0;
            else if (k >= S - 1) k = S - 1;
            else alpha = (double)(t - b.tb);                           // times inv_dt_k below
        }
        double row[kSegStride], ref[12];                           // ref: the frame's reference pose (kSlerpLocal)
        const double2* sr = reinterpret_cast<const double2*>(P.samp_tab + kSegStride * k);
#pragma unroll
        for (int q = 0; q < kSegStride / 2; ++q) { const double2 v = __ldg(sr + q); row[2 * q] = v.x; row[2 * q + 1] = v.y; }
        if constexpr (MODE == kSlerpLocal) load_pose12(P.pose_Rt + 12 * (int64_t)f, ref);
        alpha = __dmul_rn(alpha, row[19]);
        if constexpr (MODE == kSlerp)           slerp_apply(row, alpha, in, out);
        else if constexpr (MODE == kSlerpLocal) slerp_local_apply(row, alpha, ref, in, out);
        else                                    distort_apply(row, alpha, in, out);
    }
    return out;
}
template <bool F64, int MODE>
__device__ __noinline__ Pt point_eval_slow(const Params& P, int32_t f, bool single, int64_t fs, int64_t tsraw, Pt in,
                                           int64_t t0, double rate) {
    return point_eval<F64, MODE>(P, f, single, fs, tsraw, in, t0, rate);
}

// ------------------------------------------------------------------------------------------
// Per-thread context for PAIRS of consecutive points: caches the pose / sample row of the previous
// pair (consecutive points almost always share it).  pair() takes a straight-line fast path -- no
// branches between the two points, so their FP64 chains overlap -- when both points share a frame
// pose (Mode A) or a pose segment whose own [t_k, t_{k+1}) verifies the bracket guess (Mode C); any
// other case goes to point_eval().  Both routes execute the same operations in the same order, so
// the results are bit-identical.
// ------------------------------------------------------------------------------------------
template <bool F64, int MODE>
struct PointCtx {
    double  tab[kSlerpFamily<MODE> ? kSegStride : 12];
    int32_t key = -1;            // frame (Mode A) or sample index (Mode C) held in tab
    int64_t t0 = 0;              // Mode B/C: first sample time and mean sample rate for the bracket guess
    double  rate = 0.0;

    __device__ __forceinline__ void init(const Params& P) {
        if constexpr (MODE == kGyro || kSlerpFamily<MODE>) {
            if (P.n_samp > 0) {
                t0 = __ldg(P.samp_ts);
                const int64_t span = __ldg(P.samp_ts + P.n_samp - 1) - t0;
                rate = span > 0 ? (double)(P.n_samp - 1) / (double)span : 0.0;
            }
        }
    }

    __device__ __forceinline__ Pt one(const Params& P, int32_t f, bool single, int64_t fs, int64_t tsraw, const Pt& in) const {
        if constexpr (MODE == kQuantOnly) return in;
        else return point_eval_slow<F64, MODE>(P, f, single, fs, tsraw, in, t0, rate);
    }

    // LEAN: the launcher has checked hold_idx == NULL, 2 <= n_samp < 2^31 (Mode C) -- no runtime tests here
    // CACHE: the producer of the streaming kernel may have staged the pose rows [k_base, k_base + n_rows) of this tile in
    // shared memory (rows_s = their address, info_s + 56 = {k_base, n_rows}); rows found there are read from it.
    template <bool LEAN = false, bool CACHE = false>
    __device__ __forceinline__ void pair(const Params& P, const int32_t (&f)[2], const bool (&single)[2], const int64_t (&fs)[2],
                                         const int64_t (&tsraw)[2], const Pt (&in)[2], Pt (&out)[2],
                                         uint32_t info_s = 0, uint32_t rows_s = 0) {
        if constexpr (MODE == kRigid) {
            if (f[0] == f[1] && !single[0]) {
                if (f[0] != (int32_t)key) {
                    const double2* pr = reinterpret_cast<const double2*>(P.pose_Rt + 12 * (int64_t)f[0]);
#pragma unroll
                    for (int q = 0; q < 6; ++q) { const double2 v = __ldg(pr + q); tab[2 * q] = v.x; tab[2 * q + 1] = v.y; }
                    key = f[0];
                }
                rigid_apply(tab, false, in[0], out[0]);
                rigid_apply(tab, false, in[1], out[1]);
                return;
            }
        }
        if constexpr (kSlerpFamily<MODE>) {
            const int64_t S = P.n_samp;
            if (LEAN || (P.hold_idx == nullptr && S >= 2 && S < 0x7fffffffLL)) {
                const int64_t ta = F64 ? tsraw[0] : tsraw[0] + fs[0];
                const int64_t tb = F64 ? tsraw[1] : tsraw[1] + fs[1];
                // bracket guess from the mean sample rate (saturating conversion, then clamp to a real segment)
                int32_t k = __double2int_rz(__dmul_rn((double)(ta - t0), rate));
                k = max(0, min(k, (int32_t)S - 2));
                const double2* sr = reinterpret_cast<const double2*>(P.samp_tab + (int64_t)kSegStride * k);
                [[maybe_unused]] bool in_s = false; [[maybe_unused]] uint32_t row_s = 0;
                if constexpr (CACHE) {
                    uint32_t kb, nr;
                    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(kb), "=r"(nr) : "r"(info_s + 56u));
                    const uint32_t r = (uint32_t)k - kb;
                    in_s = r < nr; row_s = rows_s + r * (uint32_t)(kSegStride * 8);      // explicit LDS below: a generic pointer costs V4 2.5 %
                }
                // Only the "front" of the row (axis, theta, dpos, 1/dt, t_k, dt_k = columns 12..21) is kept in
                // registers across pairs; R_k and pos_k (columns 0..11) are re-read per pair from L1, where the
                // row stays hot -- holding all 22 doubles plus two points in flight overflows 128 registers
                // and the spills cost more LSU traffic than six broadcast loads.
                if (k != key) {
                    if (CACHE && in_s) {
#pragma unroll
                        for (int q = 6; q < kSegStride / 2; ++q) lds_f64x2(row_s + 16 * q, tab[2 * q], tab[2 * q + 1]);
                    } else {
#pragma unroll
                        for (int q = 6; q < kSegStride / 2; ++q) { const double2 v = __ldg(sr + q); tab[2 * q] = v.x; tab[2 * q + 1] = v.y; }
                    }
                    key = k;
                }
                const int64_t tk = __double_as_longlong(tab[20]);
                const uint64_t dtk = (uint64_t)__double_as_longlong(tab[21]);
                const int64_t da = ta - tk, db = tb - tk;
                // the row's own [t_k, t_k + dt_k) verifies the guess for both points at once
                if ((uint64_t)da < dtk && (uint64_t)db < dtk && tab[15] <= kSmallAngle) {
                    double row[kSegStride];
                    if (CACHE && in_s) {
#pragma unroll
                        for (int q = 0; q < 6; ++q) lds_f64x2(row_s + 16 * q, row[2 * q], row[2 * q + 1]);
                    } else {
#pragma unroll
                        for (int q = 0; q < 6; ++q) { const double2 v = __ldg(sr + q); row[2 * q] = v.x; row[2 * q + 1] = v.y; }
                    }
#pragma unroll
                    for (int q = 12; q < kSegStride; ++q) row[q] = tab[q];
                    const double a0 = __dmul_rn((double)da, row[19]);
                    const double a1 = __dmul_rn((double)db, row[19]);
                    if constexpr (MODE == kSlerp) {
                        slerp_apply<true>(row, a0, in[0], out[0]);
                        slerp_apply<true>(row, a1, in[1], out[1]);
                    } else if constexpr (MODE == kSlerpDistort) {
                        distort_apply<true>(row, a0, in[0], out[0]);
                        distort_apply<true>(row, a1, in[1], out[1]);
                    } else {                                          // the frame's reference pose row: L1, like R_k / pos_k
                        double ref[12];
                        load_pose12(P.pose_Rt + 12 * (int64_t)f[0], ref);
                        slerp_local_apply<true>(row, a0, ref, in[0], out[0]);
                        if (f[1] != f[0]) load_pose12(P.pose_Rt + 12 * (int64_t)f[1], ref);      // (a frame boundary inside the pair: rare)
                        slerp_local_apply<true>(row, a1, ref, in[1], out[1]);
                    }
                    return;
                }
            }
        }
        if constexpr (MODE == kGyro) {
            // (a6)-(a8) CS:1435-1536 for two points bracketed by the same IMU sample pair
            const int64_t S = P.n_samp;
            if (S >= 2 && S < 0x7fffffffLL) {
                const int64_t ta = F64 ? tsraw[0] : tsraw[0] + fs[0];
                const int64_t tb = F64 ? tsraw[1] : tsraw[1] + fs[1];
                int32_t k = __double2int_rz(__dmul_rn((double)(ta - t0), rate));
                k = max(0, min(k, (int32_t)S - 2));
                if (k != key) {
                    const int64_t tk = __ldg(P.samp_ts + k), tn = __ldg(P.samp_ts + k + 1);
                    const double* g = P.samp_tab + 3 * (int64_t)k;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const double gb = __ldg(g + c), ga = __ldg(g + 3 + c);
                        tab[c] = gb;
                        tab[3 + c] = __dsub_rn(ga, gb);                               // CS:1507 (after - before)
                    }
                    tab[6] = __longlong_as_double(tk);
                    tab[7] = __longlong_as_double(((tn - tk) >> 50) == 0 ? tn - tk : 0);   // >= 2^50 ns (13 days): general path
                    tab[8] = (double)(tn - tk);
                    tab[9] = tn > tk ? 1.0 / tab[8] : 0.0;                            // correctly rounded reciprocal (IEEE division)
                    key = k;
                }
                const int64_t tk = __double_as_longlong(tab[6]);
                const uint64_t dtk = (uint64_t)__double_as_longlong(tab[7]);
                const int64_t dd[2] = { ta - tk, tb - tk };
                if ((uint64_t)dd[0] < dtk && (uint64_t)dd[1] < dtk) {
                    double ang[2][3];
                    // max |angle| per point, compared on the high words (exact for the power-of-two tier limits; a NaN
                    // ranks above everything and takes the general path) -- integer ALU instead of DSETP + selects
                    uint32_t am[2] = {0u, 0u};
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        // alpha = (t - t_before) / (t_after - t_before) (CS:1503): reciprocal + ONE Markstein correction
                        // is the correctly rounded quotient here.  a < b are integers, b < 2^50 (checked where the row
                        // is loaded): q0 = a * RN(1/b) is within 2 ulp, the remainder a - b*q0 is exact, so
                        // q0 + rem * r = a/b (1 + 2^-104); and an integer quotient a/b stays >= 2^-51 ulp away from any
                        // rounding boundary when b < 2^50.  (oracle/check_div.c: 4.5e8 (a, b) pairs against IEEE division, none differs.)
                        const double a = (double)dd[h];
                        double q = __dmul_rn(a, tab[9]);
                        q = __fma_rn(__fma_rn(-tab[8], q, a), tab[9], q);
                        const double dt = __dmul_rn((double)((h == 0 ? ta : tb) - fs[h]), 1e-9);      // CS:1454
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const double gc = __dadd_rn(tab[c], __dmul_rn(q, tab[3 + c]));             // CS:1507-1509
                            ang[h][c] = __dmul_rn(gc, dt);                                            // CS:1457-1458
                            am[h] = max(am[h], (uint32_t)__double2hiint(ang[h][c]) & 0x7fffffffu);
                        }
                    }
                    const uint32_t amax = max(am[0], am[1]);
                    if (amax < kTinyHi) {                                     // what a vehicle-mounted IMU produces
                        gyro_rotate_small<true>(ang[0][0], ang[0][1], ang[0][2], in[0], out[0]);
                        gyro_rotate_small<true>(ang[1][0], ang[1][1], ang[1][2], in[1], out[1]);
                        return;
                    }
                    if (amax < kSmallHi) {                                    // polynomial tier per point, as gyro_rotate() picks it
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            if (am[h] < kTinyHi) gyro_rotate_small<true>(ang[h][0], ang[h][1], ang[h][2], in[h], out[h]);
                            else                    gyro_rotate_small<false>(ang[h][0], ang[h][1], ang[h][2], in[h], out[h]);
                        }
                        return;
                    }
                }
            }
        }
        out[0] = one(P, f[0], single[0], fs[0], tsraw[0], in[0]);
        out[1] = one(P, f[1], single[1], fs[1], tsraw[1], in[1]);
    }
};

// LVX record words of one point: x, y, z as u32 and (reflectivity | tag << 8)
template <int MODE>
__device__ __forceinline__ void lvx_words(const Params& P, const Pt& in, const Pt& out, uint32_t tagbyte,
                                          uint32_t& x, uint32_t& y, uint32_t& z, uint32_t& rt, uint32_t& fl) {
    if (P.lvx_mode == LMC_LVX_TYPE2_OF_INPUT) {                       // LMC:252-272 on the raw point
        x = (uint32_t)q_mm_clip(in.x, fl); y = (uint32_t)q_mm_clip(in.y, fl); z = (uint32_t)q_mm_clip(in.z, fl);
        rt = q_refl(in.w, fl);                                         // tag byte = 0
    } else {                                                           // CS:365-374 on the compensated point
        x = (uint32_t)q_mm_noclip(out.x, fl); y = (uint32_t)q_mm_noclip(out.y, fl); z = (uint32_t)q_mm_noclip(out.z, fl);
        rt = q_u8_copy(out.w, fl) | (tagbyte << 8);
    }
}

// 28 bytes of two consecutive records as 7 aligned words
__device__ __forceinline__ void lvx_pair_words(uint32_t* w, const uint32_t (&x)[2], const uint32_t (&y)[2],
                                               const uint32_t (&z)[2], const uint32_t (&rt)[2]) {
    w[0] = x[0]; w[1] = y[0]; w[2] = z[0];
    w[3] = rt[0] | (x[1] << 16);
    w[4] = (x[1] >> 16) | (y[1] << 16);
    w[5] = (y[1] >> 16) | (z[1] << 16);
    w[6] = (z[1] >> 16) | (rt[1] << 16);
}

// ---- point pair load / store ------------------------------------------------------------
template <bool F64, bool FULL>
__device__ __forceinline__ void load_pair(const void* base, int64_t p, bool va, bool vb, Pt& a, Pt& b) {
    if constexpr (F64) {
        const double* src = reinterpret_cast<const double*>(base) + 4 * p;
        if (FULL || va) ldg256(src, a.x, a.y, a.z, a.w);
        if (FULL || vb) ldg256(src + 4, b.x, b.y, b.z, b.w);
    } else {
        const float* src = reinterpret_cast<const float*>(base) + 4 * p;
        if (FULL || (va && vb)) {
            float v[8];
            ldg256(src, v);
            a = { (double)v[0], (double)v[1], (double)v[2], (double)v[3] };
            b = { (double)v[4], (double)v[5], (double)v[6], (double)v[7] };
        } else {
            if (va) { const float4 v = __ldg(reinterpret_cast<const float4*>(src));     a = { (double)v.x, (double)v.y, (double)v.z, (double)v.w }; }
            if (vb) { const float4 v = __ldg(reinterpret_cast<const float4*>(src) + 1); b = { (double)v.x, (double)v.y, (double)v.z, (double)v.w }; }
        }
    }
}

template <bool F64, bool FULL>
__device__ __forceinline__ void store_pair(void* base, int64_t p, bool va, bool vb, const Pt& a, const Pt& b) {
    if constexpr (F64) {
        double* dst = reinterpret_cast<double*>(base) + 4 * p;
        if (FULL || va) stg256(dst, a.x, a.y, a.z, a.w);
        if (FULL || vb) stg256(dst + 4, b.x, b.y, b.z, b.w);
    } else {
        float* dst = reinterpret_cast<float*>(base) + 4 * p;
        if (FULL || (va && vb)) {
            const float v[8] = { (float)a.x, (float)a.y, (float)a.z, (float)a.w, (float)b.x, (float)b.y, (float)b.z, (float)b.w };
            stg256(dst, v);
        } else {
            if (va) *reinterpret_cast<float4*>(dst)     = make_float4((float)a.x, (float)a.y, (float)a.z, (float)a.w);
            if (vb) *reinterpret_cast<float4*>(dst + 4) = make_float4((float)b.x, (float)b.y, (float)b.z, (float)b.w);
        }
    }
}

// LAS integer stores of one pair (SoA, 64-bit per array for a full pair)
template <bool FULL, bool OOL = true>
__device__ __forceinline__ void store_las_pair(const Params& P, int64_t p, bool va, bool vb, const Pt& a, const Pt& b, uint32_t& fl) {
    if (P.las_x != nullptr) {
        int32_t X[2] = {0, 0}, Y[2] = {0, 0}, Z[2] = {0, 0};
        if (FULL || va) { X[0] = q_las<OOL>(a.x, P.las_scale[0], P.las_rcp[0], P.las_off[0], fl); Y[0] = q_las<OOL>(a.y, P.las_scale[1], P.las_rcp[1], P.las_off[1], fl); Z[0] = q_las<OOL>(a.z, P.las_scale[2], P.las_rcp[2], P.las_off[2], fl); }
        if (FULL || vb) { X[1] = q_las<OOL>(b.x, P.las_scale[0], P.las_rcp[0], P.las_off[0], fl); Y[1] = q_las<OOL>(b.y, P.las_scale[1], P.las_rcp[1], P.las_off[1], fl); Z[1] = q_las<OOL>(b.z, P.las_scale[2], P.las_rcp[2], P.las_off[2], fl); }
        if (FULL || (va && vb)) {
            *reinterpret_cast<int2*>(P.las_x + p) = make_int2(X[0], X[1]);
            *reinterpret_cast<int2*>(P.las_y + p) = make_int2(Y[0], Y[1]);
            *reinterpret_cast<int2*>(P.las_z + p) = make_int2(Z[0], Z[1]);
        } else {
            if (va) { P.las_x[p] = X[0]; P.las_y[p] = Y[0]; P.las_z[p] = Z[0]; }
            if (vb) { P.las_x[p + 1] = X[1]; P.las_y[p + 1] = Y[1]; P.las_z[p + 1] = Z[1]; }
        }
    }
    if (P.las_int != nullptr) {
        uint32_t i0 = 0, i1 = 0;
        if (FULL || va) i0 = q_las_intensity(a.w, P.las_int_mode, fl);
        if (FULL || vb) i1 = q_las_intensity(b.w, P.las_int_mode, fl);
        if (FULL || (va && vb)) *reinterpret_cast<uint32_t*>(P.las_int + p) = i0 | (i1 << 16);
        else { if (va) P.las_int[p] = (uint16_t)i0; if (vb) P.las_int[p + 1] = (uint16_t)i1; }
    }
}

}  // namespace lmc
