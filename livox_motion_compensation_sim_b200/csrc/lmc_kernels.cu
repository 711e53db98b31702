// lmc_kernels.cu -- "direct" kernels: one 1024-point tile per CTA, 256-bit LDG/STG, fused
// pose lookup + transform + quantise.  The TMA bulk-copy pipelined variant lives in lmc_tma.cu.
//
// Data flow of one CTA (tile = 1024 consecutive points of the merged, frame-major cloud):
//   1. every thread issues its 256-bit point loads (2 pairs of consecutive points) -- no
//      dependence on frame lookup, so the DRAM latency overlaps step 2
//   2. warp 0 finds the frames intersecting the tile: one 32-ary search of the CSR offsets
//      (3 dependent L2 loads for 36 000 frames) + one coalesced read of the following offsets
//   3. per point: frame -> pose (L1 broadcast) -> f64 transform in the reference's op order
//   4. aligned points leave as 256-bit stores; LAS ints as 64-bit SoA stores; LVX 14-byte
//      records are assembled as 7 words per point pair in shared memory (stride 7 words is
//      coprime with 32 banks: conflict-free) and leave as one TMA bulk store per tile
//
//   LMC = lidar_motion_compensation.py        CS = livox_mid70_complete_simulator.py
#include "lmc_device.cuh"

namespace lmc {

constexpr int kThreads        = 256;                       // 8 warps per CTA
constexpr int kPairsPerThread = 2;                         // each thread owns 2 pairs of consecutive points
constexpr int kTilePairs      = kThreads * kPairsPerThread;
constexpr int kTile           = 2 * kTilePairs;            // 1024 points per tile

// ---- fused kernel body ---------------------------------------------------------------------
template <bool F64, int MODE, bool FULL>
__device__ __forceinline__ void tile_body(const Params& P, int64_t base, int64_t lim_lo, int64_t lim_hi,
                                          uint32_t* s_lvx, TileMeta& s_tm)
{
    const int tid = threadIdx.x, lane = tid & 31;

    // ---- 1. loads --------------------------------------------------------------------------
    Pt in[kPairsPerThread][2];
    bool valid[kPairsPerThread][2];
    int64_t tsv[kPairsPerThread][2];
    uint32_t tagv[kPairsPerThread];
#pragma unroll
    for (int j = 0; j < kPairsPerThread; ++j) {
        const int64_t p = base + 2 * (tid + j * kThreads);
        const bool va = FULL || (p >= lim_lo && p < lim_hi), vb = FULL || (p + 1 >= lim_lo && p + 1 < lim_hi);
        valid[j][0] = va; valid[j][1] = vb;
        in[j][0] = in[j][1] = Pt{ 0.0, 0.0, 0.0, 0.0 };
        load_pair<F64, FULL>(P.pts, p, va, vb, in[j][0], in[j][1]);
        tsv[j][0] = tsv[j][1] = 0;
        if constexpr (MODE == kGyro || kSlerpFamily<MODE>) {
            if (P.ts != nullptr) {
                if constexpr (F64) {
                    const int64_t* t = reinterpret_cast<const int64_t*>(P.ts) + p;
                    if (va && vb) { const longlong2 v = __ldg(reinterpret_cast<const longlong2*>(t)); tsv[j][0] = v.x; tsv[j][1] = v.y; }
                    else { if (va) tsv[j][0] = __ldg(t); if (vb) tsv[j][1] = __ldg(t + 1); }
                } else {
                    const uint32_t* t = reinterpret_cast<const uint32_t*>(P.ts) + p;
                    if (va && vb) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(t)); tsv[j][0] = v.x; tsv[j][1] = v.y; }
                    else { if (va) tsv[j][0] = __ldg(t); if (vb) tsv[j][1] = __ldg(t + 1); }
                }
            }
        }
        tagv[j] = 0;
        if (P.lvx14 != nullptr && P.tag != nullptr && P.lvx_mode == LMC_LVX2_OF_OUTPUT) {
            if (va) tagv[j] |= __ldg(P.tag + p);
            if (vb) tagv[j] |= (uint32_t)__ldg(P.tag + p + 1) << 8;
        }
    }

    // ---- 2. frames intersecting the tile ------------------------------------------------------
    if constexpr (MODE != kQuantOnly) {
        if (tid < 32) tile_meta(P, lim_lo, lim_hi - 1, s_tm, lane);
        __syncthreads();
    }

    // ---- 3. compute ---------------------------------------------------------------------------
    Pt outp[kPairsPerThread][2];
    uint32_t fl = 0;
    PointCtx<F64, MODE> ctx;
    ctx.init(P);
#pragma unroll
    for (int j = 0; j < kPairsPerThread; ++j) {
        int32_t f[2] = {0, 0}; bool single[2] = {false, false}; int64_t fs[2] = {0, 0};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            outp[j][h] = in[j][h];
            if constexpr (MODE != kQuantOnly) {
                if (FULL || valid[j][h]) {
                    f[h] = frame_of(P, s_tm, base + 2 * (tid + j * kThreads) + h, single[h]);
                    if constexpr (MODE == kGyro || kSlerpFamily<MODE>) { if (P.frame_start != nullptr) fs[h] = frame_start_of(P, s_tm, f[h]); }
                }
            }
        }
        if (FULL || (valid[j][0] && valid[j][1])) ctx.pair(P, f, single, fs, tsv[j], in[j], outp[j]);
        else {
            if (valid[j][0]) outp[j][0] = ctx.one(P, f[0], single[0], fs[0], tsv[j][0], in[j][0]);
            if (valid[j][1]) outp[j][1] = ctx.one(P, f[1], single[1], fs[1], tsv[j][1], in[j][1]);
        }
    }

    // ---- 4. stores + export epilogues ---------------------------------------------------------
#pragma unroll
    for (int j = 0; j < kPairsPerThread; ++j) {
        const int q = tid + j * kThreads;
        const int64_t p = base + 2 * q;
        const bool va = valid[j][0], vb = valid[j][1];
        if (P.out != nullptr) store_pair<F64, FULL>(P.out, p, va, vb, outp[j][0], outp[j][1]);
        store_las_pair<FULL>(P, p, va, vb, outp[j][0], outp[j][1], fl);
        if (P.lvx14 != nullptr) {
            uint32_t x[2] = {0, 0}, y[2] = {0, 0}, z[2] = {0, 0}, rt[2] = {0, 0};
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (FULL || valid[j][h]) lvx_words<MODE>(P, in[j][h], outp[j][h], (tagv[j] >> (8 * h)) & 0xffu, x[h], y[h], z[h], rt[h], fl);
            lvx_pair_words(s_lvx + 7 * q, x, y, z, rt);              // 28 B per pair, conflict-free stride
        }
    }

    if (P.lvx14 != nullptr)      // bytes [b0, b1) of the tile's record block: one TMA bulk store for the 16-byte body, byte-wise ragged ends
        cta_image_out(P.lvx14 + 14 * base, reinterpret_cast<const uint8_t*>(s_lvx), (int)(lim_lo - base) * 14, (int)(lim_hi - base) * 14, tid, kThreads);
    if (fl != 0 && P.status != nullptr) atomicOr(P.status, fl);
}

template <bool F64, int MODE>
__global__ void __launch_bounds__(kThreads, 2) k_fused(const __grid_constant__ Params P)
{
    __shared__ __align__(16) uint32_t s_lvx[kTilePairs * 7];      // 1024 x 14 B records
    __shared__ TileMeta s_tm;
    const int64_t tile0 = (P.p_begin / kTile) * kTile;            // tiles are aligned in GLOBAL index space
    const int64_t base  = tile0 + (int64_t)blockIdx.x * kTile;
    const int64_t lim_lo = base > P.p_begin ? base : P.p_begin;
    const int64_t lim_hi = base + kTile < P.p_end ? base + kTile : P.p_end;
    if (lim_lo >= lim_hi) return;
    if (lim_lo == base && lim_hi == base + kTile) tile_body<F64, MODE, true>(P, base, lim_lo, lim_hi, s_lvx, s_tm);
    else                                          tile_body<F64, MODE, false>(P, base, lim_lo, lim_hi, s_lvx, s_tm);
}

// (a1) LMC:802-812: one thread per frame
__global__ void k_pose_lookup(const double* __restrict__ traj_t, int64_t n_t, const double* __restrict__ traj_Rt,
                              const double* __restrict__ frame_t, int32_t n_frames,
                              double* __restrict__ pose_Rt, int32_t* __restrict__ pose_idx)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    const double t = frame_t[f];
    int64_t lo = 0, hi = n_t;                       // np.searchsorted side='left'
    while (lo < hi) { const int64_t mid = lo + ((hi - lo) >> 1); if (traj_t[mid] < t) lo = mid + 1; else hi = mid; }
    if (lo > n_t - 1) lo = n_t - 1;
    if (lo < 0) lo = 0;
    const double2* src = reinterpret_cast<const double2*>(traj_Rt + 12 * lo);
    double2* dst = reinterpret_cast<double2*>(pose_Rt + 12 * (int64_t)f);
#pragma unroll
    for (int q = 0; q < 6; ++q) dst[q] = __ldg(src + q);
    if (pose_idx) pose_idx[f] = (int32_t)lo;
}

// (north_star subsystem 1) the pose-segment table of Mode C, one thread per sample: what
// frames.slerp_segment_table builds on the host with SciPy (1.7 s for a 1 h / 200 Hz stream), as a kernel.
//   row k = [R_k (9) | pos_k (3) | unit axis of R_k^-1 R_{k+1} (3) | angle | pos_{k+1} - pos_k (3) | 1/dt_k | t_k bits | dt_k bits]
// R_k from the normalised quaternion with SciPy's as_matrix formula; the relative rotation
// q_k^-1 (x) q_{k+1} gives axis = v/|v| and angle = 2 atan2(|v|, w) (w >= 0), i.e. as_rotvec's angle.
__global__ void k_slerp_table(const double* __restrict__ quat, const double* __restrict__ pos, const int64_t* __restrict__ ts,
                              int64_t S, double* __restrict__ seg)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= S) return;
    double q[2][4];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int64_t i = k + j < S ? k + j : k;
        const double2 a = __ldg(reinterpret_cast<const double2*>(quat + 4 * i)), b = __ldg(reinterpret_cast<const double2*>(quat + 4 * i) + 1);
        const double n = sqrt(a.x * a.x + a.y * a.y + b.x * b.x + b.y * b.y);
        q[j][0] = a.x / n; q[j][1] = a.y / n; q[j][2] = b.x / n; q[j][3] = b.y / n;
    }
    double row[kSegStride];
    {
        const double x = q[0][0], y = q[0][1], z = q[0][2], w = q[0][3];
        const double x2 = x * x, y2 = y * y, z2 = z * z, w2 = w * w, xy = x * y, zw = z * w, xz = x * z, yw = y * w, yz = y * z, xw = x * w;
        row[0] = x2 - y2 - z2 + w2; row[1] = 2.0 * (xy - zw);      row[2] = 2.0 * (xz + yw);
        row[3] = 2.0 * (xy + zw);    row[4] = -x2 + y2 - z2 + w2;  row[5] = 2.0 * (yz - xw);
        row[6] = 2.0 * (xz - yw);    row[7] = 2.0 * (yz + xw);     row[8] = -x2 - y2 + z2 + w2;
    }
    const double p0 = pos[3 * k], p1 = pos[3 * k + 1], p2 = pos[3 * k + 2];
    row[9] = p0; row[10] = p1; row[11] = p2;
    row[12] = 1.0; row[13] = 0.0; row[14] = 0.0; row[15] = 0.0; row[16] = 0.0; row[17] = 0.0; row[18] = 0.0; row[19] = 0.0;
    const int64_t tk = ts[k];
    int64_t dt = 0;
    if (k + 1 < S) {
        // q_rel = conj(q_k) (x) q_{k+1}
        const double ax = -q[0][0], ay = -q[0][1], az = -q[0][2], aw = q[0][3];
        const double bx = q[1][0], by = q[1][1], bz = q[1][2], bw = q[1][3];
        // separately rounded products (no FMA contraction): identical samples cancel to an exact zero rotation
        double vx = __dadd_rn(__dadd_rn(__dmul_rn(aw, bx), __dmul_rn(ax, bw)), __dsub_rn(__dmul_rn(ay, bz), __dmul_rn(az, by)));
        double vy = __dadd_rn(__dadd_rn(__dmul_rn(aw, by), __dmul_rn(ay, bw)), __dsub_rn(__dmul_rn(az, bx), __dmul_rn(ax, bz)));
        double vz = __dadd_rn(__dadd_rn(__dmul_rn(aw, bz), __dmul_rn(az, bw)), __dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx)));
        double w  = __dsub_rn(__dsub_rn(__dmul_rn(aw, bw), __dmul_rn(ax, bx)), __dadd_rn(__dmul_rn(ay, by), __dmul_rn(az, bz)));
        if (w < 0.0) { vx = -vx; vy = -vy; vz = -vz; w = -w; }
        const double vn = sqrt(vx * vx + vy * vy + vz * vz);
        const double th = 2.0 * atan2(vn, w);
        if (th > 0.0 && vn > 0.0) { row[12] = vx / vn; row[13] = vy / vn; row[14] = vz / vn; }
        row[15] = th;
        row[16] = pos[3 * k + 3] - p0; row[17] = pos[3 * k + 4] - p1; row[18] = pos[3 * k + 5] - p2;
        dt = ts[k + 1] - tk;
        row[19] = dt > 0 ? 1.0 / (double)dt : 0.0;
    }
    row[20] = __longlong_as_double(tk);
    row[21] = __longlong_as_double(dt);
    double2* dst = reinterpret_cast<double2*>(seg + kSegStride * k);
#pragma unroll
    for (int j = 0; j < kSegStride / 2; ++j) dst[j] = make_double2(row[2 * j], row[2 * j + 1]);
}

// Pose at a time (definition: oracle/lmc_oracle_local.c::orc_slerp_pose_at), one thread per query: Mode C's bracket, clamps and
// alpha, then column j of R(t) = R_k (Rodrigues step of e_j) and pos(t) = pos_k + alpha dpos_k -- 12 doubles laid out as a
// Mode A pose row.
__global__ void k_slerp_pose_at(const int64_t* __restrict__ sample_ts, const double* __restrict__ seg, int64_t S,
                                const int64_t* __restrict__ query_ts, int64_t n_query, double* __restrict__ pose)
{
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_query) return;
    const int64_t t0 = __ldg(sample_ts), span = __ldg(sample_ts + S - 1) - t0;
    const double rate = span > 0 ? (double)(S - 1) / (double)span : 0.0;
    const int64_t t = __ldg(query_ts + q);
    const Bracket b = bracket_of(sample_ts, S, t, t0, rate);
    int64_t k = b.k; double alpha = 0.0;
    if (k < 0) k = 0;
    else if (k >= S - 1) k = S - 1;
    else alpha = (double)(t - b.tb);
    double row[kSegStride];
    const double2* sr = reinterpret_cast<const double2*>(seg + kSegStride * k);
#pragma unroll
    for (int j = 0; j < kSegStride / 2; ++j) { const double2 v = __ldg(sr + j); row[2 * j] = v.x; row[2 * j + 1] = v.y; }
    alpha = __dmul_rn(alpha, row[19]);
    double M[12];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        double x1, y1, z1;
        slerp_rotate<false>(row, alpha, j == 0 ? 1.0 : 0.0, j == 1 ? 1.0 : 0.0, j == 2 ? 1.0 : 0.0, x1, y1, z1);
#pragma unroll
        for (int r = 0; r < 3; ++r) M[3 * r + j] = dot_gemm(row[3 * r], x1, row[3 * r + 1], y1, row[3 * r + 2], z1);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) M[9 + r] = __fma_rn(alpha, row[16 + r], row[9 + r]);
    double2* dst = reinterpret_cast<double2*>(pose + 12 * q);
#pragma unroll
    for (int j = 0; j < 6; ++j) dst[j] = make_double2(M[2 * j], M[2 * j + 1]);
}

// ---- launchers -------------------------------------------------------------------------------
template <bool F64, int MODE>
static cudaError_t launch_fused(const Params& P, cudaStream_t st) {
    if (P.p_end <= P.p_begin) return cudaSuccess;
    const int64_t tile0 = (P.p_begin / kTile) * kTile;
    const int64_t tiles = (P.p_end - tile0 + kTile - 1) / kTile;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    k_fused<F64, MODE><<<(unsigned)tiles, kThreads, 0, st>>>(P);
    return cudaGetLastError();
}

cudaError_t launch_direct(bool f64, int mode, const Params& P, cudaStream_t st) {
    return dispatch_layout_mode(f64, mode, [&](auto f64_c, auto mode_c) {
        return launch_fused<decltype(f64_c)::value, decltype(mode_c)::value>(P, st);
    });
}

cudaError_t launch_pose_lookup(const double* traj_t, int64_t n_t, const double* traj_Rt, const double* frame_t,
                               int32_t n_frames, double* pose_Rt, int32_t* pose_idx, cudaStream_t st) {
    if (n_frames <= 0) return cudaSuccess;
    k_pose_lookup<<<(n_frames + 127) / 128, 128, 0, st>>>(traj_t, n_t, traj_Rt, frame_t, n_frames, pose_Rt, pose_idx);
    return cudaGetLastError();
}

cudaError_t launch_slerp_pose_at(const int64_t* sample_ts, const double* seg, int64_t S, const int64_t* query_ts, int64_t n_query,
                                 double* pose, cudaStream_t st) {
    if (n_query <= 0) return cudaSuccess;
    const int64_t blocks = (n_query + 127) / 128;
    if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
    k_slerp_pose_at<<<(unsigned)blocks, 128, 0, st>>>(sample_ts, seg, S, query_ts, n_query, pose);
    return cudaGetLastError();
}

cudaError_t launch_slerp_table(const double* quat, const double* pos, const int64_t* ts, int64_t S, double* seg, cudaStream_t st) {
    if (S <= 0) return cudaSuccess;
    const int64_t blocks = (S + 127) / 128;
    if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
    k_slerp_table<<<(unsigned)blocks, 128, 0, st>>>(quat, pos, ts, S, seg);
    return cudaGetLastError();
}

}  // namespace lmc
