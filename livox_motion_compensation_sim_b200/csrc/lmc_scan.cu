// lmc_scan.cu -- (SURVEY 8f N4) LiDARMotionSimulator.scan_environment (LMC:701-770) for every frame of
// a run at once: range cull, world -> sensor rotation, FOV cull, order-preserving compaction and the
// systematic subsample.  This is 90 % of the reference's run_simulation wall time.
//
// The one thing that stays on the host is the noise: the reference draws it from the seeded GLOBAL
// NumPy RNG (np.random.normal sized by each frame's visible count, LMC:765-768), so the caller reads
// the per-frame counts back, draws the identical stream in one call, and k_scan_emit adds it.
//
// Arithmetic in the reference's order: d2 = (dx*dx + dy*dy) + dz*dz (np.sum over 3 columns),
// rotated = R^T t through dgemm (k = 0,1,2 FMA chain from +0.0 -- also for a single column, measured),
// az = atan2(y,x)*180/pi, el = asin(clip(z / max(sqrt(d2),1e-6), -1, 1))*180/pi.  Coordinates are
// bit-exact.  The FOV decisions could differ from NumPy's only for a point within a few ulp of the FOV
// edge (device atan2/asin vs the host libm): k_scan_mark therefore marks every point whose |azimuth| or
// |elevation| lies within edge_eps degrees of the limit as UNCERTAIN (flag bit 1) and counts them; the
// caller re-decides exactly those on the host with the reference's own NumPy calls, patches the flags
// and calls lmc_scan_recount.  (In the golden runs -- 1.8 M emitted points -- no point is uncertain.)
//
//   k_scan_mark     grid (tile, frame): visibility flag per (frame, env point) + per-tile counts
//   k_scan_count    grid (tile, frame): per-tile counts again from (host-patched) flags
//   k_scan_offsets  grid (frame): exclusive scan of the tile counts, visible total per frame
//   k_scan_emit     grid (tile, frame): compaction rank -> subsample rule -> rotated xyz (+ noise), intensity; or (<true>) the
//                   environment row index of every emitted point
#include "lmc_device.cuh"

namespace lmc {

constexpr int kScanTile = 256;

struct ScanGeom { double x, y, z, d2; bool in_range; };

__device__ __forceinline__ ScanGeom scan_geom(const double* __restrict__ env, int64_t i, const double* __restrict__ pos,
                                              const double* __restrict__ R, double rmax2) {
    ScanGeom g;
    double ex, ey, ez, ew;
    ldg256(env + 4 * i, ex, ey, ez, ew);
    const double dx = __dsub_rn(ex, pos[0]), dy = __dsub_rn(ey, pos[1]), dz = __dsub_rn(ez, pos[2]);
    g.d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));     // LMC:713
    g.in_range = g.d2 <= rmax2;                                                                // LMC:717
    // (R^T t)[r] = sum_k R[k][r] t[k]                                                         // LMC:726-728
    // accumulated from +0.0 as dgemm does: three -0.0 products then sum to +0.0, not -0.0 (atan2 would turn that into 180 deg)
    g.x = __fma_rn(R[6], dz, __fma_rn(R[3], dy, __fma_rn(R[0], dx, 0.0)));
    g.y = __fma_rn(R[7], dz, __fma_rn(R[4], dy, __fma_rn(R[1], dx, 0.0)));
    g.z = __fma_rn(R[8], dz, __fma_rn(R[5], dy, __fma_rn(R[2], dx, 0.0)));
    return g;
}

__device__ __forceinline__ bool scan_visible(const ScanGeom& g, double fov_h_half, double fov_v_half, double range_min, double edge_eps,
                                             bool& uncertain) {
    uncertain = false;
    if (!g.in_range) return false;
    const double pi = 3.141592653589793;
    const double rng = sqrt(g.d2);                                                             // LMC:732
    const double az = __ddiv_rn(__dmul_rn(atan2(g.y, g.x), 180.0), pi);                        // LMC:735
    const double sr = rng > 1e-6 ? rng : 1e-6;
    double q = __ddiv_rn(g.z, sr);
    q = q < -1.0 ? -1.0 : (q > 1.0 ? 1.0 : q);
    const double el = __ddiv_rn(__dmul_rn(asin(q), 180.0), pi);                                // LMC:738
    uncertain = rng >= range_min && (fabs(fabs(az) - fov_h_half) <= edge_eps || fabs(fabs(el) - fov_v_half) <= edge_eps);
    return fabs(az) <= fov_h_half && fabs(el) <= fov_v_half && rng >= range_min;               // LMC:743-745
}

__device__ __forceinline__ int block_count_and_rank(bool flag, int* s_warp, int& total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) s_warp[w] = __popc(m);
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < kScanTile / 32; ++k) { const int c = s_warp[k]; if (k < w) base += c; tot += c; }
    total = tot;
    return base + __popc(m & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(kScanTile) k_scan_mark(const double* __restrict__ env, int64_t M, const double* __restrict__ pos_f3,
                                                         const double* __restrict__ R_f9, double rmax2, double fov_h_half, double fov_v_half,
                                                         double range_min, double edge_eps, uint8_t* __restrict__ flags, int32_t* __restrict__ tile_off,
                                                         int tiles, int32_t* __restrict__ n_uncertain) {
    __shared__ int s_warp[kScanTile / 32];
    const int f = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * kScanTile + threadIdx.x;
    bool vis = false;
    if (i < M) {
        const ScanGeom g = scan_geom(env, i, pos_f3 + 3 * f, R_f9 + 9 * f, rmax2);
        bool unc;
        vis = scan_visible(g, fov_h_half, fov_v_half, range_min, edge_eps, unc);
        flags[(int64_t)f * M + i] = (vis ? 1 : 0) | (unc ? 2 : 0);
        if (unc && n_uncertain != nullptr) atomicAdd(n_uncertain, 1);
    }
    int total;
    block_count_and_rank(vis, s_warp, total);
    if (threadIdx.x == 0) tile_off[(int64_t)f * (tiles + 1) + blockIdx.x + 1] = total;         // counts now, offsets after the scan
}

// per-tile counts from the flags (bit 0), after the host re-decided the uncertain points
__global__ void __launch_bounds__(kScanTile) k_scan_count(const uint8_t* __restrict__ flags, int64_t M, int32_t* __restrict__ tile_off, int tiles) {
    __shared__ int s_warp[kScanTile / 32];
    const int f = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * kScanTile + threadIdx.x;
    const bool vis = i < M && (flags[(int64_t)f * M + i] & 1) != 0;
    int total;
    block_count_and_rank(vis, s_warp, total);
    if (threadIdx.x == 0) tile_off[(int64_t)f * (tiles + 1) + blockIdx.x + 1] = total;
}

__global__ void k_scan_offsets(int32_t* __restrict__ tile_off, int tiles, int32_t* __restrict__ n_visible) {
    const int f = blockIdx.x;
    if (threadIdx.x != 0) return;
    int32_t* t = tile_off + (int64_t)f * (tiles + 1);
    int acc = 0;
    t[0] = 0;
    for (int k = 0; k < tiles; ++k) { acc += t[k + 1]; t[k + 1] = acc; }
    n_visible[f] = acc;
}

// IDX = false: raw_out rows (rotated xyz + noise, intensity).  IDX = true: the environment row of every emitted point instead
// (idx_out[o] = i), the same compaction and subsample -- for the caller that re-observes the points from other poses.
template <bool IDX>
__global__ void __launch_bounds__(kScanTile) k_scan_emit(const double* __restrict__ env, int64_t M, const double* __restrict__ pos_f3,
                                                         const double* __restrict__ R_f9, double rmax2, const uint8_t* __restrict__ flags,
                                                         const int32_t* __restrict__ tile_off, int tiles, const int32_t* __restrict__ n_visible,
                                                         const int64_t* __restrict__ frame_off, int32_t max_points,
                                                         const double* __restrict__ noise, double* __restrict__ out, int64_t* __restrict__ idx_out) {
    __shared__ int s_warp[kScanTile / 32];
    const int f = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * kScanTile + threadIdx.x;
    const bool vis = i < M && (flags[(int64_t)f * M + i] & 1) != 0;
    int total;
    const int rank = block_count_and_rank(vis, s_warp, total);
    if (!vis) return;
    const int j = tile_off[(int64_t)f * (tiles + 1) + blockIdx.x] + rank;                      // index among the frame's visible points
    const int n = n_visible[f];
    int64_t o = j;
    if (n > max_points) {                                                                      // LMC:756-761 systematic subsample
        const int step = n / max_points;
        if (j % step != 0 || j / step >= max_points) return;
        o = j / step;
    }
    o += frame_off[f];
    if constexpr (IDX) {
        idx_out[o] = i;
    } else {
        const ScanGeom g = scan_geom(env, i, pos_f3 + 3 * f, R_f9 + 9 * f, rmax2);
        double nx = 0.0, ny = 0.0, nz = 0.0;
        if (noise != nullptr) { nx = noise[3 * o]; ny = noise[3 * o + 1]; nz = noise[3 * o + 2]; }
        const double w = env[4 * i + 3];
        if (noise != nullptr) stg256(out + 4 * o, __dadd_rn(g.x, nx), __dadd_rn(g.y, ny), __dadd_rn(g.z, nz), w);   // LMC:768 visible_points += noise
        else                  stg256(out + 4 * o, g.x, g.y, g.z, w);
    }
}

// grid.y carries the frame index (<= 65535 per launch): longer runs go in frame chunks
constexpr int kScanMaxFramesPerLaunch = 65535;

cudaError_t launch_scan_mark(const double* env, int64_t M, const double* pos, const double* R, int32_t F, double rmax2, double fh, double fv,
                             double rmin, double edge_eps, uint8_t* flags, int32_t* tile_off, int32_t* n_visible, int32_t* n_uncertain, cudaStream_t st) {
    if (n_uncertain != nullptr) { cudaError_t e = cudaMemsetAsync(n_uncertain, 0, sizeof(int32_t), st); if (e != cudaSuccess) return e; }
    const int64_t tiles = (M + kScanTile - 1) / kScanTile;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    for (int32_t f0 = 0; f0 < F; f0 += kScanMaxFramesPerLaunch) {
        const int nf = F - f0 < kScanMaxFramesPerLaunch ? F - f0 : kScanMaxFramesPerLaunch;
        int32_t* toff = tile_off + (int64_t)f0 * (tiles + 1);
        if (tiles > 0) k_scan_mark<<<dim3((unsigned)tiles, (unsigned)nf), kScanTile, 0, st>>>(env, M, pos + 3 * (int64_t)f0, R + 9 * (int64_t)f0, rmax2, fh, fv, rmin,
                                                                                             edge_eps, flags + (int64_t)f0 * M, toff, (int)tiles, n_uncertain);
        k_scan_offsets<<<nf, 32, 0, st>>>(toff, (int)tiles, n_visible + f0);
    }
    return cudaGetLastError();
}

cudaError_t launch_scan_recount(const uint8_t* flags, int64_t M, int32_t F, int32_t* tile_off, int32_t* n_visible, cudaStream_t st) {
    const int64_t tiles = (M + kScanTile - 1) / kScanTile;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    for (int32_t f0 = 0; f0 < F; f0 += kScanMaxFramesPerLaunch) {
        const int nf = F - f0 < kScanMaxFramesPerLaunch ? F - f0 : kScanMaxFramesPerLaunch;
        int32_t* toff = tile_off + (int64_t)f0 * (tiles + 1);
        if (tiles > 0) k_scan_count<<<dim3((unsigned)tiles, (unsigned)nf), kScanTile, 0, st>>>(flags + (int64_t)f0 * M, M, toff, (int)tiles);
        k_scan_offsets<<<nf, 32, 0, st>>>(toff, (int)tiles, n_visible + f0);
    }
    return cudaGetLastError();
}

cudaError_t launch_scan_emit(const double* env, int64_t M, const double* pos, const double* R, int32_t F, double rmax2, const uint8_t* flags,
                             const int32_t* tile_off, const int32_t* n_visible, const int64_t* frame_off, int32_t max_points,
                             const double* noise, double* out, int64_t* idx_out, cudaStream_t st) {
    const int64_t tiles = (M + kScanTile - 1) / kScanTile;
    if (tiles == 0) return cudaSuccess;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    for (int32_t f0 = 0; f0 < F; f0 += kScanMaxFramesPerLaunch) {
        const int nf = F - f0 < kScanMaxFramesPerLaunch ? F - f0 : kScanMaxFramesPerLaunch;
        const dim3 grid((unsigned)tiles, (unsigned)nf);
        if (idx_out != nullptr)
            k_scan_emit<true><<<grid, kScanTile, 0, st>>>(env, M, pos + 3 * (int64_t)f0, R + 9 * (int64_t)f0, rmax2, flags + (int64_t)f0 * M,
                                                          tile_off + (int64_t)f0 * (tiles + 1), (int)tiles, n_visible + f0, frame_off + f0,
                                                          max_points, nullptr, nullptr, idx_out);
        else
            k_scan_emit<false><<<grid, kScanTile, 0, st>>>(env, M, pos + 3 * (int64_t)f0, R + 9 * (int64_t)f0, rmax2, flags + (int64_t)f0 * M,
                                                           tile_off + (int64_t)f0 * (tiles + 1), (int)tiles, n_visible + f0, frame_off + f0,
                                                           max_points, noise, out, nullptr);
    }
    return cudaGetLastError();
}

}  // namespace lmc
