// lmc_register.cu -- a prior point map on the device: exact fixed-radius nearest neighbours through a voxel hash, and
// per-frame point-to-point Gauss-Newton pose refinement against it (definition: oracle/lmc_oracle_register.py).
//
// Map: the points sorted by voxel (f64 rows + original index), CSR voxel offsets, and an open-addressing table
// key -> voxel rank (capacity the power of two >= 2V, linear probing) that k_map_insert fills from each voxel's first
// row.  Keys come from vox_point (lmc_voxel.cuh), the voxel map's own expressions.
// Nearest: the query's cell, then the 27 cells around it; d = w - m and d2 = (dx dx + dy dy) + dz dz, every operation
// rounded to nearest (no contraction); accepted when d2 <= r2; the minimum over (d2, original index).
// Register, per iteration (no host synchronisation inside the loop):
//   k_reg_accum  one CTA per (frame, 256-point chunk): a = R p, w = a + t, its nearest map point q, r = w - q; 17 f64
//                sums of the inliers, reduced shuffle-then-warp in a fixed order, one partial per chunk
//   k_reg_solve  one warp per frame: the chunk partials in chunk order, the 6x6 normal equations, Cholesky, update
//                t <- t + tau, R <- Exp(phi) R (rotation about the sensor position, so H stays well conditioned)
// Normals: k_map_normals, one thread per map row: the ball of radius r around it, its covariance, a cyclic Jacobi
// eigen-decomposition, (normal, planarity).  Point-to-plane registration: k_reg_accum_plane / k_reg_solve_plane, the
// same two launches per iteration with the residual along the nearest map row's normal (29 sums)
// (definition: oracle/lmc_oracle_plane.py).
#include "lmc_voxel.cuh"

namespace lmc {
cudaError_t launch_tile_scan(int64_t* tile_off, int64_t tiles, cudaStream_t st);    // lmc_pcd.cu

constexpr int kRegTile = 256;                        // points (= threads) per chunk
constexpr int kRegSums = 17;                         // n, Sa(3), Saa(6: xx xy xz yy yz zz), Sr(3), S a x r(3), S |r|^2
constexpr int kRegPlaneSums = 29;                    // n, H = S J J^T (21: upper triangle, row-major), g = S J e (6), S e^2
constexpr int32_t kRegConverged = 1, kRegDegenerate = 2;
constexpr uint32_t kMapNoRank = ~0u;

struct MapView {
    const double* pts;              // [M][4] rows sorted by voxel
    const int64_t* idx;             // [M] original row of each sorted row
    const int64_t* vox_off;         // [V + 1]
    const unsigned long long* keys; // [cap] packed key, kVoxEmpty
    const uint32_t* rank;           // [cap] voxel rank of the slot
    uint64_t cap;
    VoxGrid G;
    double r2;
};

static inline size_t reg_align(size_t b) { return (b + 255) & ~size_t(255); }
size_t map_table_bytes(int64_t V) { const uint64_t cap = vox_cap(V); return reg_align(8 * cap) + reg_align(4 * cap); }

static MapView map_view(const double* pts, const int64_t* idx, const int64_t* vox_off, const void* table, int64_t V,
                        const double* leaf, const double* origin, double r2) {
    MapView M;
    M.pts = pts; M.idx = idx; M.vox_off = vox_off; M.cap = vox_cap(V); M.r2 = r2;
    M.keys = static_cast<const unsigned long long*>(table);
    M.rank = reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(table) + reg_align(8 * M.cap));
    for (int c = 0; c < 3; ++c) { M.G.o[c] = origin[c]; M.G.L[c] = leaf[c]; }
    return M;
}

__global__ void __launch_bounds__(kRegTile) k_map_insert(const double* __restrict__ pts, const int64_t* __restrict__ vox_off, int64_t V,
                                                         const VoxGrid G, unsigned long long* __restrict__ keys,
                                                         uint32_t* __restrict__ rank, uint64_t cap) {
    const int64_t r = (int64_t)blockIdx.x * kRegTile + threadIdx.x;
    if (r >= V) return;
    double v[4];
    vox_load<true>(pts, vox_off[r], v);
    VoxPt p;
    vox_point(G, v, p);                                              // (a map row is a kept point: flag 0)
    const uint64_t mask = cap - 1;
    for (uint64_t h = vox_hash(p.key) & mask;; h = (h + 1) & mask) {
        if (atomicCAS(keys + h, kVoxEmpty, p.key) == kVoxEmpty) { rank[h] = (uint32_t)r; return; }   // keys are distinct
    }
}

__device__ __forceinline__ uint32_t map_lookup(const MapView& M, unsigned long long key) {
    const uint64_t mask = M.cap - 1;
    for (uint64_t h = vox_hash(key) & mask;; h = (h + 1) & mask) {
        const unsigned long long k = __ldg(M.keys + h);
        if (k == key) return __ldg(M.rank + h);
        if (k == kVoxEmpty) return kMapNoRank;
    }
}

// The nearest map row of w within the gate: its sorted row (-1: none), original index and d2; OR-s LMC_FLAG_NAN into fl
// for a non-finite query.  A query whose own cell is outside the key range has no match.
__device__ __forceinline__ int64_t map_nearest(const MapView& M, const double (&w)[3], int64_t& best_i, double& best_d2, uint32_t& fl) {
    best_i = -1;
    best_d2 = __longlong_as_double(0x7ff0000000000000ll);
    const double v[4] = {w[0], w[1], w[2], 0.0};
    VoxPt p;
    const uint32_t f = vox_point(M.G, v, p);
    if (f != 0) { fl |= f & LMC_FLAG_NAN; return -1; }
    int64_t best_row = -1;
    for (int dz = -1; dz <= 1; ++dz) {
        const long long kz = (long long)((p.key >> 42) & 0x1fffff) + dz;
        if (kz < 0 || kz > 0x1fffff) continue;
        for (int dy = -1; dy <= 1; ++dy) {
            const long long ky = (long long)((p.key >> 21) & 0x1fffff) + dy;
            if (ky < 0 || ky > 0x1fffff) continue;
            for (int dx = -1; dx <= 1; ++dx) {
                const long long kx = (long long)(p.key & 0x1fffff) + dx;
                if (kx < 0 || kx > 0x1fffff) continue;
                const uint32_t r = map_lookup(M, (unsigned long long)kx | ((unsigned long long)ky << 21) | ((unsigned long long)kz << 42));
                if (r == kMapNoRank) continue;
                const int64_t e = __ldg(M.vox_off + r + 1);
                for (int64_t j = __ldg(M.vox_off + r); j < e; ++j) {
                    double m0, m1, m2, m3;
                    ldg256(M.pts + 4 * j, m0, m1, m2, m3);
                    const double ex = __dsub_rn(w[0], m0), ey = __dsub_rn(w[1], m1), ez = __dsub_rn(w[2], m2);
                    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
                    if (d2 <= M.r2) {
                        const int64_t id = __ldg(M.idx + j);
                        if (d2 < best_d2 || (d2 == best_d2 && id < best_i)) { best_d2 = d2; best_i = id; best_row = j; }
                    }
                }
            }
        }
    }
    return best_row;
}

template <bool F64>
__global__ void __launch_bounds__(kRegTile) k_map_nearest(const void* __restrict__ pts, int64_t n, const MapView M,
                                                          int64_t* __restrict__ idx_out, double* __restrict__ d2_out,
                                                          uint32_t* __restrict__ status) {
    const int64_t i = (int64_t)blockIdx.x * kRegTile + threadIdx.x;
    uint32_t fl = 0;
    if (i < n) {
        double v[4];
        vox_load<F64>(pts, i, v);
        const double w[3] = {v[0], v[1], v[2]};
        int64_t bi;
        double bd;
        map_nearest(M, w, bi, bd, fl);
        idx_out[i] = bi;
        d2_out[i] = bd;
    }
    fl = __reduce_or_sync(0xffffffffu, fl);
    if (fl != 0 && (threadIdx.x & 31) == 0) atomicOr(status, fl);
}

// ---- registration ------------------------------------------------------------------------------------------------
struct RegWs {
    int64_t* coff;                  // [F + 1] chunk offsets by frame
    int32_t* chunk_frame;           // [C] frame of each chunk, -1 past the last one
    double* part;                   // [C][sums] partial sums by chunk (kRegSums, or kRegPlaneSums point-to-plane)
    int64_t chunks;                 // C: an upper bound of the chunk count, min(F, N) + ceil(N / 256)
};
static int64_t reg_chunks(int64_t n, int64_t F) { return (n < F ? n : F) + (n + kRegTile - 1) / kRegTile; }
static RegWs reg_layout(void* ws, int64_t n, int64_t F, size_t& total, int sums = kRegSums) {
    RegWs W;
    W.chunks = reg_chunks(n, F);
    uint8_t* b = static_cast<uint8_t*>(ws);
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t* p = b ? b + off : nullptr; off += reg_align(bytes); return p; };
    W.coff = reinterpret_cast<int64_t*>(take(8 * (size_t)(F + 1)));
    W.chunk_frame = reinterpret_cast<int32_t*>(take(4 * (size_t)W.chunks));
    W.part = reinterpret_cast<double*>(take(8 * (size_t)sums * (size_t)W.chunks));
    total = off;
    return W;
}
size_t register_workspace_bytes(int64_t n, int64_t F) { size_t t; reg_layout(nullptr, n, F, t); return t; }
size_t register_plane_workspace_bytes(int64_t n, int64_t F) { size_t t; reg_layout(nullptr, n, F, t, kRegPlaneSums); return t; }
int64_t register_max_chunks(int64_t n, int64_t F) { return reg_chunks(n, F); }

__global__ void __launch_bounds__(kRegTile) k_reg_count(const int64_t* __restrict__ frame_off, int64_t F, int64_t* __restrict__ coff) {
    const int64_t f = (int64_t)blockIdx.x * kRegTile + threadIdx.x;
    if (f < F) coff[f + 1] = (frame_off[f + 1] - frame_off[f] + kRegTile - 1) / kRegTile;
}

__global__ void __launch_bounds__(kRegTile) k_reg_chunks(const int64_t* __restrict__ coff, int64_t F, int64_t chunks,
                                                         int32_t* __restrict__ chunk_frame) {
    const int64_t c = (int64_t)blockIdx.x * kRegTile + threadIdx.x;
    if (c >= chunks) return;
    int64_t lo = 0, hi = F;                                          // the last frame f with coff[f] <= c
    while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if (coff[mid] <= c) lo = mid; else hi = mid; }
    chunk_frame[c] = c < coff[F] ? (int32_t)lo : -1;
}

template <bool F64>
__global__ void __launch_bounds__(kRegTile) k_reg_accum(const void* __restrict__ pts, const int64_t* __restrict__ frame_off,
                                                        const RegWs W, const double* __restrict__ pose,
                                                        const int32_t* __restrict__ flags, const MapView M,
                                                        uint32_t* __restrict__ status) {
    __shared__ double s_warp[kRegTile / 32][kRegSums];
    const int64_t c = blockIdx.x;
    const int32_t f = W.chunk_frame[c];
    if (f < 0 || flags[f] != 0) return;                              // past the last chunk, or the frame is done
    const int64_t i = frame_off[f] + (c - W.coff[f]) * kRegTile + threadIdx.x;
    uint32_t fl = 0;
    int64_t j = -1;
    double a[3] = {0.0, 0.0, 0.0}, w[3] = {0.0, 0.0, 0.0};
    if (i < frame_off[f + 1]) {
        double v[4];
        vox_load<F64>(pts, i, v);
        const double* P = pose + 12 * (int64_t)f;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            a[r] = __dadd_rn(__dadd_rn(__dmul_rn(P[3 * r], v[0]), __dmul_rn(P[3 * r + 1], v[1])), __dmul_rn(P[3 * r + 2], v[2]));
            w[r] = __dadd_rn(a[r], P[9 + r]);
        }
        int64_t bi;
        double bd;
        j = map_nearest(M, w, bi, bd, fl);
    }
    double s[kRegSums];
#pragma unroll
    for (int k = 0; k < kRegSums; ++k) s[k] = 0.0;
    if (j >= 0) {
        const double r0 = __dsub_rn(w[0], M.pts[4 * j]), r1 = __dsub_rn(w[1], M.pts[4 * j + 1]), r2 = __dsub_rn(w[2], M.pts[4 * j + 2]);
        s[0] = 1.0;
        s[1] = a[0]; s[2] = a[1]; s[3] = a[2];
        s[4] = a[0] * a[0]; s[5] = a[0] * a[1]; s[6] = a[0] * a[2]; s[7] = a[1] * a[1]; s[8] = a[1] * a[2]; s[9] = a[2] * a[2];
        s[10] = r0; s[11] = r1; s[12] = r2;
        s[13] = a[1] * r2 - a[2] * r1; s[14] = a[2] * r0 - a[0] * r2; s[15] = a[0] * r1 - a[1] * r0;
        s[16] = r0 * r0 + r1 * r1 + r2 * r2;
    }
    fl = __reduce_or_sync(0xffffffffu, fl);
    if (fl != 0 && (threadIdx.x & 31) == 0) atomicOr(status, fl);
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < kRegSums; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_down_sync(0xffffffffu, s[k], o);
        if (lane == 0) s_warp[wp][k] = s[k];
    }
    __syncthreads();
    if (threadIdx.x < kRegSums) {
        double t = s_warp[0][threadIdx.x];
#pragma unroll
        for (int k = 1; k < kRegTile / 32; ++k) t += s_warp[k][threadIdx.x];
        W.part[kRegSums * c + threadIdx.x] = t;
    }
}

// The Gauss-Newton step shared by both metrics: Cholesky of H (a pivot <= 1e-12 trace(H) is degenerate and keeps the
// pose), [tau; phi] = -H^-1 g, t <- t + tau, R <- Exp(phi) R, and the convergence test.
__device__ __forceinline__ void reg_step(const double (&H)[6][6], const double (&g)[6], double* P, int32_t* flag, double tol_t,
                                         double tol_r) {
    double Hd = 0.0;
    for (int k = 0; k < 6; ++k) Hd += H[k][k];
    double L[6][6] = {};
    for (int j = 0; j < 6; ++j) {
        double d = H[j][j];
        for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
        if (!(d > 1e-12 * Hd)) { *flag = kRegDegenerate; return; }
        L[j][j] = sqrt(d);
        for (int i = j + 1; i < 6; ++i) {
            double e = H[i][j];
            for (int k = 0; k < j; ++k) e -= L[i][k] * L[j][k];
            L[i][j] = e / L[j][j];
        }
    }
    double y[6], x[6];
    for (int i = 0; i < 6; ++i) { double e = -g[i]; for (int k = 0; k < i; ++k) e -= L[i][k] * y[k]; y[i] = e / L[i][i]; }
    for (int i = 5; i >= 0; --i) { double e = y[i]; for (int k = i + 1; k < 6; ++k) e -= L[k][i] * x[k]; x[i] = e / L[i][i]; }
    const double th2 = x[3] * x[3] + x[4] * x[4] + x[5] * x[5], th = sqrt(th2);
    const double sA = th < 1e-8 ? 1.0 - th2 / 6.0 : sin(th) / th;
    const double sB = th < 1e-8 ? 0.5 - th2 / 24.0 : (1.0 - cos(th)) / th2;
    const double K[3][3] = {{0.0, -x[5], x[4]}, {x[5], 0.0, -x[3]}, {-x[4], x[3], 0.0}};
    double E[3][3], Rn[3][3];
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) {
            double k2 = 0.0;
            for (int k = 0; k < 3; ++k) k2 += K[r][k] * K[k][q];
            E[r][q] = (r == q ? 1.0 : 0.0) + sA * K[r][q] + sB * k2;
        }
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) Rn[r][q] = E[r][0] * P[q] + E[r][1] * P[3 + q] + E[r][2] * P[6 + q];
    for (int r = 0; r < 3; ++r) {
        for (int q = 0; q < 3; ++q) P[3 * r + q] = Rn[r][q];
        P[9 + r] += x[r];
    }
    if (sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]) <= tol_t && th <= tol_r) *flag = kRegConverged;
}

// One warp per frame: lane k < 17 sums partial k over the frame's chunks in chunk order; lane 0 solves and updates.
__global__ void __launch_bounds__(kRegTile) k_reg_solve(int64_t F, const RegWs W, double* __restrict__ pose, int32_t* __restrict__ flags,
                                                        int32_t* __restrict__ inliers, double* __restrict__ rms,
                                                        int32_t* __restrict__ iterations, double tol_t, double tol_r) {
    const int64_t f = ((int64_t)blockIdx.x * kRegTile + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (f >= F || flags[f] != 0) return;                             // (warp-uniform)
    double t = 0.0;
    if (lane < kRegSums)
        for (int64_t c = W.coff[f]; c < W.coff[f + 1]; ++c) t += W.part[kRegSums * c + lane];
    double s[kRegSums];
#pragma unroll
    for (int k = 0; k < kRegSums; ++k) s[k] = __shfl_sync(0xffffffffu, t, k);
    if (lane != 0) return;
    const double n = s[0];
    iterations[f] += 1;
    inliers[f] = (int32_t)n;
    rms[f] = n > 0.0 ? sqrt(s[16] / n) : __longlong_as_double(0x7ff8000000000000ll);
    if (n < 6.0) { flags[f] = kRegDegenerate; return; }
    const double sa[3] = {s[1], s[2], s[3]};
    const double A[3][3] = {{s[4], s[5], s[6]}, {s[5], s[7], s[8]}, {s[6], s[8], s[9]}};
    const double tr = s[4] + s[7] + s[9];
    double H[6][6] = {};
    const double X[3][3] = {{0.0, -sa[2], sa[1]}, {sa[2], 0.0, -sa[0]}, {-sa[1], sa[0], 0.0}};     // [Sa]x
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) {
            H[r][q] = r == q ? n : 0.0;
            H[r][3 + q] = -X[r][q];
            H[3 + r][q] = X[r][q];
            H[3 + r][3 + q] = (r == q ? tr : 0.0) - A[r][q];
        }
    const double g[6] = {s[10], s[11], s[12], s[13], s[14], s[15]};
    reg_step(H, g, pose + 12 * f, flags + f, tol_t, tol_r);
}

// ---- normals ------------------------------------------------------------------------------------------------------
// One thread per map row p (sorted order): every map row m with d2 <= r2 (the row itself included), visited in
// map_nearest's cell order then sorted-row order; d = m - p, sequential sums S d and S dd^T, mu = S d / n,
// C = S dd^T / n - mu mu^T, a cyclic Jacobi eigen-decomposition of C, and (normal of lambda_min, planarity).  Every
// operation is an IEEE-rounded + - x / sqrt, so NumPy computes the same bits (oracle/lmc_oracle_plane.py).  (A walk of its own: sharing
// map_nearest's would change k_map_nearest's code.)
constexpr int kJacobiSweeps = 32;                    // a sweep cap; a 3x3 reaches exact zeros in about 10

// Rotate the pair (p, q) of the symmetric 3x3 A (a[r][c]) and accumulate the rotation into the columns of V.
__device__ __forceinline__ void jacobi_rotate(double (&a)[3][3], double (&V)[3][3], int p, int q) {
    const double apq = a[p][q];
    if (apq == 0.0) return;
    const int r = 3 - p - q;
    const double th = __ddiv_rn(__dsub_rn(a[q][q], a[p][p]), __dmul_rn(2.0, apq));
    double t = __ddiv_rn(1.0, __dadd_rn(fabs(th), __dsqrt_rn(__dadd_rn(__dmul_rn(th, th), 1.0))));
    if (th < 0.0) t = -t;
    const double c = __ddiv_rn(1.0, __dsqrt_rn(__dadd_rn(__dmul_rn(t, t), 1.0))), s = __dmul_rn(t, c);
    a[p][p] = __dsub_rn(a[p][p], __dmul_rn(t, apq));
    a[q][q] = __dadd_rn(a[q][q], __dmul_rn(t, apq));
    a[p][q] = a[q][p] = 0.0;
    const double arp = a[r][p], arq = a[r][q];
    a[r][p] = a[p][r] = __dsub_rn(__dmul_rn(c, arp), __dmul_rn(s, arq));
    a[r][q] = a[q][r] = __dadd_rn(__dmul_rn(s, arp), __dmul_rn(c, arq));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double vp = V[k][p], vq = V[k][q];
        V[k][p] = __dsub_rn(__dmul_rn(c, vp), __dmul_rn(s, vq));
        V[k][q] = __dadd_rn(__dmul_rn(s, vp), __dmul_rn(c, vq));
    }
}

__global__ void __launch_bounds__(kRegTile) k_map_normals(int64_t M_rows, const MapView M, int32_t min_nb, double* __restrict__ out,
                                                          int32_t* __restrict__ nb_out) {
    const int64_t i = (int64_t)blockIdx.x * kRegTile + threadIdx.x;
    if (i >= M_rows) return;
    double p[4];
    ldg256(M.pts + 4 * i, p[0], p[1], p[2], p[3]);
    const double v[4] = {p[0], p[1], p[2], 0.0};
    VoxPt vp;
    vox_point(M.G, v, vp);                                           // (a map row has a key in range)
    int32_t n = 0;
    double sd[3] = {0.0, 0.0, 0.0}, sdd[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};    // xx xy xz yy yz zz
    for (int dz = -1; dz <= 1; ++dz) {
        const long long kz = (long long)((vp.key >> 42) & 0x1fffff) + dz;
        if (kz < 0 || kz > 0x1fffff) continue;
        for (int dy = -1; dy <= 1; ++dy) {
            const long long ky = (long long)((vp.key >> 21) & 0x1fffff) + dy;
            if (ky < 0 || ky > 0x1fffff) continue;
            for (int dx = -1; dx <= 1; ++dx) {
                const long long kx = (long long)(vp.key & 0x1fffff) + dx;
                if (kx < 0 || kx > 0x1fffff) continue;
                const uint32_t r = map_lookup(M, (unsigned long long)kx | ((unsigned long long)ky << 21) | ((unsigned long long)kz << 42));
                if (r == kMapNoRank) continue;
                const int64_t e = __ldg(M.vox_off + r + 1);
                for (int64_t j = __ldg(M.vox_off + r); j < e; ++j) {
                    double m0, m1, m2, m3;
                    ldg256(M.pts + 4 * j, m0, m1, m2, m3);
                    const double d[3] = {__dsub_rn(m0, p[0]), __dsub_rn(m1, p[1]), __dsub_rn(m2, p[2])};
                    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(d[0], d[0]), __dmul_rn(d[1], d[1])), __dmul_rn(d[2], d[2]));
                    if (d2 <= M.r2) {
                        ++n;
#pragma unroll
                        for (int c = 0; c < 3; ++c) sd[c] = __dadd_rn(sd[c], d[c]);
                        sdd[0] = __dadd_rn(sdd[0], __dmul_rn(d[0], d[0]));
                        sdd[1] = __dadd_rn(sdd[1], __dmul_rn(d[0], d[1]));
                        sdd[2] = __dadd_rn(sdd[2], __dmul_rn(d[0], d[2]));
                        sdd[3] = __dadd_rn(sdd[3], __dmul_rn(d[1], d[1]));
                        sdd[4] = __dadd_rn(sdd[4], __dmul_rn(d[1], d[2]));
                        sdd[5] = __dadd_rn(sdd[5], __dmul_rn(d[2], d[2]));
                    }
                }
            }
        }
    }
    if (nb_out) nb_out[i] = n;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    double* o = out + 4 * i;
    if (n < min_nb) { stg256(o, nan, nan, nan, 0.0); return; }
    const double dn = (double)n;
    const double mu[3] = {__ddiv_rn(sd[0], dn), __ddiv_rn(sd[1], dn), __ddiv_rn(sd[2], dn)};
    double a[3][3], V[3][3] = {{1.0, 0.0, 0.0}, {0.0, 1.0, 0.0}, {0.0, 0.0, 1.0}};
    a[0][0] = __dsub_rn(__ddiv_rn(sdd[0], dn), __dmul_rn(mu[0], mu[0]));
    a[0][1] = a[1][0] = __dsub_rn(__ddiv_rn(sdd[1], dn), __dmul_rn(mu[0], mu[1]));
    a[0][2] = a[2][0] = __dsub_rn(__ddiv_rn(sdd[2], dn), __dmul_rn(mu[0], mu[2]));
    a[1][1] = __dsub_rn(__ddiv_rn(sdd[3], dn), __dmul_rn(mu[1], mu[1]));
    a[1][2] = a[2][1] = __dsub_rn(__ddiv_rn(sdd[4], dn), __dmul_rn(mu[1], mu[2]));
    a[2][2] = __dsub_rn(__ddiv_rn(sdd[5], dn), __dmul_rn(mu[2], mu[2]));
    for (int sw = 0; sw < kJacobiSweeps && (a[0][1] != 0.0 || a[0][2] != 0.0 || a[1][2] != 0.0); ++sw) {
        jacobi_rotate(a, V, 0, 1);
        jacobi_rotate(a, V, 0, 2);
        jacobi_rotate(a, V, 1, 2);
    }
    double lam[3] = {a[0][0], a[1][1], a[2][2]};
    int ix[3] = {0, 1, 2};                                           // stable ascending: strict compares keep index order
    auto cswap = [&](int u, int w) { if (lam[ix[w]] < lam[ix[u]]) { const int t = ix[u]; ix[u] = ix[w]; ix[w] = t; } };
    cswap(0, 1); cswap(1, 2); cswap(0, 1);
    const double l0 = lam[ix[0]] > 0.0 ? lam[ix[0]] : 0.0, l1 = lam[ix[1]] > 0.0 ? lam[ix[1]] : 0.0, l2 = lam[ix[2]] > 0.0 ? lam[ix[2]] : 0.0;
    if (l2 == 0.0) { stg256(o, nan, nan, nan, 0.0); return; }
    double nv[3] = {V[0][ix[0]], V[1][ix[0]], V[2][ix[0]]};
    const double nr = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(nv[0], nv[0]), __dmul_rn(nv[1], nv[1])), __dmul_rn(nv[2], nv[2])));
    int big = 0;
#pragma unroll
    for (int c = 1; c < 3; ++c) if (fabs(nv[c]) > fabs(nv[big])) big = c;
    const double sg = nv[big] < 0.0 ? -1.0 : 1.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) nv[c] = sg * __ddiv_rn(nv[c], nr);
    stg256(o, nv[0], nv[1], nv[2], __ddiv_rn(__dsub_rn(l1, l0), l2));
}

// ---- point-to-plane registration ----------------------------------------------------------------------------------
// Per inlier (nearest map row q with planarity >= min_planarity): e = n . (w - q), J = [n; a x n]; the 29 sums are
// products x_u x_v of x = [J(6), e, 1]: n, H = S J J^T (upper triangle, row-major), g = S J e, S e^2.
__constant__ uint8_t c_plane_u[kRegPlaneSums] = {7, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 4, 4, 5, 0, 1, 2, 3, 4, 5, 6};
__constant__ uint8_t c_plane_v[kRegPlaneSums] = {7, 0, 1, 2, 3, 4, 5, 1, 2, 3, 4, 5, 2, 3, 4, 5, 3, 4, 5, 4, 5, 5, 6, 6, 6, 6, 6, 6, 6};

// The chunk's sums in a fixed order through shared memory (the 29 products never sit in registers at once): each of
// 8 segments (points g, g + 8, ..., g + 248) sums its products sequentially, then the 8 segment sums in order.
template <bool F64>
__global__ void __launch_bounds__(kRegTile) k_reg_accum_plane(const void* __restrict__ pts, const int64_t* __restrict__ frame_off,
                                                              const RegWs W, const double* __restrict__ pose,
                                                              const int32_t* __restrict__ flags, const MapView M,
                                                              const double* __restrict__ normals, double min_planarity,
                                                              uint32_t* __restrict__ status) {
    constexpr int kSeg = 8, kSegLen = kRegTile / kSeg;
    __shared__ double s_x[8][kRegTile];
    __shared__ double s_seg[kRegPlaneSums][kSeg];
    const int64_t c = blockIdx.x;
    const int32_t f = W.chunk_frame[c];
    if (f < 0 || flags[f] != 0) return;                              // past the last chunk, or the frame is done
    const int64_t i = frame_off[f] + (c - W.coff[f]) * kRegTile + threadIdx.x;
    uint32_t fl = 0;
    double x[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (i < frame_off[f + 1]) {
        double v[4], a[3], w[3];
        vox_load<F64>(pts, i, v);
        const double* P = pose + 12 * (int64_t)f;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            a[r] = __dadd_rn(__dadd_rn(__dmul_rn(P[3 * r], v[0]), __dmul_rn(P[3 * r + 1], v[1])), __dmul_rn(P[3 * r + 2], v[2]));
            w[r] = __dadd_rn(a[r], P[9 + r]);
        }
        int64_t bi;
        double bd;
        const int64_t j = map_nearest(M, w, bi, bd, fl);
        if (j >= 0) {
            double nx, ny, nz, pl;
            ldg256(normals + 4 * j, nx, ny, nz, pl);
            if (pl >= min_planarity) {
                const double rx = __dsub_rn(w[0], M.pts[4 * j]), ry = __dsub_rn(w[1], M.pts[4 * j + 1]), rz = __dsub_rn(w[2], M.pts[4 * j + 2]);
                x[0] = nx; x[1] = ny; x[2] = nz;
                x[3] = __dsub_rn(__dmul_rn(a[1], nz), __dmul_rn(a[2], ny));
                x[4] = __dsub_rn(__dmul_rn(a[2], nx), __dmul_rn(a[0], nz));
                x[5] = __dsub_rn(__dmul_rn(a[0], ny), __dmul_rn(a[1], nx));
                x[6] = __dadd_rn(__dadd_rn(__dmul_rn(nx, rx), __dmul_rn(ny, ry)), __dmul_rn(nz, rz));
                x[7] = 1.0;
            }
        }
    }
    fl = __reduce_or_sync(0xffffffffu, fl);
    if (fl != 0 && (threadIdx.x & 31) == 0) atomicOr(status, fl);
#pragma unroll
    for (int k = 0; k < 8; ++k) s_x[k][threadIdx.x] = x[k];
    __syncthreads();
    if (threadIdx.x < kRegPlaneSums * kSeg) {
        const int k = threadIdx.x / kSeg, g = threadIdx.x % kSeg;
        const double* xu = s_x[c_plane_u[k]] + g;
        const double* xv = s_x[c_plane_v[k]] + g;
        double t = 0.0;
        for (int m = 0; m < kSegLen; ++m) t = __dadd_rn(t, __dmul_rn(xu[kSeg * m], xv[kSeg * m]));
        s_seg[k][g] = t;
    }
    __syncthreads();
    if (threadIdx.x < kRegPlaneSums) {
        double t = s_seg[threadIdx.x][0];
#pragma unroll
        for (int g = 1; g < kSeg; ++g) t = __dadd_rn(t, s_seg[threadIdx.x][g]);
        W.part[kRegPlaneSums * c + threadIdx.x] = t;
    }
}

// One warp per frame: lane k < 29 sums partial k over the frame's chunks in chunk order; lane 0 solves and updates.
__global__ void __launch_bounds__(kRegTile) k_reg_solve_plane(int64_t F, const RegWs W, double* __restrict__ pose,
                                                              int32_t* __restrict__ flags, int32_t* __restrict__ inliers,
                                                              double* __restrict__ rms, int32_t* __restrict__ iterations,
                                                              double tol_t, double tol_r) {
    const int64_t f = ((int64_t)blockIdx.x * kRegTile + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (f >= F || flags[f] != 0) return;                             // (warp-uniform)
    double t = 0.0;
    if (lane < kRegPlaneSums)
        for (int64_t c = W.coff[f]; c < W.coff[f + 1]; ++c) t += W.part[kRegPlaneSums * c + lane];
    double s[kRegPlaneSums];
#pragma unroll
    for (int k = 0; k < kRegPlaneSums; ++k) s[k] = __shfl_sync(0xffffffffu, t, k);
    if (lane != 0) return;
    const double n = s[0];
    iterations[f] += 1;
    inliers[f] = (int32_t)n;
    rms[f] = n > 0.0 ? sqrt(s[28] / n) : __longlong_as_double(0x7ff8000000000000ll);
    if (n < 6.0) { flags[f] = kRegDegenerate; return; }
    double H[6][6];
    for (int r = 0, k = 1; r < 6; ++r)
        for (int q = r; q < 6; ++q, ++k) H[r][q] = H[q][r] = s[k];
    const double g[6] = {s[22], s[23], s[24], s[25], s[26], s[27]};
    reg_step(H, g, pose + 12 * f, flags + f, tol_t, tol_r);
}

cudaError_t launch_map_build(const double* pts, const int64_t* vox_off, int64_t V, const double* leaf, const double* origin,
                             void* table, cudaStream_t st) {
    const MapView M = map_view(pts, nullptr, vox_off, table, V, leaf, origin, 0.0);
    cudaError_t e;
    if ((e = cudaMemsetAsync(table, 0xff, map_table_bytes(V), st)) != cudaSuccess) return e;
    if (V > 0)
        k_map_insert<<<(unsigned)((V + kRegTile - 1) / kRegTile), kRegTile, 0, st>>>(pts, vox_off, V, M.G,
                                                                                      const_cast<unsigned long long*>(M.keys),
                                                                                      const_cast<uint32_t*>(M.rank), M.cap);
    return cudaGetLastError();
}

cudaError_t launch_map_nearest(bool f64, const void* q, int64_t n, const double* pts, const int64_t* idx, const int64_t* vox_off,
                               const void* table, int64_t V, const double* leaf, const double* origin, double r2,
                               int64_t* idx_out, double* d2_out, uint32_t* status, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const MapView M = map_view(pts, idx, vox_off, table, V, leaf, origin, r2);
    const unsigned blocks = (unsigned)((n + kRegTile - 1) / kRegTile);
    if (f64) k_map_nearest<true><<<blocks, kRegTile, 0, st>>>(q, n, M, idx_out, d2_out, status);
    else     k_map_nearest<false><<<blocks, kRegTile, 0, st>>>(q, n, M, idx_out, d2_out, status);
    return cudaGetLastError();
}

// Outputs initialised, chunk table built: the set-up both metrics share.
static cudaError_t reg_setup(const int64_t* frame_off, int64_t F, const RegWs& W, const double* pose_in, double* pose_out, int32_t* inliers,
                             double* rms, int32_t* iterations, int32_t* flags, cudaStream_t st) {
    cudaError_t e;
    if ((e = cudaMemcpyAsync(pose_out, pose_in, 12 * sizeof(double) * (size_t)F, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(flags, 0, 4 * (size_t)F, st)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(iterations, 0, 4 * (size_t)F, st)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(inliers, 0, 4 * (size_t)F, st)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(rms, 0xff, 8 * (size_t)F, st)) != cudaSuccess) return e;      // (NaN until a frame's first pass)
    const unsigned fb = (unsigned)((F + kRegTile - 1) / kRegTile);
    k_reg_count<<<fb, kRegTile, 0, st>>>(frame_off, F, W.coff);
    if ((e = launch_tile_scan(W.coff, F, st)) != cudaSuccess) return e;
    if (W.chunks > 0) k_reg_chunks<<<(unsigned)((W.chunks + kRegTile - 1) / kRegTile), kRegTile, 0, st>>>(W.coff, F, W.chunks, W.chunk_frame);
    return cudaSuccess;
}

cudaError_t launch_register_frames(bool f64, const void* q, int64_t n, const int64_t* frame_off, int64_t F, const double* pose_in,
                                   const double* pts, const int64_t* idx, const int64_t* vox_off, const void* table, int64_t V,
                                   const double* leaf, const double* origin, double r2, int32_t iters, double tol_t, double tol_r,
                                   void* ws, double* pose_out, int32_t* inliers, double* rms, int32_t* iterations, int32_t* flags,
                                   uint32_t* status, cudaStream_t st) {
    if (F == 0) return cudaSuccess;
    size_t total;
    const RegWs W = reg_layout(ws, n, F, total);
    const MapView M = map_view(pts, idx, vox_off, table, V, leaf, origin, r2);
    cudaError_t e;
    if ((e = reg_setup(frame_off, F, W, pose_in, pose_out, inliers, rms, iterations, flags, st)) != cudaSuccess) return e;
    const unsigned sb = (unsigned)((32 * F + kRegTile - 1) / kRegTile);
    for (int32_t it = 0; it < iters; ++it) {
        if (W.chunks > 0) {
            if (f64) k_reg_accum<true><<<(unsigned)W.chunks, kRegTile, 0, st>>>(q, frame_off, W, pose_out, flags, M, status);
            else     k_reg_accum<false><<<(unsigned)W.chunks, kRegTile, 0, st>>>(q, frame_off, W, pose_out, flags, M, status);
        }
        k_reg_solve<<<sb, kRegTile, 0, st>>>(F, W, pose_out, flags, inliers, rms, iterations, tol_t, tol_r);
    }
    return cudaGetLastError();
}

cudaError_t launch_map_normals(const double* pts, const int64_t* idx, const int64_t* vox_off, const void* table, int64_t M_rows,
                               int64_t V, const double* leaf, const double* origin, double r2, int32_t min_nb, double* normals,
                               int32_t* neighbours, cudaStream_t st) {
    if (M_rows == 0) return cudaSuccess;
    const MapView M = map_view(pts, idx, vox_off, table, V, leaf, origin, r2);
    k_map_normals<<<(unsigned)((M_rows + kRegTile - 1) / kRegTile), kRegTile, 0, st>>>(M_rows, M, min_nb, normals, neighbours);
    return cudaGetLastError();
}

cudaError_t launch_register_frames_plane(bool f64, const void* q, int64_t n, const int64_t* frame_off, int64_t F, const double* pose_in,
                                         const double* pts, const int64_t* idx, const int64_t* vox_off, const void* table, int64_t V,
                                         const double* leaf, const double* origin, double r2, const double* normals,
                                         double min_planarity, int32_t iters, double tol_t, double tol_r, void* ws, double* pose_out,
                                         int32_t* inliers, double* rms, int32_t* iterations, int32_t* flags, uint32_t* status,
                                         cudaStream_t st) {
    if (F == 0) return cudaSuccess;
    size_t total;
    const RegWs W = reg_layout(ws, n, F, total, kRegPlaneSums);
    const MapView M = map_view(pts, idx, vox_off, table, V, leaf, origin, r2);
    cudaError_t e;
    if ((e = reg_setup(frame_off, F, W, pose_in, pose_out, inliers, rms, iterations, flags, st)) != cudaSuccess) return e;
    const unsigned sb = (unsigned)((32 * F + kRegTile - 1) / kRegTile);
    for (int32_t it = 0; it < iters; ++it) {
        if (W.chunks > 0) {
            if (f64) k_reg_accum_plane<true><<<(unsigned)W.chunks, kRegTile, 0, st>>>(q, frame_off, W, pose_out, flags, M, normals,
                                                                                       min_planarity, status);
            else     k_reg_accum_plane<false><<<(unsigned)W.chunks, kRegTile, 0, st>>>(q, frame_off, W, pose_out, flags, M, normals,
                                                                                        min_planarity, status);
        }
        k_reg_solve_plane<<<sb, kRegTile, 0, st>>>(F, W, pose_out, flags, inliers, rms, iterations, tol_t, tol_r);
    }
    return cudaGetLastError();
}

}  // namespace lmc
