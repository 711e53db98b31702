// lmc_voxel.cu -- voxel-grid map of an (N,4) cloud [x y z intensity] on the device: one centroid, one point count per
// occupied voxel, voxels ranked by their first point (definition: oracle/lmc_oracle_voxel.py).
//
// Per point, in IEEE f64 with explicit rounding: u_c = (p_c - o_c) / L_c, k_c = floor(u_c) in [-2^20, 2^20), the
// fixed-point offset q_c = min(trunc((u_c - k_c) 2^32), 2^32 - 1) and q_I = rint(I 2^24) for |I| < 256.  The voxel's
// sums of q are 64-bit integers, so the order in which the atomics land changes nothing: the map is bit-identical from
// run to run and under any permutation of the input.  Two calls (the caller sizes the outputs from V in between):
//   index   k_voxel_insert  keys -> open-addressing table (64-bit CAS, linear probing, capacity pow2 >= 2N, so it never
//                           fills), atomicMin of the first point index per slot, the point's slot
//           k_voxel_count   first points per tile of 256  (a point is first when its slot's first index is its own)
//           launch_tile_scan (lmc_pcd.cu) -> the rank of every tile's first first-point; tile_off[tiles] = V
//           k_voxel_rank    the rank of every first point into its slot, and the voxel's key by rank
//   reduce  k_voxel_accum   q_x q_y q_z q_I 1 of every point into its voxel's u64 sums (red.global.add.u64), point_voxel
//           k_voxel_finalize centroid o_c + (k_c + (S_c / n) 2^-32) L_c and mean intensity (S_I / n) 2^-24, count
#include "lmc_voxel.cuh"

namespace lmc {
cudaError_t launch_tile_scan(int64_t* tile_off, int64_t tiles, cudaStream_t st);    // lmc_pcd.cu

constexpr int kVoxTile = 256;                        // points (= threads) per tile of every pass
constexpr uint32_t kVoxNoSlot = ~0u;                 // slot of a dropped point
constexpr int kVoxAcc = 5;                           // u64 sums per voxel: q_x q_y q_z q_I n

struct VoxWs {
    unsigned long long* keys;       // [cap] packed key of the slot, kVoxEmpty
    uint32_t* first;                // [cap] smallest point index in the slot
    uint32_t* rank;                 // [cap] the slot's voxel rank
    uint32_t* slot;                 // [n]   the point's slot, kVoxNoSlot for a dropped point
    int64_t* tile_off;              // [tiles + 1] first points per tile -> rank offsets (tile_off[tiles] = V)
    unsigned long long* vkey;       // [n]   packed key by rank
    unsigned long long* acc;        // [n][kVoxAcc] sums by rank
    uint64_t cap;
};

static inline size_t vox_align(size_t b) { return (b + 255) & ~size_t(255); }
static VoxWs vox_layout(void* ws, int64_t n, size_t& total) {
    const uint64_t cap = vox_cap(n), tiles = ((uint64_t)n + kVoxTile - 1) / kVoxTile;
    uint8_t* b = static_cast<uint8_t*>(ws);
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t* p = b ? b + off : nullptr; off += vox_align(bytes); return p; };
    VoxWs W;
    W.cap = cap;
    W.keys = reinterpret_cast<unsigned long long*>(take(8 * cap));
    W.first = reinterpret_cast<uint32_t*>(take(4 * cap));
    W.rank = reinterpret_cast<uint32_t*>(take(4 * cap));
    W.slot = reinterpret_cast<uint32_t*>(take(4 * (size_t)n));
    W.tile_off = reinterpret_cast<int64_t*>(take(8 * (tiles + 1)));
    W.vkey = reinterpret_cast<unsigned long long*>(take(8 * (size_t)n));
    W.acc = reinterpret_cast<unsigned long long*>(take(8 * kVoxAcc * (size_t)n));
    total = off;
    return W;
}
size_t voxel_workspace_bytes(int64_t n) { size_t t; vox_layout(nullptr, n, t); return t; }

template <bool F64>
__global__ void __launch_bounds__(kVoxTile) k_voxel_insert(const void* __restrict__ pts, int64_t n, const VoxGrid G, const VoxWs W,
                                                           uint32_t* __restrict__ status) {
    const int64_t i = (int64_t)blockIdx.x * kVoxTile + threadIdx.x;
    uint32_t fl = 0;
    if (i < n) {
        double v[4];
        vox_load<F64>(pts, i, v);
        VoxPt p;
        fl = vox_point(G, v, p);
        uint32_t s = kVoxNoSlot;
        if (fl == 0) {
            const uint64_t mask = W.cap - 1;
            uint64_t h = vox_hash(p.key) & mask;
            for (;; h = (h + 1) & mask) {
                if (h == kVoxNoSlot) continue;                         // (a 2^32-slot table leaves its last slot unused)
                unsigned long long cur = __ldcg(W.keys + h);          // a set key never changes; a stale empty goes to the CAS
                if (cur == kVoxEmpty) cur = atomicCAS(W.keys + h, kVoxEmpty, p.key);
                if (cur == kVoxEmpty || cur == p.key) break;
            }
            s = (uint32_t)h;
            atomicMin(W.first + s, (uint32_t)i);
        }
        W.slot[i] = s;
    }
    fl = __reduce_or_sync(0xffffffffu, fl);
    if (fl != 0 && (threadIdx.x & 31) == 0) atomicOr(status, fl);
}

__device__ __forceinline__ bool vox_is_first(const VoxWs& W, int64_t i, int64_t n, uint32_t& s) {
    if (i >= n) return false;
    s = W.slot[i];
    return s != kVoxNoSlot && __ldg(W.first + s) == (uint32_t)i;
}

__global__ void __launch_bounds__(kVoxTile) k_voxel_count(int64_t n, const VoxWs W) {
    const int64_t i = (int64_t)blockIdx.x * kVoxTile + threadIdx.x;
    uint32_t s;
    const int c = __syncthreads_count(vox_is_first(W, i, n, s));
    if (threadIdx.x == 0) W.tile_off[blockIdx.x + 1] = c;
}

__global__ void __launch_bounds__(kVoxTile) k_voxel_rank(int64_t n, const VoxWs W) {
    __shared__ uint32_t s_warp[kVoxTile / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * kVoxTile + threadIdx.x;
    uint32_t s = 0;
    const bool first = vox_is_first(W, i, n, s);
    const uint32_t b = __ballot_sync(0xffffffffu, first);
    if (lane == 0) s_warp[w] = __popc(b);
    __syncthreads();
    if (!first) return;
    uint32_t before = __popc(b & ((1u << lane) - 1u));
    for (int k = 0; k < w; ++k) before += s_warp[k];
    const int64_t r = W.tile_off[blockIdx.x] + before;
    W.rank[s] = (uint32_t)r;
    W.vkey[r] = W.keys[s];
}

template <bool F64>
__global__ void __launch_bounds__(kVoxTile) k_voxel_accum(const void* __restrict__ pts, int64_t n, const VoxGrid G, const VoxWs W,
                                                          int32_t* __restrict__ point_voxel) {
    const int64_t i = (int64_t)blockIdx.x * kVoxTile + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = W.slot[i];
    int32_t r = -1;
    if (s != kVoxNoSlot) {
        r = (int32_t)__ldg(W.rank + s);
        double v[4];
        vox_load<F64>(pts, i, v);
        VoxPt p;
        vox_point(G, v, p);
        unsigned long long* a = W.acc + (uint64_t)kVoxAcc * (uint32_t)r;
        atomicAdd(a + 0, p.q[0]);                                    // (result unused: red.global.add.u64)
        atomicAdd(a + 1, p.q[1]);
        atomicAdd(a + 2, p.q[2]);
        atomicAdd(a + 3, (unsigned long long)p.qi);                  // two's complement: the u64 sum is the int64 sum
        atomicAdd(a + 4, 1ull);
    }
    if (point_voxel != nullptr) point_voxel[i] = r;
}

template <bool F64>
__global__ void __launch_bounds__(kVoxTile) k_voxel_finalize(int64_t V, const VoxGrid G, const VoxWs W, void* __restrict__ out,
                                                             int32_t* __restrict__ counts) {
    const int64_t r = (int64_t)blockIdx.x * kVoxTile + threadIdx.x;
    if (r >= V) return;
    const unsigned long long* a = W.acc + (uint64_t)kVoxAcc * r;
    const unsigned long long cnt = a[4], key = W.vkey[r];
    const double dn = (double)cnt;                                   // exact: n < 2^31
    double c[4];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        const double k = (double)((long long)((key >> (21 * ax)) & 0x1fffffull) - (1 << 20));
        const double m = __dmul_rn(__ddiv_rn(__ull2double_rn(a[ax]), dn), 0x1p-32);
        c[ax] = __dadd_rn(G.o[ax], __dmul_rn(__dadd_rn(k, m), G.L[ax]));
    }
    c[3] = __dmul_rn(__ddiv_rn(__ll2double_rn((long long)a[3]), dn), 0x1p-24);
    if constexpr (F64) stg256(reinterpret_cast<double*>(out) + 4 * r, c[0], c[1], c[2], c[3]);
    else reinterpret_cast<float4*>(out)[r] = make_float4(__double2float_rn(c[0]), __double2float_rn(c[1]), __double2float_rn(c[2]),
                                                         __double2float_rn(c[3]));
    counts[r] = (int32_t)cnt;
}

static VoxGrid vox_grid(const double* leaf, const double* origin) {
    VoxGrid G;
    for (int c = 0; c < 3; ++c) { G.o[c] = origin[c]; G.L[c] = leaf[c]; }
    return G;
}

cudaError_t launch_voxel_index(bool f64, const void* pts, int64_t n, const double* leaf, const double* origin, void* ws,
                               int64_t* n_voxels, uint32_t* status, cudaStream_t st) {
    size_t total;
    const VoxWs W = vox_layout(ws, n, total);
    const VoxGrid G = vox_grid(leaf, origin);
    const int64_t tiles = (n + kVoxTile - 1) / kVoxTile;
    cudaError_t e;
    if (n > 0) {
        if ((e = cudaMemsetAsync(W.keys, 0xff, 8 * W.cap, st)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(W.first, 0xff, 4 * W.cap, st)) != cudaSuccess) return e;
        if (f64) k_voxel_insert<true><<<(unsigned)tiles, kVoxTile, 0, st>>>(pts, n, G, W, status);
        else     k_voxel_insert<false><<<(unsigned)tiles, kVoxTile, 0, st>>>(pts, n, G, W, status);
        k_voxel_count<<<(unsigned)tiles, kVoxTile, 0, st>>>(n, W);
    }
    if ((e = launch_tile_scan(W.tile_off, tiles, st)) != cudaSuccess) return e;
    if (n > 0) k_voxel_rank<<<(unsigned)tiles, kVoxTile, 0, st>>>(n, W);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cudaMemcpyAsync(n_voxels, W.tile_off + tiles, sizeof(int64_t), cudaMemcpyDeviceToDevice, st);
}

cudaError_t launch_voxel_reduce(bool f64, const void* pts, int64_t n, const double* leaf, const double* origin, void* ws,
                                int64_t V, void* out, int32_t* counts, int32_t* point_voxel, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    size_t total;
    const VoxWs W = vox_layout(ws, n, total);
    const VoxGrid G = vox_grid(leaf, origin);
    cudaError_t e;
    if (V > 0 && (e = cudaMemsetAsync(W.acc, 0, 8 * kVoxAcc * (size_t)V, st)) != cudaSuccess) return e;
    const unsigned tiles = (unsigned)((n + kVoxTile - 1) / kVoxTile);
    if (f64) k_voxel_accum<true><<<tiles, kVoxTile, 0, st>>>(pts, n, G, W, point_voxel);
    else     k_voxel_accum<false><<<tiles, kVoxTile, 0, st>>>(pts, n, G, W, point_voxel);
    if (V > 0) {
        const unsigned vt = (unsigned)((V + kVoxTile - 1) / kVoxTile);
        if (f64) k_voxel_finalize<true><<<vt, kVoxTile, 0, st>>>(V, G, W, out, counts);
        else     k_voxel_finalize<false><<<vt, kVoxTile, 0, st>>>(V, G, W, out, counts);
    }
    return cudaGetLastError();
}

}  // namespace lmc
