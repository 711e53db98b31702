// lmc_voxel.cuh -- the voxel key of a point, shared by the voxel-grid map (lmc_voxel.cu) and the point map's
// nearest-neighbour queries (lmc_register.cu), so both derive a cell from exactly the same f64 expressions.
#pragma once
#include "lmc_device.cuh"

namespace lmc {

constexpr uint64_t kVoxEmpty = ~0ull;                // a packed key has 63 bits: all-ones marks an empty slot
constexpr double kVoxKeyLim = 1048576.0;             // |k_c| range: [-2^20, 2^20), 21 bits per axis

struct VoxGrid { double o[3], L[3]; };

static inline uint64_t vox_cap(int64_t n) { uint64_t c = 64; while (c < 2 * (uint64_t)n) c <<= 1; return c; }

template <bool F64>
__device__ __forceinline__ void vox_load(const void* __restrict__ pts, int64_t i, double (&v)[4]) {
    if constexpr (F64) ldg256(reinterpret_cast<const double*>(pts) + 4 * i, v[0], v[1], v[2], v[3]);
    else { const float4 f = __ldg(reinterpret_cast<const float4*>(pts) + i); v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w; }
}

struct VoxPt { unsigned long long key; unsigned long long q[3]; long long qi; };

// 0 for a kept point, else the flag that drops it (a non-finite value: NAN, before the range checks: OVERFLOW)
__device__ __forceinline__ uint32_t vox_point(const VoxGrid& G, const double (&v)[4], VoxPt& p) {
    if (!(isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2]) && isfinite(v[3]))) return LMC_FLAG_NAN;
    double u[3], k[3];
    bool ok = fabs(v[3]) < 256.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        u[c] = __ddiv_rn(__dsub_rn(v[c], G.o[c]), G.L[c]);
        k[c] = floor(u[c]);
        ok &= k[c] >= -kVoxKeyLim && k[c] < kVoxKeyLim;          // (an infinite u fails here)
    }
    if (!ok) return LMC_FLAG_OVERFLOW;
    p.key = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        p.key |= (unsigned long long)((long long)k[c] + (1 << 20)) << (21 * c);
        // u - k rounds up to 1.0 for a tiny negative u: the clamp keeps q inside the voxel
        const unsigned long long q = (unsigned long long)__dmul_rn(__dsub_rn(u[c], k[c]), 4294967296.0);
        p.q[c] = q < 0xffffffffull ? q : 0xffffffffull;
    }
    p.qi = __double2ll_rn(__dmul_rn(v[3], 16777216.0));
    return 0;
}

__device__ __forceinline__ uint64_t vox_hash(uint64_t k) {         // murmur3 / splitmix finaliser: neighbouring voxels scatter
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}

}  // namespace lmc
