// lmc_las.cu -- (SURVEY 8f N2) a complete LAS 1.2 / point-format-3 file image built on the device:
// what `save_las` (LMC:950-963) / `_export_las` (CS:1671-1698) obtain from laspy.
//
// PARITY UNPINNED: laspy is neither vendored nor installed, so there are no reference bytes to
// compare with.  The file follows the public LAS 1.2 specification: 227-byte public header block,
// no VLRs, 34-byte PF3 records {X Y Z int32, intensity u16, return/flag byte, classification,
// scan angle, user data, point source id u16, gps_time f64, R G B u16}.  X/Y/Z are the same
// rint((v - offset) / scale) integers as the fused LAS epilogue (bit-exact against the restatement),
// intensity follows the two call sites (LMC:961 unit scale, CS:1686 raw), every field the reference
// never sets stays 0 (as laspy's zero-initialised record array would leave it), and the header's
// min / max are the scaled extremes X*scale + offset (what laspy's update_header computes), reduced on
// the GPU with integer atomics.
//
// Two launches: k_las_records (records + min/max reduction; the 227-byte data offset makes every
// record start at an odd address, so each CTA assembles its contiguous byte range in shared memory at
// the destination's 16-byte phase and hands the aligned body to the TMA engine as one bulk store), then k_las_header.
#include "lmc_device.cuh"

namespace lmc {

constexpr int kLasHeader  = 227;
constexpr int kLasRec     = 34;
constexpr int kLasTile    = 512;                    // points per CTA
constexpr int kLasThreads = 256;
constexpr int kLasImg     = ((kLasTile * kLasRec + 32 + 15) / 16) * 16;

__device__ __forceinline__ void put_le(uint8_t* p, uint64_t v, int nbytes) {
#pragma unroll
    for (int k = 0; k < 8; ++k) if (k < nbytes) p[k] = (uint8_t)(v >> (8 * k));
}

template <bool F64>
__global__ void __launch_bounds__(kLasThreads) k_las_records(const __grid_constant__ LasParams L) {
    __shared__ __align__(16) uint8_t s_img[kLasImg];
    __shared__ int32_t s_mm[6];
    const int tid = threadIdx.x;
    // points [p_begin, n) of the cloud; L.out is the (possibly virtual) address of file byte 0 (see lmc_las_pf3_records_*)
    const int64_t first = L.p_begin + (int64_t)blockIdx.x * kLasTile;
    const int cnt = (int)min((int64_t)kLasTile, L.n - first);
    const int64_t dst0 = kLasHeader + first * kLasRec;
    const int phase = (int)(reinterpret_cast<uintptr_t>(L.out + dst0) & 15);
    uint8_t* img = s_img + phase;
    if (tid < 6) s_mm[tid] = (tid & 1) ? INT32_MIN : INT32_MAX;
    __syncthreads();
    uint32_t fl = 0;
    int32_t mn[3] = { INT32_MAX, INT32_MAX, INT32_MAX }, mx[3] = { INT32_MIN, INT32_MIN, INT32_MIN };
    // (the always-exact quantiser route: this kernel is bound by its 34-byte records, not by FP64 -- the tie test of q_las costs it 2 %)
    auto quantise = [&](const Pt& p, uint32_t (&q)[4]) {
        const int2 qx = q_las_exact_body(p.x, L.scale[0], L.rcp[0], L.off[0]), qy = q_las_exact_body(p.y, L.scale[1], L.rcp[1], L.off[1]),
                   qz = q_las_exact_body(p.z, L.scale[2], L.rcp[2], L.off[2]);
        fl |= (uint32_t)(qx.y | qy.y | qz.y);
        mn[0] = min(mn[0], qx.x); mx[0] = max(mx[0], qx.x); mn[1] = min(mn[1], qy.x); mx[1] = max(mx[1], qy.x); mn[2] = min(mn[2], qz.x); mx[2] = max(mx[2], qz.x);
        q[0] = (uint32_t)qx.x; q[1] = (uint32_t)qy.x; q[2] = (uint32_t)qz.x; q[3] = q_las_intensity(p.w, L.intensity_mode, fl) & 0xffffu;
    };
    // record bytes: 0-11 X Y Z | 12-13 intensity | 14-19 return byte, classification, scan angle, user data, point source id = 0
    // | 20-27 gps_time | 28-33 R G B = 0
    if (cnt == kLasTile) {
        // Full tile: a thread owns two consecutive records = 68 bytes = 17 words w[], which start m = phase & 3 bytes into a
        // shared-memory word.  The words are shifted in registers (funnel shifts) and stored as 32-bit words at an odd word stride
        // (conflict-free); the word two neighbouring threads share is merged by a shuffle, the warp's two end words go byte-wise.
        const int64_t i = first + 2 * tid;
        Pt a, b;
        const bool al32 = ((reinterpret_cast<uintptr_t>(L.pts) + (F64 ? 32 : 16) * (uintptr_t)first) & 31) == 0;
        if (F64 || al32) load_pair<F64, true>(L.pts, i, true, true, a, b);
        else             load_pair<F64, false>(L.pts, i, true, false, a, b), load_pair<F64, false>(L.pts, i + 1, true, false, b, b);
        uint64_t g0 = 0, g1 = 0;
        if (L.gps_time) { g0 = (uint64_t)__double_as_longlong(__ldg(L.gps_time + i)); g1 = (uint64_t)__double_as_longlong(__ldg(L.gps_time + i + 1)); }
        uint32_t qa[4], qb[4];
        quantise(a, qa); quantise(b, qb);
        const uint32_t g0l = (uint32_t)g0, g0h = (uint32_t)(g0 >> 32), g1l = (uint32_t)g1, g1h = (uint32_t)(g1 >> 32);
        const uint32_t w[17] = { qa[0], qa[1], qa[2], qa[3], 0u, g0l, g0h, 0u,
                                 qb[0] << 16, (qb[0] >> 16) | (qb[1] << 16), (qb[1] >> 16) | (qb[2] << 16), (qb[2] >> 16) | (qb[3] << 16), 0u,
                                 g1l << 16, (g1l >> 16) | (g1h << 16), g1h >> 16, 0u };
        const int m = phase & 3;
        const uint32_t sh = 8u * (uint32_t)m;
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_img + (phase & ~3)) + 17 * tid;      // word holding the pair's first byte
        const uint32_t o0 = w[0] << sh;                                                    // bytes m..3 of word 0
        const uint32_t o17 = __funnelshift_l(w[16], 0u, sh);                               // bytes 0..m-1 of word 17 (0 when m == 0)
#pragma unroll
        for (int k = 1; k < 17; ++k) dst[k] = __funnelshift_l(w[k - 1], w[k], sh);
        const uint32_t nxt = __shfl_down_sync(0xffffffffu, o0, 1);
        const int lane = tid & 31;
        if (lane != 31) dst[17] = o17 | nxt;
        else {
            uint8_t* e = reinterpret_cast<uint8_t*>(dst + 17);
#pragma unroll
            for (int k = 0; k < 3; ++k) if (k < m) e[k] = (uint8_t)(o17 >> (8 * k));
        }
        if (lane == 0) {
            uint8_t* e = reinterpret_cast<uint8_t*>(dst);
#pragma unroll
            for (int k = 0; k < 4; ++k) if (k >= m) e[k] = (uint8_t)(o0 >> (8 * k));
        }
    } else {
        for (int j = tid; j < cnt; j += kLasThreads) {
            Pt p, unused;
            const int64_t i = first + j;
            load_pair<F64, false>(L.pts, i, true, false, p, unused);
            uint32_t q[4];
            quantise(p, q);
            // the record starts at an odd address (227 + 34 j): one byte, sixteen aligned halfwords, one byte
            uint8_t* r = img + j * kLasRec;
            const uint64_t gb = (uint64_t)__double_as_longlong(L.gps_time ? __ldg(L.gps_time + i) : 0.0);
            const uint32_t W[9] = { q[0], q[1], q[2], q[3], 0u, (uint32_t)gb, (uint32_t)(gb >> 32), 0u, 0u };
            if ((reinterpret_cast<uintptr_t>(r) & 1) != 0) {
                r[0] = (uint8_t)W[0];
                uint16_t* h = reinterpret_cast<uint16_t*>(r + 1);
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const int bb = 1 + 2 * k;                             // first byte of this halfword
                    h[k] = (bb & 3) == 1 ? (uint16_t)(W[bb >> 2] >> 8) : (uint16_t)((W[bb >> 2] >> 24) | (W[(bb >> 2) + 1] << 8));
                }
                r[33] = 0;
            } else {
                uint16_t* h = reinterpret_cast<uint16_t*>(r);
#pragma unroll
                for (int k = 0; k < 17; ++k) h[k] = (uint16_t)(W[k >> 1] >> (16 * (k & 1)));
            }
        }
    }
    // block min / max -> one atomic per value per CTA
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { mn[c] = min(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o)); mx[c] = max(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o)); }
        if ((tid & 31) == 0) { atomicMin(&s_mm[2 * c], mn[c]); atomicMax(&s_mm[2 * c + 1], mx[c]); }
    }
    __syncthreads();
    if (tid < 6 && cnt > 0) {
        // same-address atomics serialise in L2: peek first, only CTAs that actually move an extreme issue one
        const int32_t cur = *reinterpret_cast<volatile int32_t*>(L.minmax + tid), mine = s_mm[tid];
        if (tid & 1) { if (mine > cur) atomicMax(L.minmax + tid, mine); } else { if (mine < cur) atomicMin(L.minmax + tid, mine); }
    }
    cta_image_out(L.out + (dst0 - phase), s_img, phase, phase + cnt * kLasRec, tid, kLasThreads);   // TMA bulk store of the aligned body
    if (fl != 0 && L.status != nullptr) atomicOr(L.status, fl);
}

// LAS 1.2 public header block (227 bytes), written after the records so the extremes are final
__global__ void k_las_header(const __grid_constant__ LasParams L) {
    __shared__ uint8_t h[kLasHeader];
    const int tid = threadIdx.x;
    for (int i = tid; i < kLasHeader; i += blockDim.x) h[i] = 0;
    __syncthreads();
    if (tid == 0) {
        h[0] = 'L'; h[1] = 'A'; h[2] = 'S'; h[3] = 'F';
        h[24] = 1; h[25] = 2;                                                       // version 1.2
        const char sys[] = "OTHER"; for (int i = 0; i < 5; ++i) h[26 + i] = (uint8_t)sys[i];
        const char gen[] = "livox_mc_b200"; for (int i = 0; i < 13; ++i) h[58 + i] = (uint8_t)gen[i];
        put_le(h + 90, L.day, 2); put_le(h + 92, L.year, 2);
        put_le(h + 94, kLasHeader, 2);                                              // header size
        put_le(h + 96, kLasHeader, 4);                                              // offset to point data
        h[104] = 3;                                                                 // point data format
        put_le(h + 105, kLasRec, 2);
        put_le(h + 107, (uint64_t)L.n, 4);                                          // number of point records
        // number of points by return (5 x u32) stays 0: the reference never sets return numbers
        for (int c = 0; c < 3; ++c) {
            put_le(h + 131 + 8 * c, (uint64_t)__double_as_longlong(L.scale[c]), 8);
            put_le(h + 155 + 8 * c, (uint64_t)__double_as_longlong(L.off[c]), 8);
            const bool any = L.n > 0;
            // X * scale + offset as NumPy evaluates it: a rounded product, then a rounded sum (an fma differs in the last bit)
            const double vmax = any ? __dadd_rn(__dmul_rn((double)L.minmax[2 * c + 1], L.scale[c]), L.off[c]) : 0.0;
            const double vmin = any ? __dadd_rn(__dmul_rn((double)L.minmax[2 * c], L.scale[c]), L.off[c]) : 0.0;
            put_le(h + 179 + 16 * c, (uint64_t)__double_as_longlong(vmax), 8);
            put_le(h + 187 + 16 * c, (uint64_t)__double_as_longlong(vmin), 8);
        }
    }
    __syncthreads();
    for (int i = tid; i < kLasHeader; i += blockDim.x) L.out[i] = h[i];
}

__global__ void k_las_init(int32_t* mm) { if (threadIdx.x < 6) mm[threadIdx.x] = (threadIdx.x & 1) ? INT32_MIN : INT32_MAX; }

// parts: 1 = records of points [p_begin, n) + min / max reduction into L.minmax, 2 = header from L.minmax, 3 = both
cudaError_t launch_las_pf3(bool f64, const LasParams& L, int parts, cudaStream_t st) {
    const int64_t tiles = (L.n - L.p_begin + kLasTile - 1) / kLasTile;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    if (parts & 1) {
        k_las_init<<<1, 32, 0, st>>>(L.minmax);
        if (tiles > 0) {
            if (f64) k_las_records<true><<<(unsigned)tiles, kLasThreads, 0, st>>>(L);
            else     k_las_records<false><<<(unsigned)tiles, kLasThreads, 0, st>>>(L);
        }
    }
    if (parts & 2) k_las_header<<<1, 256, 0, st>>>(L);
    return cudaGetLastError();
}

}  // namespace lmc
