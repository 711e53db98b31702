// lmc_tma.cu -- persistent, warp-specialised streaming kernels (the default path on large inputs).
//
// One CTA per SM, 15 consumer warps + 1 producer warp, each CTA walks a contiguous run of tiles.
//
//   producer warp   per tile: find the frames intersecting the tile (one coalesced read of the CSR
//                   offsets after the previous tile's frame), then ONE elected lane issues TMA bulk
//                   copies (cp.async.bulk global -> shared, UBLKCP) for the tile's points / timestamps
//                   / tag bytes into a 4-stage ring; completion is signalled on an mbarrier with
//                   expect_tx.  Up to 4 x 42 KB are in flight per SM, independent of registers.
//   consumer warps  wait on the stage's "full" mbarrier, pull their point pairs out of shared memory,
//                   resolve frames, release the stage ("empty" mbarrier) and only then do the f64
//                   work: pose / sample-row fetch (L1 broadcast), transform, quantise.  Results leave
//                   straight from registers as 256-bit stores (aligned cloud) and 64-bit SoA stores
//                   (LAS ints); the 14-byte LVX records are transposed through a warp-private shared
//                   slab (7 words per point pair, conflict-free) and leave as ONE TMA bulk store per warp and tile, so the
//                   output side needs no CTA-wide barrier at all.
//
// Edge tiles (a shard's ragged first / last tile) skip TMA and take guarded global loads.
#include <type_traits>
#include "lmc_device.cuh"

namespace lmc {

constexpr int kStreamThreads = 32 * (kCW + 1);           // + producer warp

// tile shape: lmc_plan.h (the launch plan sizes the grid with the same tile)
template <bool F64, int MODE> struct StreamCfg {
    static constexpr int PPT      = stream_pairs_per_thread(F64, MODE);   // point pairs per consumer thread per tile
    static constexpr int STAGES   = (!F64 && (MODE == kSlerp || MODE == kSlerpDistort)) ? 3 : 4;
    static constexpr int TP       = stream_tile_points(F64, MODE);
    static constexpr int PT_BYTES = F64 ? 32 : 16;
    static constexpr int TS_BYTES = F64 ? 8 : 4;
    static constexpr int PTS_STAGE = TP * PT_BYTES;
    static constexpr int TS_STAGE  = TP * TS_BYTES;
    static constexpr int TAG_STAGE = TP;
    static constexpr int STAGE     = PTS_STAGE + TS_STAGE + TAG_STAGE;
    static constexpr int LVX_SLAB  = PPT * 64 * 14;              // bytes per consumer warp
    static constexpr int ROWS      = (kSlerpFamily<MODE> && !F64) ? 12 : 0;   // pose rows staged per tile (Mode C, float4 layout): a 2880-point tile of a 10 us / 200 Hz stream touches 7
    static constexpr int ROW_STAGE = ROWS * kSegStride * 8;
    static constexpr int SMEM      = STAGES * (STAGE + ROW_STAGE) + kCW * LVX_SLAB + STAGES * (int)sizeof(TileMeta) + STAGES * 64 + 2 * STAGES * 8 + 128;
    static_assert(SMEM <= 227 * 1024, "stage ring does not fit the 227 KB of shared memory a CTA can have");
};

// Everything a consumer needs to know about a tile, prepared once by the producer (64 bytes = four
// broadcast LDS.128): bounds, and -- when the tile holds at most one frame boundary ("simple", the
// common case) -- the frame facts themselves, so consumers never touch TileMeta.
struct TileInfo {
    int64_t base, lim_lo, lim_hi;
    int32_t full;                 // 1: whole tile inside [p_begin, p_end) and staged by TMA
    int32_t f_lo;                 // frame of the tile's first point
    int32_t rel_e1;               // tile-local index of the first point of frame f_lo + 1 (INT_MAX: none)
    int32_t flags;                // bit 0 simple, bit 1 / 2: frame f_lo / f_lo + 1 holds exactly one point
    int64_t fs0, fs1;             // frame_start of f_lo and f_lo + 1 (Mode B/C)
    int32_t k_base, n_rows;       // Mode C: pose rows [k_base, k_base + n_rows) are staged in shared memory with the tile
};

// ---- mbarrier / bulk-copy PTX ---------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra D;\n\tbra W;\n\tD:\n\t}"
        :: "r"(bar), "r"(parity), "r"(0x100000u) : "memory");
}
// global -> shared bulk copy (TMA, 1-D): 16-byte aligned addresses, size multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// 16 bytes to the multicast address (PTX multimem.st; the switch fans the write out to every member of the group)
__device__ __forceinline__ void mc_st128(void* mc, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(mc), "f"(__uint_as_float(a)), "f"(__uint_as_float(b)), "f"(__uint_as_float(c)), "f"(__uint_as_float(d)) : "memory");
}

// ---- one tile on the consumer side ------------------------------------------------------------
template <bool F64, int MODE, int EX, bool FULL>
__device__ __forceinline__ void consume_tile(const Params& P, const TileInfo& ti, const TileMeta& tm,
                                             const uint8_t* s_pts, const uint8_t* s_ts, const uint8_t* s_tag,
                                             uint8_t* slab, uint32_t empty_bar, PointCtx<F64, MODE>& ctx,
                                             uint32_t& fl, int cw, int lane, uint32_t info_s = 0, uint32_t rows_s = 0)
{
    using Cfg = StreamCfg<F64, MODE>;
    constexpr int PPT = Cfg::PPT;
    constexpr bool GEN = EX == kExGeneric;
    constexpr bool MC = !GEN && (EX & kExMc);                    // full tiles: multimem.st only; edge tiles: local + per-peer stores
    constexpr bool PB = !GEN && (EX & kExPb) && !F64;            // full tiles: results written back into the stage, bulk stores per destination
    const bool do_out = GEN ? P.out != nullptr : bool(EX & kExOut);
    const bool do_lvx = GEN ? P.lvx14 != nullptr : bool(EX & kExLvx);
    const bool do_las = GEN ? (P.las_x != nullptr || P.las_int != nullptr) : bool(EX & kExLas);
    const bool has_ts = (MODE == kGyro || kSlerpFamily<MODE>) && (GEN ? P.ts != nullptr : true);
    const bool has_fs = (MODE == kGyro || kSlerpFamily<MODE>) && (GEN ? P.frame_start != nullptr : (MODE == kGyro || !F64));
    constexpr bool LVX2 = !GEN && (EX & kExLvx2);                // lean, records of the output
    const bool has_tag = LVX2 ? P.tag != nullptr : (GEN && do_lvx && P.tag != nullptr && P.lvx_mode == LMC_LVX2_OF_OUTPUT);
    const int64_t base = ti.base;

    // tile-level frame facts (prepared by the producer) in registers
    const int32_t m_flo = ti.f_lo, rel_e1 = ti.rel_e1;
    const bool m_simple = MODE == kQuantOnly || (ti.flags & 1), m_single0 = ti.flags & 2, m_single1 = ti.flags & 4;
    const int64_t m_fs0 = ti.fs0, m_fs1 = ti.fs1;

    // Lean full tiles hand the warp's LVX records (one contiguous, 16-byte aligned run of the output) to the TMA engine
    // as ONE bulk store out of the warp-private slab: no LDS + STG round trip through registers, full-line writes,
    // and the store drains while the warp is already in the next tile (V5: 86 -> 93 % of the measured peak).  The LAS
    // integers (four short runs per warp) gain nothing from it and keep their register stores.
    if (do_lvx) {                                                // (edge tiles too: the tile before them may have been a full one)
        if (lane == 0) bulk_wait_read0();                        // the previous tile's bulk store has finished READING the slab
        __syncwarp();                                            // ... and every lane is done with its own reads of it
    }
    // one point pair at a time: stage -> registers -> f64 work -> stores (short live ranges); the
    // stage is handed back to the producer as soon as the LAST pair has been pulled out of it
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
        // keep pair j+1's shared-memory loads behind pair j's work: hoisting all pairs' inputs to the top
        // of the tile makes ptxas spill a dozen doubles per pair
        if (j > 0) asm volatile("" ::: "memory");
        const int q = (cw * PPT + j) * 32 + lane;            // pair index inside the tile
        const int64_t p = base + 2 * q;
        const bool va = FULL || (p >= ti.lim_lo && p < ti.lim_hi), vb = FULL || (p + 1 >= ti.lim_lo && p + 1 < ti.lim_hi);
        Pt in[2];
        float wraw[2] = {0.f, 0.f};
        int64_t tsv[2] = {0, 0};
        uint32_t tagv = 0;
        in[0] = in[1] = Pt{ 0.0, 0.0, 0.0, 0.0 };
        if constexpr (FULL) {
            if constexpr (F64) {
                const double2* s = reinterpret_cast<const double2*>(s_pts) + 4 * q;
                const double2 pa0 = s[0], pa1 = s[1], pb0 = s[2], pb1 = s[3];
                in[0] = Pt{ pa0.x, pa0.y, pa1.x, pa1.y }; in[1] = Pt{ pb0.x, pb0.y, pb1.x, pb1.y };
                if (has_ts) { const longlong2 t = reinterpret_cast<const longlong2*>(s_ts)[q]; tsv[0] = t.x; tsv[1] = t.y; }
            } else {
                const float4* s = reinterpret_cast<const float4*>(s_pts) + 2 * q;
                const float4 ra = s[0], rb = s[1];
                in[0] = Pt{ (double)ra.x, (double)ra.y, (double)ra.z, (double)ra.w };
                in[1] = Pt{ (double)rb.x, (double)rb.y, (double)rb.z, (double)rb.w };
                wraw[0] = ra.w; wraw[1] = rb.w;
                if (has_ts) { const uint2 t = reinterpret_cast<const uint2*>(s_ts)[q]; tsv[0] = t.x; tsv[1] = t.y; }
            }
            if (has_tag) tagv = reinterpret_cast<const uint16_t*>(s_tag)[q];
        } else {
            load_pair<F64, false>(P.pts, p, va, vb, in[0], in[1]);
            wraw[0] = (float)in[0].w; wraw[1] = (float)in[1].w;
            if (has_ts) {
                if constexpr (F64) { const int64_t* t = reinterpret_cast<const int64_t*>(P.ts) + p; if (va) tsv[0] = __ldg(t); if (vb) tsv[1] = __ldg(t + 1); }
                else { const uint32_t* t = reinterpret_cast<const uint32_t*>(P.ts) + p; if (va) tsv[0] = __ldg(t); if (vb) tsv[1] = __ldg(t + 1); }
            }
            if (has_tag) { if (va) tagv |= __ldg(P.tag + p); if (vb) tagv |= (uint32_t)__ldg(P.tag + p + 1) << 8; }
        }
        int32_t fr[2] = {0, 0}; bool single[2] = {false, false}; int64_t fsv[2] = {0, 0};
        if constexpr (MODE != kQuantOnly) {
            if (m_simple) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const bool second = 2 * q + h >= rel_e1;
                    fr[h] = m_flo + (second ? 1 : 0);
                    if constexpr (MODE == kRigid) single[h] = second ? m_single1 : m_single0;
                    fsv[h] = second ? m_fs1 : m_fs0;
                }
            } else {
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (FULL || (h == 0 ? va : vb)) {
                        fr[h] = frame_of(P, tm, p + h, single[h]);
                        if (has_fs) fsv[h] = frame_start_of(P, tm, fr[h]);
                    }
            }
        }
        // with staged pose rows the stage is still being read by ctx.pair() below: release it after the last pair's math
        constexpr bool ROWS_STAGED = FULL && !GEN && kSlerpFamily<MODE> && !F64;   // (f64 tiles are one pair per thread: holding the stage through the math costs more than the row reads)
        constexpr bool PB_FULL = PB && FULL;                 // the stage is the staging buffer of the bulk stores: released after they have read it
        if (j == PPT - 1 && !ROWS_STAGED && !PB_FULL) {      // everything this warp needs from the stage is in registers
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_bar);
        }

        if constexpr (!GEN && !LVX2) {
            // lean: the LVX record is LMC:252-272 on the RAW input point -- independent of the transform,
            // so pack it first and let its temporaries die before the FP64-heavy part
            if (do_lvx) {
                uint32_t x[2] = {0, 0}, y[2] = {0, 0}, z[2] = {0, 0}, rt[2] = {0, 0}, nan = 0;
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (FULL || (h == 0 ? va : vb)) {
                        x[h] = (uint32_t)q_mm_clip<false>(in[h].x, nan); y[h] = (uint32_t)q_mm_clip<false>(in[h].y, nan);
                        z[h] = (uint32_t)q_mm_clip<false>(in[h].z, nan); rt[h] = q_refl<false>(in[h].w, nan);
                    }
                if (nan) {                                       // rare: a NaN field quantises to 0
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        if (in[h].x != in[h].x) x[h] = 0;
                        if (in[h].y != in[h].y) y[h] = 0;
                        if (in[h].z != in[h].z) z[h] = 0;
                        if (in[h].w != in[h].w) rt[h] = 0;
                    }
                    fl |= nan;
                }
                lvx_pair_words(reinterpret_cast<uint32_t*>(slab) + 7 * (j * 32 + lane), x, y, z, rt);
            }
        }
        Pt o[2] = { in[0], in[1] };
        if (FULL || (va && vb)) ctx.template pair<!GEN, ROWS_STAGED>(P, fr, single, fsv, tsv, in, o, info_s, rows_s);
        else {
            if (va) o[0] = ctx.one(P, fr[0], single[0], fsv[0], tsv[0], in[0]);
            if (vb) o[1] = ctx.one(P, fr[1], single[1], fsv[1], tsv[1], in[1]);
        }
        if (j == PPT - 1 && ROWS_STAGED && !PB_FULL) {
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_bar);
        }
        if (do_out) {
            if constexpr (F64) store_pair<true, FULL>(P.out, p, va, vb, o[0], o[1]);
            else {
                float* dst = reinterpret_cast<float*>(P.out) + 4 * p;
                if constexpr (PB_FULL) {
                    float4* sp = reinterpret_cast<float4*>(const_cast<uint8_t*>(s_pts)) + 2 * q;       // over the pair's own input
                    sp[0] = make_float4((float)o[0].x, (float)o[0].y, (float)o[0].z, wraw[0]);
                    sp[1] = make_float4((float)o[1].x, (float)o[1].y, (float)o[1].z, wraw[1]);
                } else if constexpr (MC && FULL) {
                    float* mc = reinterpret_cast<float*>(P.mc_out) + 4 * p;
                    mc_st128(mc, __float_as_uint((float)o[0].x), __float_as_uint((float)o[0].y), __float_as_uint((float)o[0].z), __float_as_uint(wraw[0]));
                    mc_st128(mc + 4, __float_as_uint((float)o[1].x), __float_as_uint((float)o[1].y), __float_as_uint((float)o[1].z), __float_as_uint(wraw[1]));
                } else if (FULL || (va && vb)) {
                    const float v[8] = { (float)o[0].x, (float)o[0].y, (float)o[0].z, wraw[0], (float)o[1].x, (float)o[1].y, (float)o[1].z, wraw[1] };
                    stg256(dst, v);
                } else {
                    if (va) *reinterpret_cast<float4*>(dst)     = make_float4((float)o[0].x, (float)o[0].y, (float)o[0].z, wraw[0]);
                    if (vb) *reinterpret_cast<float4*>(dst + 4) = make_float4((float)o[1].x, (float)o[1].y, (float)o[1].z, wraw[1]);
                }
            }
        }
        if constexpr (GEN || ((MC || PB) && !FULL)) {
            // fused merged-cloud assembly: the same pair goes to every peer's copy of the merged buffer
            for (int r = 0; r < P.n_peers; ++r)
                if (P.peer_out[r] != nullptr) store_pair<F64, FULL>(P.peer_out[r], p, va, vb, o[0], o[1]);
        }
        if (do_las) store_las_pair<FULL, MODE == kRigid>(P, p, va, vb, o[0], o[1], fl);
        if constexpr (GEN || LVX2) {
            if (do_lvx) {
                uint32_t x[2] = {0, 0}, y[2] = {0, 0}, z[2] = {0, 0}, rt[2] = {0, 0};
                if (FULL || va) lvx_words<MODE>(P, in[0], o[0], tagv & 0xffu, x[0], y[0], z[0], rt[0], fl);
                if (FULL || vb) lvx_words<MODE>(P, in[1], o[1], (tagv >> 8) & 0xffu, x[1], y[1], z[1], rt[1], fl);
                lvx_pair_words(reinterpret_cast<uint32_t*>(slab) + 7 * (j * 32 + lane), x, y, z, rt);
            }
        }
    }
    if (do_lvx) {
        // the warp's PPT x 64 records are contiguous in the output
        const int64_t wfirst = base + 2 * (int64_t)(cw * PPT) * 32;          // first point of the warp's block
        uint8_t* g = P.lvx14 + 14 * wfirst;
        constexpr int NB = PPT * 64 * 14;
        if constexpr (PB && FULL) {
            // the warp's PPT x 64 results are one contiguous run of the stage (16 bytes per point) and of every destination
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
                constexpr uint32_t OB = PPT * 64 * 16;
                const uint8_t* src = s_pts + 16 * (size_t)(cw * PPT) * 64;
                bulk_s2g(reinterpret_cast<uint8_t*>(P.out) + 16 * wfirst, src, OB);
                bulk_s2g(g, slab, NB);
                for (int r = 0; r < P.n_peers; ++r) {
                    if (P.peer_out[r] != nullptr) bulk_s2g(reinterpret_cast<uint8_t*>(P.peer_out[r]) + 16 * wfirst, src, OB);
                    if (P.peer_lvx[r] != nullptr) bulk_s2g(P.peer_lvx[r] + 14 * wfirst, slab, NB);
                }
                bulk_commit();
                bulk_wait_read0();                                   // stage and slab have been read: hand the stage back
                mbar_arrive(empty_bar);
            }
        } else if constexpr (MC && FULL) {
            __syncwarp();
            uint8_t* mc = P.mc_lvx + 14 * wfirst;
            for (int i = lane; i < NB / 16; i += 32) {
                const uint4 v = reinterpret_cast<const uint4*>(slab)[i];
                mc_st128(mc + 16 * i, v.x, v.y, v.z, v.w);
            }
        } else if constexpr (FULL) {
            fence_async_smem();
            __syncwarp();
            if (lane == 0) { bulk_s2g(g, slab, NB); bulk_commit(); }
        } else {
            __syncwarp();
            int64_t lo = ti.lim_lo - wfirst, hi = ti.lim_hi - wfirst;
            lo = lo < 0 ? 0 : lo; hi = hi > PPT * 64 ? PPT * 64 : hi;
            if (lo < hi) {
                const int b0 = (int)lo * 14, b1 = (int)hi * 14;
                int a0 = (b0 + 15) & ~15; if (a0 > b1) a0 = b1;
                int a1 = b1 & ~15;        if (a1 < a0) a1 = a0;
                for (int i = a0 / 16 + lane; i < a1 / 16; i += 32) reinterpret_cast<uint4*>(g)[i] = reinterpret_cast<const uint4*>(slab)[i];
                for (int i = b0 + lane; i < a0; i += 32) g[i] = slab[i];
                for (int i = a1 + lane; i < b1; i += 32) g[i] = slab[i];
            }
        }
        if constexpr (GEN || ((MC || PB) && !FULL)) {
            for (int r = 0; r < P.n_peers; ++r) {
                uint8_t* gp = P.peer_lvx[r];
                if (gp == nullptr) continue;
                gp += 14 * wfirst;
                if constexpr (FULL) {
                    for (int i = lane; i < NB / 16; i += 32) reinterpret_cast<uint4*>(gp)[i] = reinterpret_cast<const uint4*>(slab)[i];
                } else {
                    int64_t lo = ti.lim_lo - wfirst, hi = ti.lim_hi - wfirst;
                    lo = lo < 0 ? 0 : lo; hi = hi > PPT * 64 ? PPT * 64 : hi;
                    for (int i = (int)lo * 14 + lane; i < (int)hi * 14; i += 32) gp[i] = slab[i];
                }
            }
        }
    }                                                                         // (the next tile waits for the slab at its top)
}

template <bool F64, int MODE, int EX>
__device__ __forceinline__ void stream_body(const Params& P, int64_t tile0, int64_t n_tiles)
{
    using Cfg = StreamCfg<F64, MODE>;
    constexpr bool GEN = EX == kExGeneric;
    extern __shared__ __align__(128) uint8_t smem[];                            // no static smem in this kernel: base is aligned
    uint8_t*  s_stage = smem;                                                   // Cfg::STAGES x STAGE
    uint8_t*  s_slab  = s_stage + Cfg::STAGES * Cfg::STAGE;                         // kCW x LVX_SLAB
    TileMeta* s_meta  = reinterpret_cast<TileMeta*>(s_slab + kCW * Cfg::LVX_SLAB);
    TileInfo* s_info  = reinterpret_cast<TileInfo*>(s_meta + Cfg::STAGES);
    uint64_t* s_full  = reinterpret_cast<uint64_t*>(s_info + Cfg::STAGES);
    uint64_t* s_empty = s_full + Cfg::STAGES;
    uint8_t*  s_rows  = reinterpret_cast<uint8_t*>(s_empty + Cfg::STAGES);        // Cfg::STAGES x ROW_STAGE (16-byte aligned)

    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    asm volatile("" : "+r"(warp), "+r"(lane));                                  // keep them in registers (no S2R re-reads in the loop)
    const int64_t t_begin = n_tiles * (int64_t)blockIdx.x / gridDim.x;
    const int32_t my_tiles = (int32_t)(n_tiles * (int64_t)(blockIdx.x + 1) / gridDim.x - t_begin);   // <= 2^31 tiles per CTA

    if (threadIdx.x == 0) {
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(smem_u32(s_full + s), 1); mbar_init(smem_u32(s_empty + s), kCW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t full0 = smem_u32(s_full), empty0 = smem_u32(s_empty);       // barrier s lives at +8*s

    const bool has_ts = (MODE == kGyro || kSlerpFamily<MODE>) && (GEN ? P.ts != nullptr : true);
    const bool has_tag = (GEN || (EX & kExLvx2)) && P.lvx14 != nullptr && P.tag != nullptr && P.lvx_mode == LMC_LVX2_OF_OUTPUT;

    if (warp == kCW) {
        // ================================ producer warp ==========================================
        int s = 0; uint32_t ph = 0;
        int64_t hint = -1;
        int64_t base = tile0 + t_begin * Cfg::TP;
        [[maybe_unused]] int64_t p_t0 = 0; [[maybe_unused]] double p_rate = 0.0;   // same bracket guess as PointCtx::init
        if constexpr (kSlerpFamily<MODE> && !GEN && !F64) {
            p_t0 = __ldg(P.samp_ts);
            const int64_t span = __ldg(P.samp_ts + P.n_samp - 1) - p_t0;
            p_rate = span > 0 ? (double)(P.n_samp - 1) / (double)span : 0.0;
        }
        for (int32_t it = 0; it < my_tiles; ++it, base += Cfg::TP) {
            mbar_wait(empty0 + 8 * s, ph ^ 1);                                   // slot free (first lap passes)
            const int64_t lim_lo = base > P.p_begin ? base : P.p_begin;
            const int64_t lim_hi = base + Cfg::TP < P.p_end ? base + Cfg::TP : P.p_end;
            const bool full = lim_lo == base && lim_hi == base + Cfg::TP;
            if constexpr (MODE != kQuantOnly) {
                tile_meta(P, lim_lo, lim_hi - 1, s_meta[s], lane, hint);
                __syncwarp();
                hint = (int64_t)s_meta[s].f_lo + (s_meta[s].overflow ? 0 : s_meta[s].nb);   // frame of the tile's last point
            }
            if (lane == 0) {
                TileInfo inf{ base, lim_lo, lim_hi, full ? 1 : 0, 0, 0x7fffffff, 1, 0, 0, 0, 0 };
                if constexpr (MODE != kQuantOnly) {
                    const TileMeta& tm = s_meta[s];
                    const int32_t nb = tm.nb;
                    const bool simple = !tm.overflow && nb <= 1;
                    inf.f_lo = tm.f_lo;
                    inf.flags = simple ? 1 : 0;
                    if (simple) {
                        const int64_t e1 = tm.edge[1];
                        if (nb == 1) inf.rel_e1 = (int32_t)(e1 - base);
                        if (e1 - tm.edge[0] == 1) inf.flags |= 2;
                        if (tm.edge[nb + 1] - e1 == 1) inf.flags |= 4;
                        if (P.frame_start != nullptr) { inf.fs0 = tm.fstart[0]; inf.fs1 = tm.fstart[nb]; }
                    }
                }
                uint32_t row_bytes = 0;
                const double* row_src = nullptr;
                if constexpr (kSlerpFamily<MODE> && !GEN && !F64) {
                    // the pose rows this tile reads, from the times of its first and last point (exact for time-ordered
                    // points; anything outside the staged window is simply read from global memory by the consumer)
                    if (full && !s_meta[s].overflow && (reinterpret_cast<uintptr_t>(P.samp_tab) & 15u) == 0) {
                        int64_t ta, tb;
                        if constexpr (F64) {
                            ta = __ldg(reinterpret_cast<const int64_t*>(P.ts) + lim_lo); tb = __ldg(reinterpret_cast<const int64_t*>(P.ts) + lim_hi - 1);
                        } else {
                            ta = (int64_t)__ldg(reinterpret_cast<const uint32_t*>(P.ts) + lim_lo) + s_meta[s].fstart[0];
                            tb = (int64_t)__ldg(reinterpret_cast<const uint32_t*>(P.ts) + lim_hi - 1) + s_meta[s].fstart[s_meta[s].nb];
                        }
                        int64_t ka = (int64_t)__double2ll_rz((double)(ta - p_t0) * p_rate) - 1, kb = (int64_t)__double2ll_rz((double)(tb - p_t0) * p_rate) + 2;
                        ka = ka < 0 ? 0 : ka; kb = kb > P.n_samp ? P.n_samp : kb;
                        if (kb > ka) {
                            if (kb - ka > Cfg::ROWS) kb = ka + Cfg::ROWS;
                            inf.k_base = (int32_t)ka; inf.n_rows = (int32_t)(kb - ka);
                            row_bytes = (uint32_t)(kb - ka) * (uint32_t)(kSegStride * 8);
                            row_src = P.samp_tab + kSegStride * ka;
                        }
                    }
                }
                s_info[s] = inf;
                uint8_t* st = s_stage + s * Cfg::STAGE;
                if (full) {
                    const uint32_t bytes = Cfg::PTS_STAGE + (has_ts ? Cfg::TS_STAGE : 0) + (has_tag ? Cfg::TAG_STAGE : 0) + row_bytes;
                    mbar_arrive_expect_tx(full0 + 8 * s, bytes);
                    if (row_bytes) bulk_g2s(s_rows + s * Cfg::ROW_STAGE, row_src, row_bytes, full0 + 8 * s);
                    bulk_g2s(st, reinterpret_cast<const uint8_t*>(P.pts) + base * Cfg::PT_BYTES, Cfg::PTS_STAGE, full0 + 8 * s);
                    if (has_ts)  bulk_g2s(st + Cfg::PTS_STAGE, reinterpret_cast<const uint8_t*>(P.ts) + base * Cfg::TS_BYTES, Cfg::TS_STAGE, full0 + 8 * s);
                    if (has_tag) bulk_g2s(st + Cfg::PTS_STAGE + Cfg::TS_STAGE, P.tag + base, Cfg::TAG_STAGE, full0 + 8 * s);
                } else {
                    mbar_arrive(full0 + 8 * s);                                    // edge tile: consumers read global memory
                }
            }
            __syncwarp();
            if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
        }
    } else {
        // ================================ consumer warps =========================================
        PointCtx<F64, MODE> ctx;
        ctx.init(P);
        uint32_t fl = 0;
        uint8_t* slab = s_slab + warp * Cfg::LVX_SLAB;
        int s = 0; uint32_t ph = 0;
        for (int32_t it = 0; it < my_tiles; ++it) {
            mbar_wait(full0 + 8 * s, ph);
            const TileInfo ti = s_info[s];
            const uint8_t* st = s_stage + s * Cfg::STAGE;
            if (ti.full) consume_tile<F64, MODE, EX, true>(P, ti, s_meta[s], st, st + Cfg::PTS_STAGE, st + Cfg::PTS_STAGE + Cfg::TS_STAGE, slab, empty0 + 8 * s, ctx, fl, warp, lane,
                                                           smem_u32(s_info + s), smem_u32(s_rows + s * Cfg::ROW_STAGE));
            else         consume_tile<F64, MODE, EX, false>(P, ti, s_meta[s], st, st + Cfg::PTS_STAGE, st + Cfg::PTS_STAGE + Cfg::TS_STAGE, slab, empty0 + 8 * s, ctx, fl, warp, lane);
            if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
        }
        if constexpr (GEN || (EX & kExLvx)) { if (lane == 0) bulk_wait0(); }                   // bulk stores of the last tile (all destinations)
        if (fl != 0 && P.status != nullptr) atomicOr(P.status, fl);
    }
}
// (stream_body stays a separate inline function: folding it into k_stream changes the machine code of k_stream's instantiations)
template <bool F64, int MODE, int EX>
__global__ void __launch_bounds__(kStreamThreads, 1) k_stream(const __grid_constant__ Params P, int64_t tile0, int64_t n_tiles) {
    stream_body<F64, MODE, EX>(P, tile0, n_tiles);
}

// ---- launcher ----------------------------------------------------------------------------------
template <bool F64, int MODE, int EX>
static cudaError_t launch_stream_ex(const Params& P, const Plan& pl, int dev, cudaStream_t st) {
    using Cfg = StreamCfg<F64, MODE>;
    void (*kern)(const Params, int64_t, int64_t) = k_stream<F64, MODE, EX>;
    static thread_local int attr_dev = -1;
    if (attr_dev != dev) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
        if (e != cudaSuccess) return e;
        attr_dev = dev;
    }
    kern<<<pl.grid, kStreamThreads, Cfg::SMEM, st>>>(P, pl.tile0, pl.n_tiles);
    return cudaGetLastError();
}

// the variant plan_point_launch chose (the instantiations below are every variant it can choose)
cudaError_t launch_stream(bool f64, int mode, const Params& P, const Plan& pl, int dev, cudaStream_t st) {
    return dispatch_layout_mode(f64, mode, [&](auto f64_c, auto mode_c) -> cudaError_t {
        constexpr bool F64 = decltype(f64_c)::value;
        constexpr int MODE = decltype(mode_c)::value;
        if constexpr (MODE == kSlerpLocal) {
            if (pl.ex == kExOut)                    return launch_stream_ex<F64, MODE, kExOut>(P, pl, dev, st);
            if (pl.ex == (kExOut | kExLvx | kExLvx2)) return launch_stream_ex<F64, MODE, kExOut | kExLvx | kExLvx2>(P, pl, dev, st);
        } else if constexpr (MODE == kSlerpDistort) {
            if (pl.ex == kExOut)                    return launch_stream_ex<F64, MODE, kExOut>(P, pl, dev, st);
        } else if constexpr (MODE != kQuantOnly) {
            switch (pl.ex) {
            case kExOut:           return launch_stream_ex<F64, MODE, kExOut>(P, pl, dev, st);
            case kExOut | kExLvx:  return launch_stream_ex<F64, MODE, kExOut | kExLvx>(P, pl, dev, st);
            case kExOut | kExLas:  return launch_stream_ex<F64, MODE, kExOut | kExLas>(P, pl, dev, st);
            }
            if constexpr (MODE == kGyro) {
                if (pl.ex == (kExOut | kExLvx | kExLvx2)) return launch_stream_ex<F64, MODE, kExOut | kExLvx | kExLvx2>(P, pl, dev, st);
            } else if constexpr (!F64) {
                if (pl.ex == (kExOut | kExLvx | kExMc)) return launch_stream_ex<F64, MODE, kExOut | kExLvx | kExMc>(P, pl, dev, st);
                if (pl.ex == (kExOut | kExLvx | kExPb)) return launch_stream_ex<F64, MODE, kExOut | kExLvx | kExPb>(P, pl, dev, st);
            }
        }
        if (pl.ex == kExGeneric) return launch_stream_ex<F64, MODE, kExGeneric>(P, pl, dev, st);
        return cudaErrorInvalidValue;
    });
}

}  // namespace lmc
