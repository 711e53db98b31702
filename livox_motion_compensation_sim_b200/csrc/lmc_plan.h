// lmc_plan.h -- which point kernel serves an aligned-cloud call (lmc_align_rigid_*, lmc_deskew_*, lmc_quantize_*).
// Host-only and free of CUDA headers, so that the decision can be compiled and checked by a plain C++ compiler.
#pragma once
#include <cstdint>
#include <type_traits>
#include "../../include/lmc_b200.h"

namespace lmc {

// kSlerpLocal: Mode C's per-point pose, then into the sensor frame of the frame's reference pose (pose_Rt, one row per
// frame): every point of a frame in the sensor frame of one instant, rotation and translation removed
// kSlerpDistort: the inverse of Mode C -- a world point into the sensor frame of Mode C's pose at the point's own time
// (what a moving sensor records of a static world)
enum Mode : int { kRigid = 0, kGyro = 1, kSlerp = 2, kQuantOnly = 3, kSlerpLocal = 4, kSlerpDistort = 5 };
constexpr bool slerp_mode(int mode) { return mode == kSlerp || mode == kSlerpLocal || mode == kSlerpDistort; }
template <int MODE> inline constexpr bool kSlerpFamily = slerp_mode(MODE);      // (the same, usable in device code)

// One launch = one Params block in constant/param space.
struct Params {
    const void*     pts;          // (N,4) f64 or (N) float4
    void*           out;          // same layout, may be null
    const void*     ts;           // int64[N] (f64 layout) | uint32[N] ns offsets (f32 layout)
    const int64_t*  frame_off;    // CSR, n_frames + 1
    const int64_t*  frame_start;  // int64[n_frames] ns
    const double*   pose_Rt;      // Mode A: (n_frames, 12) | kSlerpLocal: reference pose per frame, same layout
    const int64_t*  samp_ts;      // Mode B: imu_ts | Mode C: sample_ts
    const double*   samp_tab;     // Mode B: imu_gyro (S,3) | Mode C: seg (S,20)
    const int32_t*  hold_idx;     // Mode C hold-next (optional)
    int64_t         n_samp;
    int64_t         n_points, p_begin, p_end;
    int32_t         n_frames;
    // fused export epilogues
    uint8_t*        lvx14;
    const uint8_t*  tag;
    int32_t*        las_x;
    int32_t*        las_y;
    int32_t*        las_z;
    uint16_t*       las_int;
    uint32_t*       status;
    double          las_scale[3], las_rcp[3], las_off[3];      // las_rcp = 1/scale (host, correctly rounded)
    int32_t         lvx_mode, las_int_mode;
    // fused merged-cloud assembly: peer-mapped copies of out / lvx14 on the other ranks
    int32_t         n_peers;
    void*           peer_out[LMC_MAX_PEERS];
    uint8_t*        peer_lvx[LMC_MAX_PEERS];
    // the same through the NVSwitch multicast mapping of the symmetric buffers (multimem.st)
    void*           mc_out;
    uint8_t*        mc_lvx;
};

// k_stream tile shape (measured on B200, see profiles/): 15 consumer warps + 1 producer warp (512 threads -> 128 registers
// each).  Mode C on float4 points amortises its per-tile bookkeeping best with 3 point pairs per thread (over a 3-stage
// ring); everything else runs 2 pairs (f32) / 1 pair (f64) per thread.  (Sensor-frame deskew holds a reference pose row
// besides Mode C's: with 3 pairs its LVX2 variant spills twice what Mode C's lean variants do, with 2 it spills less.
// Distortion holds exactly Mode C's registers and runs Mode C's shape.)
constexpr int kCW = 15;
constexpr int stream_pairs_per_thread(bool f64, int mode) { return f64 ? 1 : ((mode == kSlerp || mode == kSlerpDistort) ? 3 : 2); }
constexpr int stream_tile_points(bool f64, int mode) { return kCW * 32 * 2 * stream_pairs_per_thread(f64, mode); }   // 960 / 1920 / 2880

// k_stream export variants: the export configuration known at compile time ("lean" kernels) or tested at run time
// (kExGeneric).  Lean variants also assume what plan_point_launch has verified: LVX records are type-2-of-input without
// tag bytes, timestamps / frame starts are present where the mode needs them, no hold_idx, 2 <= n_samp < 2^31 - 1.
// kExLvx2 (with kExLvx): the records are CS:365-374 on the COMPENSATED point (+ optional tag bytes) instead of LMC:252-272 on
// the raw one -- the second simulator's product, lean for Mode B and for sensor-frame deskew.
// kExMc (with kExOut | kExLvx): fused merged-cloud assembly through the NVSwitch multicast mapping of the symmetric buffers --
// every result of a full tile leaves as ONE multimem.st (the switch replicates it into every rank's copy, this rank's
// included) instead of a local store plus one store per peer; ragged edge tiles fall back to local + per-peer stores.
// kExPb (with kExOut | kExLvx): fused merged-cloud assembly by TMA BULK stores -- the warp writes its results back over its own
// points in the stage, and its contiguous run of the tile (aligned cloud) plus its record slab leave as one bulk store per
// destination (this rank's copy and every peer's over NVLink) instead of one register store per result and peer.
constexpr int kExOut = 1, kExLvx = 2, kExLas = 4, kExGeneric = 8, kExLvx2 = 16, kExMc = 32, kExPb = 64;

struct Plan {
    int         rc = LMC_OK;      // LMC_OK, or the LMC_ERR_* code the call is refused with
    const char* msg = "";         // why it is refused
    bool        stream = false;   // k_stream<F64, MODE, ex> (true) or k_fused<F64, MODE> (false)
    int         ex = 0;           // k_stream's export variant
    int64_t     tile0 = 0;        // k_stream: first point of the first tile (tiles are aligned in GLOBAL index space) ...
    int64_t     n_tiles = 0;      // ... number of tiles up to p_end ...
    int         grid = 0;         // ... and CTAs (persistent: at most one per SM)
};

inline Plan refuse_call(const char* msg) {
    Plan pl;
    pl.rc = LMC_ERR_INVALID;
    pl.msg = msg;
    return pl;
}

// why a kSlerpLocal / kSlerpDistort call with peer or multicast pointers is refused
inline const char* no_merge_reason(int mode) {
    return mode == kSlerpLocal ? "sensor-frame deskew has no merged-cloud assembly (each frame is in its own sensor frame)"
                               : "distortion has no merged-cloud assembly (each point is in its own sensor frame)";
}

// path: lmc_set_path (0 direct, 1 auto, 2 streaming); sm_count: the current device's.  P is a validated, non-empty call.
inline Plan plan_point_launch(bool f64, int mode, const Params& P, int path, int sm_count) {
    Plan pl;
    if ((mode == kSlerpLocal || mode == kSlerpDistort) && (P.n_peers > 0 || P.mc_out || P.mc_lvx))
        return refuse_call(no_merge_reason(mode));
    const int64_t tp = stream_tile_points(f64, mode);
    pl.tile0 = (P.p_begin / tp) * tp;
    pl.n_tiles = (P.p_end - pl.tile0 + tp - 1) / tp;
    const bool peers = P.n_peers > 0;                       // peer stores exist in the streaming kernels only
    const bool small = pl.n_tiles < 2 * (int64_t)sm_count;  // too few tiles to fill a persistent grid
    // TMA sources must be 16-byte aligned: guaranteed by the 32-byte rule for points, not for timestamps / tags
    const bool tma_ok = !((reinterpret_cast<uintptr_t>(P.ts) | reinterpret_cast<uintptr_t>(P.tag)) & 15u);
    if (!tma_ok || (!peers && (path == 0 || (path == 1 && small)))) {
        if (peers) return refuse_call("peer stores need the streaming kernels (16-byte aligned timestamp / tag arrays)");
        return pl;
    }
    pl.stream = true;
    pl.grid = (int)(pl.n_tiles < sm_count ? pl.n_tiles : sm_count);
    pl.ex = kExGeneric;
    if (mode == kQuantOnly) return pl;                      // (multicast pointers are ignored: there is no aligned cloud to merge)
    const int mask = (P.out ? kExOut : 0) | (P.lvx14 ? kExLvx : 0) | ((P.las_x || P.las_int) ? kExLas : 0);
    const bool lvx2 = P.lvx14 && P.lvx_mode == LMC_LVX2_OF_OUTPUT;
    const bool mc = P.mc_out && P.mc_lvx;
    // the only shape with merged-cloud kernels (multicast / peer bulk stores): f32 Mode A / C, aligned cloud + type-2 LVX
    const bool merge_shape = !f64 && mode != kGyro && mask == (kExOut | kExLvx) && !lvx2;
    const bool pb = !mc && peers && merge_shape;
    const bool timed = P.ts && P.n_samp >= 2 && P.n_samp < 0x7fffffffLL;
    if (mode == kSlerpLocal) {                              // lean: the aligned cloud, alone or with LVX2 records of it
        const bool lean_local = timed && (f64 || P.frame_start) && (mask == kExOut || (mask == (kExOut | kExLvx) && lvx2));
        if (lean_local) pl.ex = lvx2 ? (kExOut | kExLvx | kExLvx2) : kExOut;
        return pl;
    }
    if (mode == kSlerpDistort) {                            // lean: the raw cloud alone; any export is the generic kernel's
        if (timed && (f64 || P.frame_start) && mask == kExOut) pl.ex = kExOut;
        return pl;
    }
    bool lean = (!peers || mc || pb) && (!lvx2 || mode == kGyro) && (!(mask & kExLas) || (P.las_x && P.las_int));
    if (mode == kSlerp) lean = lean && !P.hold_idx && timed && (f64 || P.frame_start);
    if (mode == kGyro)  lean = lean && timed && P.frame_start;
    if (mc && !(merge_shape && lean))
        return refuse_call("no multicast kernel for this call (there is one for f32 Mode A / C exporting the aligned cloud + type-2 LVX records)");
    if (!lean) return pl;
    if (mc)      pl.ex = kExOut | kExLvx | kExMc;
    else if (pb) pl.ex = kExOut | kExLvx | kExPb;
    else if (mask == kExOut || mask == (kExOut | kExLas)) pl.ex = mask;
    else if (mask == (kExOut | kExLvx)) pl.ex = lvx2 ? (kExOut | kExLvx | kExLvx2) : mask;   // (lean with LVX2 records: Mode B only)
    return pl;
}

// The one layout x mode -> template switch of both kernel families: fn(std::bool_constant<F64>, std::integral_constant<int, MODE>).
template <class Fn>
auto dispatch_layout_mode(bool f64, int mode, Fn&& fn) {
    using T = std::true_type;
    using F = std::false_type;
    switch (mode) {                                         // (mode is one of the six Modes: default = kQuantOnly)
    case kRigid: return f64 ? fn(T{}, std::integral_constant<int, kRigid>{}) : fn(F{}, std::integral_constant<int, kRigid>{});
    case kGyro:  return f64 ? fn(T{}, std::integral_constant<int, kGyro>{})  : fn(F{}, std::integral_constant<int, kGyro>{});
    case kSlerp: return f64 ? fn(T{}, std::integral_constant<int, kSlerp>{}) : fn(F{}, std::integral_constant<int, kSlerp>{});
    case kSlerpLocal: return f64 ? fn(T{}, std::integral_constant<int, kSlerpLocal>{}) : fn(F{}, std::integral_constant<int, kSlerpLocal>{});
    case kSlerpDistort: return f64 ? fn(T{}, std::integral_constant<int, kSlerpDistort>{}) : fn(F{}, std::integral_constant<int, kSlerpDistort>{});
    default:     return f64 ? fn(T{}, std::integral_constant<int, kQuantOnly>{}) : fn(F{}, std::integral_constant<int, kQuantOnly>{});
    }
}

}  // namespace lmc
