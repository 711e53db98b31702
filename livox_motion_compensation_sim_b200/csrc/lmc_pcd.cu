// lmc_pcd.cu -- (SURVEY 8f N2) ASCII text on the device, byte-identical to CPython's "%.{d}f" (correctly rounded,
// round-half-even on the exact binary value -- the same rule as C printf).  Two writers:
//   k_pcd_*   the per-point line of LiDARMotionSimulator.save_pcd (LMC:946-947) for every row of an (N,4) array
//                 f"{x:.6f} {y:.6f} {z:.6f} {intensity:.6f}\n"
//   k_text_*  generic delimited rows, "%.{d}f" with d = 0..9 per column (the complete simulator's exports, CS:1643-1716)
//
// Both print through one exact number core (fmtg_prepare): |v| splits into its integer part ip = trunc(|v|) (< 2^64) and
// fq = round_half_even(frac * 10^d), all in exact FP64 steps, and emit_number prints (ip, fq) in SWAR groups of four digits.
// The PCD writer takes the core only for its slow numbers (>= 10^4, nan, inf) and caps their magnitude at 9.2e12 (pcd_prepare);
// every other number -- every coordinate a LiDAR produces -- takes its branch-free fast path (piece_fast).
//
// Lines have variable length, so the text is produced in three launches:
//   k_pcd_len    per tile of 256 points: total text bytes of the tile.  The length of "%.6f" needs no digits: it is
//                sign + 7 + the digit count of the ROUNDED integer part, and |v| rounds up to 10^k exactly when
//                |v| >= 10^k - 5e-7 -- a real number no double equals, so comparing with the first double above it
//                (kDigitT) is exact.  Four compares per number; HBM-bound.
//   k_pcd_scan   one CTA: exclusive prefix sum of the tile sizes -> byte offset of every tile
//   k_pcd_write  per tile: format, lay the lines out in shared memory (block scan of the line lengths) and copy the
//                tile's contiguous byte range out as one TMA bulk store.  Numbers below 10^4 take a branch-free path: digit
//                pairs by arithmetic, characters packed into words in registers and streamed into the image as aligned
//                32-bit stores (LineStream below); the slow numbers go through the number core and emit_number.
#include <cstdlib>
#include "lmc_device.cuh"

namespace lmc {

constexpr int kPcdTile    = 256;                    // points (= threads) per tile

// ---- the number core: "%.{d}f" of a double, d = 0..9 ------------------------------------------------------------------
// One formatted number: integer part, d fractional digits as an integer, text length, special-value kind
struct Num { uint64_t ip; uint32_t fq; uint32_t len; uint8_t kind; bool neg; };   // kind 0 finite, 1 nan, 2 inf

__device__ __constant__ uint32_t kPow10[10] = { 1u, 10u, 100u, 1000u, 10000u, 100000u, 1000000u, 10000000u, 100000000u, 1000000000u };
__device__ __constant__ double kPow10d[10] = { 1.0, 10.0, 100.0, 1.0e3, 1.0e4, 1.0e5, 1.0e6, 1.0e7, 1.0e8, 1.0e9 };

// Digit count of the ROUNDED integer part of "%.{d}f" % a without making a digit: the printed value reaches 10^k exactly when
// a >= 10^k - 0.5 * 10^-d (a tie there goes to the even neighbour, and 10^(k+d) is even), so the count is found by comparing with
// kTextT[d][k] = the smallest double >= that real number (generated with exact fractions; tests/test_host.py re-derives the table).
// Which k to compare with follows from the binary exponent: 2^e <= a < 2^(e+1) has floor(e * log10 2) + 1 or + 2 digits.
__device__ const double kTextT[10][20] = {
    { 0.0, 0x1.3000000000000p+3, 0x1.8e00000000000p+6, 0x1.f3c0000000000p+9, 0x1.387c000000000p+13, 0x1.869f800000000p+16, 0x1.e847f00000000p+19, 0x1.312cff0000000p+23, 0x1.7d783fe000000p+26, 0x1.dcd64ffc00000p+29, 0x1.2a05f1ffc0000p+33, 0x1.74876e7ff8000p+36, 0x1.d1a94a1fff000p+39, 0x1.2309ce53fff00p+43, 0x1.6bcc41e8fffe0p+46, 0x1.c6bf52633fffcp+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3e66666666667p+3, 0x1.8fccccccccccdp+6, 0x1.f3f999999999ap+9, 0x1.387f99999999ap+13, 0x1.869ff33333334p+16, 0x1.e847fe6666667p+19, 0x1.312cffe666667p+23, 0x1.7d783ffcccccdp+26, 0x1.dcd64fff9999ap+29, 0x1.2a05f1fff999ap+33, 0x1.74876e7fff334p+36, 0x1.d1a94a1fffe67p+39, 0x1.2309ce53fffe7p+43, 0x1.6bcc41e8ffffdp+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3fd70a3d70a3ep+3, 0x1.8ffae147ae148p+6, 0x1.f3ff5c28f5c29p+9, 0x1.387ff5c28f5c3p+13, 0x1.869ffeb851eb9p+16, 0x1.e847ffd70a3d8p+19, 0x1.312cfffd70a3ep+23, 0x1.7d783fffae148p+26, 0x1.dcd64ffff5c29p+29, 0x1.2a05f1ffff5c3p+33, 0x1.74876e7fffeb9p+36, 0x1.d1a94a1ffffd8p+39, 0x1.2309ce53ffffep+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3ffbe76c8b43ap+3, 0x1.8fff7ced91688p+6, 0x1.f3ffef9db22d1p+9, 0x1.387ffef9db22ep+13, 0x1.869fffdf3b646p+16, 0x1.e847fffbe76c9p+19, 0x1.312cffffbe76dp+23, 0x1.7d783ffff7ceep+26, 0x1.dcd64ffffef9ep+29, 0x1.2a05f1ffffefap+33, 0x1.74876e7ffffe0p+36, 0x1.d1a94a1fffffcp+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3fff972474539p+3, 0x1.8ffff2e48e8a8p+6, 0x1.f3fffe5c91d15p+9, 0x1.387fffe5c91d2p+13, 0x1.869ffffcb923bp+16, 0x1.e847ffff97248p+19, 0x1.312cfffff9725p+23, 0x1.7d783fffff2e5p+26, 0x1.dcd64fffffe5dp+29, 0x1.2a05f1fffffe6p+33, 0x1.74876e7fffffdp+36, 0x1.d1a94a2000000p+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3ffff583a53b9p+3, 0x1.8ffffeb074a78p+6, 0x1.f3ffffd60e94fp+9, 0x1.387ffffd60e95p+13, 0x1.869fffffac1d3p+16, 0x1.e847fffff583bp+19, 0x1.312cffffff584p+23, 0x1.7d783fffffeb1p+26, 0x1.dcd64ffffffd7p+29, 0x1.2a05f1ffffffep+33, 0x1.74876e8000000p+36, 0x1.d1a94a2000000p+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3ffffef390860p+3, 0x1.8fffffde7210cp+6, 0x1.f3fffffbce422p+9, 0x1.387fffffbce43p+13, 0x1.869ffffff79c9p+16, 0x1.e847fffffef3ap+19, 0x1.312cffffffef4p+23, 0x1.7d783ffffffdfp+26, 0x1.dcd64fffffffcp+29, 0x1.2a05f20000000p+33, 0x1.74876e8000000p+36, 0x1.d1a94a2000000p+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3fffffe5280d7p+3, 0x1.8ffffffca501bp+6, 0x1.f3ffffff94a04p+9, 0x1.387ffffff94a1p+13, 0x1.869fffffff295p+16, 0x1.e847ffffffe53p+19, 0x1.312cfffffffe6p+23, 0x1.7d783fffffffdp+26, 0x1.dcd6500000000p+29, 0x1.2a05f20000000p+33, 0x1.74876e8000000p+36, 0x1.d1a94a2000000p+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3ffffffd50ce3p+3, 0x1.8fffffffaa19dp+6, 0x1.f3fffffff5434p+9, 0x1.387fffffff544p+13, 0x1.869fffffffea9p+16, 0x1.e847fffffffd6p+19, 0x1.312cffffffffep+23, 0x1.7d78400000000p+26, 0x1.dcd6500000000p+29, 0x1.2a05f20000000p+33, 0x1.74876e8000000p+36, 0x1.d1a94a2000000p+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
    { 0.0, 0x1.3fffffffbb47ep+3, 0x1.8ffffffff7690p+6, 0x1.f3fffffffeed2p+9, 0x1.387fffffffeeep+13, 0x1.869ffffffffdep+16, 0x1.e847ffffffffcp+19, 0x1.312d000000000p+23, 0x1.7d78400000000p+26, 0x1.dcd6500000000p+29, 0x1.2a05f20000000p+33, 0x1.74876e8000000p+36, 0x1.d1a94a2000000p+39, 0x1.2309ce5400000p+43, 0x1.6bcc41e900000p+46, 0x1.c6bf526340000p+49, 0x1.1c37937e08000p+53, 0x1.6345785d8a000p+56, 0x1.bc16d674ec800p+59, 0x1.158e460913d00p+63 },
};
__device__ __forceinline__ uint32_t text_nd(double a, int d) {        // 0 <= a < 2^64
    const int e = (int)(((uint32_t)__double2hiint(a) >> 20) & 0x7ffu) - 1023;
    const int k0 = e > 0 ? (e * 1233) >> 12 : 0;
    return (uint32_t)k0 + 1u + (a >= __ldg(&kTextT[d][k0 + 1]) ? 1u : 0u);
}

// q = round_half_even(fr * p10) on the exact product, for 0 <= fr < 1 and p10 = 10^d (d >= 1: at most 21 significant bits).
// hi + lo = fr * p10 exactly (FMA error term).  RNE(hi) is the answer unless hi sits exactly on a tie k + 0.5 -- the only place
// where lo can change the decision (k + 0.5 is itself a double and rounding is monotonic); on an exact tie (lo == 0) RNE(hi) is
// already the even last printed digit.
__device__ __forceinline__ uint32_t round_frac(double fr, double p10) {
    const double hi = __dmul_rn(fr, p10);
    uint32_t q = __double2uint_rn(hi);
    if (fabs(__dsub_rn(hi, __uint2double_rn(q))) == 0.5) {
        const double lo = __fma_rn(fr, p10, -hi);
        const uint32_t dn = __double2uint_rz(hi);
        if (lo > 0.0) q = dn + 1u; else if (lo < 0.0) q = dn;
    }
    return q;
}

// ip = trunc(|v|) (exact below 2^64), fr = |v| - ip (exact), q = round_frac(fr, 10^d), carried into ip when it reaches 10^d.
// Finite |v| >= 2^64 is saturated to 2^64 - 1 and flagged LMC_FLAG_OVERFLOW.
__device__ __forceinline__ Num fmtg_prepare(double v, int d, uint32_t& fl) {
    Num t;
    const uint64_t bits = (uint64_t)__double_as_longlong(v);
    t.neg = bits >> 63;
    t.ip = 0; t.fq = 0; t.kind = 0;
    const double a = fabs(v);
    if (d == 0 && a < 18446744073709551616.0) {      // '%.0f': one round-to-nearest-even conversion IS the answer (a < 2^64 - 1024)
        t.ip = __double2ull_rn(a);
        t.len = (t.neg ? 1u : 0u) + text_nd(a, 0);
        return t;
    }
    if (a < 18446744073709551616.0) {                // 2^64
        uint64_t ip = __double2ull_rz(a);
        const double fr = __dsub_rn(a, __ull2double_rn(ip));
        uint32_t q = round_frac(fr, kPow10d[d]);
        if (q >= kPow10[d]) { q -= kPow10[d]; ip += 1; }
        t.ip = ip; t.fq = q;
        t.len = (t.neg ? 1u : 0u) + text_nd(a, d) + (d ? 1u + (uint32_t)d : 0u);
        return t;
    } else if (a != a) {
        t.kind = 1; t.len = 3u; return t;
    } else if (isinf(a)) {
        t.kind = 2; t.len = t.neg ? 4u : 3u; return t;
    } else {
        fl |= LMC_FLAG_OVERFLOW; t.ip = 0xffffffffffffffffull;
    }
    t.len = (t.neg ? 1u : 0u) + 20u + (d ? 1u + (uint32_t)d : 0u);     // finite >= 2^64: saturated to 2^64 - 1 (20 digits), flagged
    return t;
}

// ---- the PCD writer's numbers ----------------------------------------------------------------------------------------
// The PCD writer prints |v| < 9.2e12 only.  That bounds a number at 13 integer digits and a line at kLineMax = 88 bytes, which
// sizes k_pcd_write's 44 KB tile image; with the core's full range (20 integer digits) a line would take 116 bytes and the image
// 58 KB, and four f32 CTAs (__launch_bounds__(256, 4)) would no longer fit in an SM's shared memory.  No point cloud coordinate
// gets near the cap: a finite |v| >= 9.2e12 prints as "9199999999999.999999" (with its sign) and sets LMC_FLAG_OVERFLOW.
constexpr int kNumMax     = 1 + 13 + 1 + 6;         // sign + 13 integer digits + '.' + 6 decimals
constexpr int kLineMax    = 4 * kNumMax + 4;        // 3 spaces + newline
__device__ __forceinline__ Num pcd_prepare(double v, uint32_t& fl) {
    const double a = fabs(v);
    if (a >= 9.2e12 && !isinf(a)) {
        fl |= LMC_FLAG_OVERFLOW;
        const bool neg = __double_as_longlong(v) < 0;
        return Num{9199999999999ull, 999999u, (neg ? 1u : 0u) + 20u, 0, neg};
    }
    return fmtg_prepare(v, 6, fl);
}

// ---- fast path: |v| below 10^4 after rounding (at most 4 integer digits) ------------------------------------------
// kDigitT[k-1] = the smallest double >= 10^k - 5e-7 (= kTextT[6][k]); for a float-valued |v| the same thresholds are
// 10, 100, 1000, 10000 (the float just below 10^k prints 9...9.99....).
__device__ __constant__ double kDigitT[4] = { 0x1.3ffffef390860p+3, 0x1.8fffffde7210cp+6, 0x1.f3fffffbce422p+9, 0x1.387fffffbce43p+13 };

// (slow-path helpers return by value: a reference to the caller's flag word or arrays would pin them in local memory)
__device__ __noinline__ uint2 pcd_len_slow_eval(double v) { uint32_t fl = 0; const uint32_t len = pcd_prepare(v, fl).len; return make_uint2(len, fl); }
__device__ __forceinline__ uint32_t pcd_len_slow(double v, uint32_t& fl) { const uint2 r = pcd_len_slow_eval(v); fl |= r.y; return r.x; }

// text length of "%.6f" % v, without any digit: four compares
__device__ __forceinline__ uint32_t fmt_len(double v, uint32_t& fl) {
    const double a = fabs(v);
    if (!(a < kDigitT[3])) return pcd_len_slow(v, fl);              // >= 10^4, inf, nan
    return ((uint32_t)__double2hiint(v) >> 31) + 8u + (a >= kDigitT[0]) + (a >= kDigitT[1]) + (a >= kDigitT[2]);
}
__device__ __forceinline__ uint32_t fmt_len(float v, uint32_t& fl) {
    const float a = fabsf(v);
    if (!(a < 10000.0f)) return pcd_len_slow((double)v, fl);
    return (__float_as_uint(v) >> 31) + 8u + (a >= 10.0f) + (a >= 100.0f) + (a >= 1000.0f);
}

// ---- rows ------------------------------------------------------------------------------------------------------------
template <bool F64>
__device__ __forceinline__ double load_cell(const void* rows, int64_t idx) {
    if constexpr (F64) return __ldg(reinterpret_cast<const double*>(rows) + idx);
    else return (double)__ldg(reinterpret_cast<const float*>(rows) + idx);
}
// the row in its own type (float4 rows are formatted from the floats: no conversion, f32 compares)
template <bool F64> struct RowT { using T = double; };
template <> struct RowT<false> { using T = float; };
template <bool F64>
__device__ __forceinline__ void load_row_native(const void* pts, int64_t i, typename RowT<F64>::T (&v)[4]) {
    if constexpr (F64) { const double* s = reinterpret_cast<const double*>(pts) + 4 * i; ldg256(s, v[0], v[1], v[2], v[3]); }
    else { const float4 f = __ldg(reinterpret_cast<const float4*>(pts) + i); v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w; }
}
// a thread's two consecutive rows (the formatting kernels work on 2 points per thread)
template <bool F64>
__device__ __forceinline__ void rows_load(const void* __restrict__ pts, int64_t row0, bool v0, bool v1, typename RowT<F64>::T (&v)[8]) {
    using T = typename RowT<F64>::T;
    if (v0) load_row_native<F64>(pts, row0, reinterpret_cast<T (&)[4]>(v[0]));
    else { v[0] = v[1] = v[2] = v[3] = 0; }
    if (v1) load_row_native<F64>(pts, row0 + 1, reinterpret_cast<T (&)[4]>(v[4]));
    else { v[4] = v[5] = v[6] = v[7] = 0; }
}
template <bool F64>
__device__ __forceinline__ uint32_t rows_len(bool v0, bool v1, const typename RowT<F64>::T (&v)[8], uint32_t& fl) {
    uint32_t len = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (h == 0 ? v0 : v1) {
            len += 4u;
#pragma unroll
            for (int c = 0; c < 4; ++c) len += fmt_len(v[4 * h + c], fl);
        }
    }
    return len;
}

__device__ __forceinline__ uint32_t block_scan_excl(uint32_t x, uint32_t* s_warp, uint32_t& total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < kPcdTile / 32; ++k) { const uint32_t t = s_warp[k]; if (k < w) base += t; tot += t; }
    total = tot;
    return base + inc - x;
}

// ---- digits: every number of a line as three registers ---------------------------------------------------------------
// The first version of this formatter spent 646 instructions per point, most of them on digit extraction (divisions by
// constants per digit pair, a table, byte stores into shared memory).  Now: SWAR -- 4 ASCII digits per 8 integer instructions,
// no table -- and the characters stay packed in registers until they leave as whole 32-bit words (LineStream).
constexpr int kFmtThreads = 256;
constexpr int kFmtTile    = 2 * kFmtThreads;                              // points per tile: 2 consecutive points per thread
constexpr int kFmtImg     = ((kFmtTile * kLineMax + 32 + 15) / 16) * 16;
static_assert(kFmtTile == 2 * kPcdTile, "tile_off has kPcdTile granularity: the two halves of a formatting tile");

// x < 10^4 -> its 4 decimal digits as ASCII, thousands in byte 0.  Two 2-digit lanes in one register:
// h | l << 16 with h = x / 100, l = x % 100; tens of both lanes by one multiply (n * 103 >> 10 == n / 10 for n < 100).
__device__ __forceinline__ uint32_t swar4(uint32_t x) {
    const uint32_t h = __umulhi(x, 42949673u);                            // ceil(2^32 / 100): exact quotient for x < 10^4
    const uint32_t P = (x - 100u * h) * 65536u + h;
    const uint32_t t = ((P * 103u) >> 10) & 0x000f000fu;
    return P * 256u + 0x30303030u - 2559u * t;                            // tens + (ones << 8) + "0000", per lane
}

// One number ready for the stream: the lead (sign + integer digits, ll = 1..5 bytes) and the fixed 8-byte tail ".dddddd<sep>".
//   T0 = [ll, d, d, d] (ll rides in byte 0, where the '.' goes),  T1 = [d, d, d, sep]
//   ll <= 4: L0 holds the ll lead bytes;  ll == 5: "-dddd", L0 holds the four digits;
//   ll & kPieceSlow: the number core prints it (|v| >= 10^4, nan, inf): L0 = text length incl. separator, T1 = the last
//   four bytes of the text (what the next thread's first word needs)
struct Piece { uint32_t L0, T0, T1; };
constexpr uint32_t kPieceSlow = 0x80u;
__device__ __forceinline__ uint32_t piece_ll(const Piece& p) { return p.T0 & 0xffu; }
__device__ __forceinline__ uint32_t piece_len(const Piece& p) { const uint32_t ll = piece_ll(p); return (ll & kPieceSlow) ? p.L0 : ll + 8u; }

__device__ __forceinline__ void piece_finish(Piece& p, uint32_t ip, uint32_t q, uint32_t neg, uint32_t sepw) {
    const uint32_t carry = q == 1000000u ? 1u : 0u;                      // 0.9999995 -> 1.000000
    q = carry ? 0u : q;
    ip += carry;
    const uint32_t A = swar4(ip);
    const uint32_t lz = (uint32_t)(__ffs((int)((A ^ 0x30303030u) | 0x01000000u)) - 1) >> 3;   // leading zero digits, at most 3
    const uint32_t digits = A >> (8u * lz), ll = 4u - lz + neg;
    p.L0 = ll == 5u ? digits : ((digits << (8u * neg)) | (neg ? 0x2du : 0u));
    const uint32_t q1 = __umulhi(q, 429497u), r = q - q1 * 10000u;       // ceil(2^32 / 10^4): exact for q < 10^6
    const uint32_t C = swar4(r);
    const uint32_t t = (q1 * 205u) >> 11;                                 // q1 / 10 for q1 < 100
    const uint32_t X = q1 * 65536u + 0x303000u - 655104u * t + ll;        // ll, tens, ones of q1 in bytes 0..2
    p.T0 = __byte_perm(X, C, 0x4210);
    p.T1 = __byte_perm(C, sepw, 0x4321);
}
__device__ __noinline__ uint3 piece_slow_eval(double v, uint32_t sepw) {     // {T1, text length incl. separator, status flags}
    uint32_t fl = 0;
    const Num t = pcd_prepare(v, fl);
    uint32_t t1;
    if (t.kind) t1 = (t.kind == 1 ? 0x006e616eu : 0x00666e69u) | (sepw << 24);            // "nan" / "inf" + separator
    else t1 = __byte_perm(swar4(t.fq % 10000u), sepw, 0x4321);
    return make_uint3(t1, t.len + 1u, fl);
}
__device__ __forceinline__ void piece_slow(Piece& p, double v, uint32_t sepw, uint32_t& fl) {
    const uint3 r = piece_slow_eval(v, sepw);
    p.L0 = r.y; p.T0 = kPieceSlow; p.T1 = r.x;
    fl |= r.z;
}
// The fast formulas run unconditionally on every number (a slow number -- |v| >= 10^4, nan, inf -- just yields garbage that the
// thread's ONE fix-up branch replaces): no branch per number in the common case.
// float4 layout: |v| - trunc(|v|) is exact in f32 and its product with 10^6 = 2^6 * 15625 is exact in f64 (24 + 14 bits),
// so ONE round-to-nearest-even conversion is printf's rounding of the exact binary value -- no tie handling at all
__device__ __forceinline__ bool piece_fast(Piece& p, float v, uint32_t sepw) {
    const float a = fabsf(v);
    const uint32_t ip = __float2uint_rz(a);
    const float fr = __fsub_rn(a, __uint2float_rn(ip));
    piece_finish(p, ip, __double2uint_rn(__dmul_rn((double)fr, 1.0e6)), __float_as_uint(v) >> 31, sepw);
    return !(a < 10000.0f);
}
// f64: the core's rounding of the exact fraction (the FMA error term decides only on a tie)
__device__ __forceinline__ bool piece_fast(Piece& p, double v, uint32_t sepw) {
    const double a = fabs(v);
    const uint32_t ip = __double2uint_rz(a);
    const double fr = __dsub_rn(a, __uint2double_rn(ip));
    piece_finish(p, ip, round_frac(fr, 1.0e6), (uint32_t)__double2hiint(v) >> 31, sepw);
    return !(a < kDigitT[3]);
}
__device__ __forceinline__ bool is_slow(float v) { return !(fabsf(v) < 10000.0f); }
__device__ __forceinline__ bool is_slow(double v) { return !(fabs(v) < kDigitT[3]); }
// the 8 numbers of a thread's two rows; returns the text length of both lines.  special: some piece needs more than
// put(lead) + put8(tail) in the stream (a slow number or a 5-byte lead "-dddd")
template <bool F64>
__device__ __forceinline__ uint32_t rows_pieces(bool v0, bool v1, const typename RowT<F64>::T (&v)[8], Piece (&pc)[8], bool& special, uint32_t& fl) {
    bool slow = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) slow |= piece_fast(pc[k], v[k], (k & 3) == 3 ? 0x0au : 0x20u);      // (invalid rows hold zeros: "0.000000")
    if (slow) {
#pragma unroll
        for (int k = 0; k < 8; ++k) if (is_slow(v[k])) piece_slow(pc[k], (double)v[k], (k & 3) == 3 ? 0x0au : 0x20u, fl);
    }
    uint32_t len = 0, odd = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const bool valid = k < 4 ? v0 : v1;
        if (valid) { len += piece_len(pc[k]); odd |= piece_ll(pc[k]) + 3u; }      // bit 3 or 7 set <=> ll > 4
    }
    special = (odd & 0x88u) != 0u;
    return len;
}

// ---- text assembly: the thread's two lines as a stream of aligned 32-bit words into the tile image ----------------------
// (byte stores were the bottleneck of the first version: 52 STS.U8 + 20 table LDS per line, the LSU data pipe 86 % busy; an
// intermediate version OR-ed the word shared by two neighbouring lines into a zero-filled image with shared-memory atomics.)
// A 1..4-byte piece is appended to a pending word with two funnel shifts, the fixed 8-byte tail of every number leaves as two
// whole words.  The word a thread shares with its predecessor starts from that thread's last bytes (handed over by shuffle /
// shared memory before the stream starts), the word it shares with its successor is left to the successor: every word of
// the image is stored exactly once, complete -- no atomics, no zero fill.
struct LineStream {
    uint32_t addr, sh, a0;          // pending word: its shared-memory address, 8 x the bytes already in it (0, 8, 16, 24), its value
    __device__ __forceinline__ void sts(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
    // the pending word starts with the last (pos & 3) bytes of the previous thread's text (prev_t1 = that text's last 4 bytes)
    __device__ __forceinline__ void start(uint32_t img_s, uint32_t pos, uint32_t prev_t1) {
        addr = img_s + (pos & ~3u); sh = 8u * (pos & 3u); a0 = __funnelshift_l(prev_t1, 0u, sh);
    }
    template <int MODE = 0>                                              // (MODE: see emit_u8; unused here)
    __device__ __forceinline__ void put(uint32_t chunk, uint32_t k) {   // the k (1..4) low bytes of chunk, the others 0
        const uint32_t w0 = a0 | (chunk << sh);
        const uint32_t hi = __funnelshift_l(chunk, 0u, sh);               // the bytes that did not fit (0 when sh == 0)
        const uint32_t nsh = sh + 8u * k;
        const bool full = nsh >= 32u;
        if (full) sts(addr, w0);
        addr += full ? 4u : 0u; a0 = full ? hi : w0; sh = nsh & 31u;
    }
    template <int MODE = 0>
    __device__ __forceinline__ void put4(uint32_t w) {                  // 4 bytes: one whole word leaves
        sts(addr, a0 | (w << sh));
        a0 = __funnelshift_l(w, 0u, sh);
        addr += 4u;
    }
    __device__ __forceinline__ void put8(uint32_t lo, uint32_t hi) {    // 8 bytes: two whole words leave
        sts(addr, a0 | (lo << sh));
        sts(addr + 4u, __funnelshift_l(lo, hi, sh));
        a0 = __funnelshift_l(hi, 0u, sh);
        addr += 8u;
    }
    __device__ __forceinline__ void flush() { if (sh) sts(addr, a0); }   // only where no later thread completes the word
};
// Word stream of one row into the (zero-filled) tile image.  Rows of the generic writer are heterogeneous (any mix of column
// widths), so the word a row shares with its predecessor is not handed over in registers as in the PCD writer: the row's FIRST
// completed word and its last partial word are OR-ed into the image (shared-memory atomics commute), every word in between is
// a plain store.
struct TextStream {
    uint32_t addr, sh, a0; bool first;
    __device__ __forceinline__ void start(uint32_t img_s, uint32_t pos) { addr = img_s + (pos & ~3u); sh = 8u * (pos & 3u); a0 = 0u; first = true; }
    // MODE 0: plain store; 1: OR (the word may be the one shared with the previous row); 2: decide at run time (generic formats)
    template <int MODE>
    __device__ __forceinline__ void out(uint32_t w) {
        if (MODE == 1 || (MODE == 2 && first)) { asm volatile("red.shared.or.b32 [%0], %1;" :: "r"(addr), "r"(w) : "memory"); first = false; }
        else asm volatile("st.shared.u32 [%0], %1;" :: "r"(addr), "r"(w) : "memory");
        addr += 4u;
    }
    template <int MODE>
    __device__ __forceinline__ void put(uint32_t chunk, uint32_t k) {   // the k (1..4) low bytes of chunk, the others 0
        const uint32_t w0 = a0 | (chunk << sh);
        const uint32_t hi = __funnelshift_l(chunk, 0u, sh);
        const uint32_t nsh = sh + 8u * k;
        if (nsh >= 32u) { out<MODE>(w0); a0 = hi; } else a0 = w0;
        sh = nsh & 31u;
    }
    template <int MODE>
    __device__ __forceinline__ void put4(uint32_t w) { out<MODE>(a0 | (w << sh)); a0 = __funnelshift_l(w, 0u, sh); }
    __device__ __forceinline__ void finish() { if (sh) asm volatile("red.shared.or.b32 [%0], %1;" :: "r"(addr), "r"(a0) : "memory"); }
};
// The digit emitters write into either word stream: MODE is TextStream's store mode, a LineStream stores every word plainly.
// x < 10^8 printed with nd (1..8) digits / with all 8 digits
template <int MODE, class Stream>
__device__ __forceinline__ void emit_u8(Stream& ts, uint32_t x, uint32_t nd) {
    if (nd > 4u) {
        const uint32_t h = (uint32_t)(((uint64_t)x * 3518437209ull) >> 45);       // x / 10^4, exact for 32-bit x
        ts.template put<MODE>(swar4(h) >> (8u * (8u - nd)), nd - 4u);
        ts.template put4<MODE>(swar4(x - h * 10000u));
    } else ts.template put<MODE>(swar4(x) >> (8u * (4u - nd)), nd);
}
template <int MODE, class Stream>
__device__ __forceinline__ void emit_u8_full(Stream& ts, uint32_t x) {
    const uint32_t h = (uint32_t)(((uint64_t)x * 3518437209ull) >> 45);
    ts.template put4<MODE>(swar4(h));
    ts.template put4<MODE>(swar4(x - h * 10000u));
}
// one number + separator: sign, integer digits in groups of four (SWAR), fraction, separator
template <int MODE, class Stream>
__device__ __forceinline__ void emit_number(Stream& ts, const Num& t, int d, uint32_t sep) {
    if (t.kind) {                                                      // "nan" | "inf" | "-inf"
        if (t.kind == 2 && t.neg) ts.template put<MODE>(0x2du, 1u);
        ts.template put<MODE>(t.kind == 1 ? 0x006e616eu : 0x00666e69u, 3u);
        ts.template put<MODE>(sep, 1u);
        return;
    }
    if (t.neg) ts.template put<MODE>(0x2du, 1u);
    const uint32_t nd = t.len - (t.neg ? 1u : 0u) - (d ? 1u + (uint32_t)d : 0u);
    if (t.ip < 100000000ull) emit_u8<MODE>(ts, (uint32_t)t.ip, nd);
    else if (t.ip < 10000000000000000ull) {
        const uint64_t h = t.ip / 100000000ull;
        emit_u8<MODE>(ts, (uint32_t)h, nd - 8u);
        emit_u8_full<MODE>(ts, (uint32_t)(t.ip - h * 100000000ull));
    } else {
        const uint64_t h = t.ip / 10000000000000000ull, r = t.ip - h * 10000000000000000ull, m = r / 100000000ull;
        emit_u8<MODE>(ts, (uint32_t)h, nd - 16u);
        emit_u8_full<MODE>(ts, (uint32_t)m);
        emit_u8_full<MODE>(ts, (uint32_t)(r - m * 100000000ull));
    }
    if (d) {
        // the d fraction digits = the last d characters of the 9-digit zero-padded fq
        const uint32_t top = t.fq / 100000000u, r8 = t.fq - top * 100000000u;
        const uint32_t h = (uint32_t)(((uint64_t)r8 * 3518437209ull) >> 45);
        const uint64_t ab = (uint64_t)swar4(h) | ((uint64_t)swar4(r8 - h * 10000u) << 32);      // 8 digits, most significant in byte 0
        if (d == 6) {                                                  // ".dddddd<sep>": two whole words
            const uint64_t x = ab >> 16;
            ts.template put4<MODE>(0x2eu | ((uint32_t)x << 8));
            ts.template put4<MODE>(((uint32_t)x >> 24) | ((uint32_t)(x >> 32) << 8) | (sep << 24));
            return;
        }
        ts.template put<MODE>(0x2eu, 1u);
        if (d == 9) ts.template put<MODE>(0x30u + top, 1u);
        const uint32_t dd = d == 9 ? 8u : (uint32_t)d;
        const uint64_t x = ab >> (8u * (8u - dd));
        if (dd > 4u) { ts.template put4<MODE>((uint32_t)x); ts.template put<MODE>((uint32_t)(x >> 32), dd - 4u); }
        else ts.template put<MODE>((uint32_t)x, dd);
    }
    ts.template put<MODE>(sep, 1u);
}

template <bool F64>
__device__ __noinline__ uint3 stream_slow(uint32_t addr, uint32_t sh, uint32_t a0, const void* pts, int64_t row, int c, uint32_t sep) {
    LineStream ws{addr, sh, a0};
    uint32_t fl = 0;                                                     // (piece_slow has flagged it already)
    emit_number<0>(ws, pcd_prepare(load_cell<F64>(pts, 4 * row + c), fl), 6, sep);   // (re-read: nothing of a slow number is kept in registers)
    return make_uint3(ws.addr, ws.sh, ws.a0);
}
template <bool F64>
__device__ __forceinline__ void stream_piece(LineStream& ws, const Piece& p, const void* pts, int64_t row, int c, uint32_t sep) {
    const uint32_t ll = piece_ll(p);
    if (ll > 4u) {                                                       // rare: "-dddd" or the number core
        if (ll & kPieceSlow) { const uint3 r = stream_slow<F64>(ws.addr, ws.sh, ws.a0, pts, row, c, sep); ws.addr = r.x; ws.sh = r.y; ws.a0 = r.z; return; }
        ws.put(0x2du, 1u); ws.put(p.L0, 4u);
    } else ws.put(p.L0, ll);
    ws.put8((p.T0 & 0xffffff00u) | 0x2eu, p.T1);
}
// both lines of a thread: rows row0 / row0 + 1 start at byte `pos` of the image; `last`: the tile's last line is this thread's;
// special (rows_pieces): take the general route with its per-piece tests
template <bool F64>
__device__ __forceinline__ void rows_stream(uint32_t img_s, uint32_t pos, uint32_t prev_t1, bool v0, bool v1, bool last, bool special,
                                            const Piece (&pc)[8], const void* pts, int64_t row0) {
    if (!v0) return;
    LineStream ws;
    ws.start(img_s, pos, prev_t1);
    if (!special) {
#pragma unroll
        for (int c = 0; c < 4; ++c) { ws.put(pc[c].L0, piece_ll(pc[c])); ws.put8((pc[c].T0 & 0xffffff00u) | 0x2eu, pc[c].T1); }
        if (v1) {
#pragma unroll
            for (int c = 4; c < 8; ++c) { ws.put(pc[c].L0, piece_ll(pc[c])); ws.put8((pc[c].T0 & 0xffffff00u) | 0x2eu, pc[c].T1); }
        }
    } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) stream_piece<F64>(ws, pc[c], pts, row0, c, c == 3 ? 0x0au : 0x20u);
        if (v1) {
#pragma unroll
            for (int c = 0; c < 4; ++c) stream_piece<F64>(ws, pc[4 + c], pts, row0 + 1, c, c == 3 ? 0x0au : 0x20u);
        }
    }
    if (last) ws.flush();                                                // nobody else completes the tile's last word
}

// ---- two-call protocol: k_pcd_len + k_pcd_scan, then k_pcd_write -------------------------------------------------------
// sizes of both 256-point halves of a 512-point tile (2 points per thread): tile_off[t + 1] = bytes of half t, offsets after k_pcd_scan
constexpr int kLenTiles = 2;                                                 // formatting tiles per CTA of the size pass: both tiles' rows are in flight
                                                                             // before the first compare (f32 rows +3 %; 4 tiles: no further gain)
template <bool F64>
__global__ void __launch_bounds__(kFmtThreads) k_pcd_len(const void* __restrict__ pts, int64_t n, int64_t* __restrict__ tile_off) {
    __shared__ uint32_t s_warp[kLenTiles][kFmtThreads / 32];
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * (kLenTiles * kFmtTile) + 2 * tid;
    typename RowT<F64>::T v[kLenTiles][8];
    uint32_t fl = 0;
#pragma unroll
    for (int t = 0; t < kLenTiles; ++t) {                                    // every tile's rows in flight before the first compare
        const int64_t row0 = base + (int64_t)t * kFmtTile;
        rows_load<F64>(pts, row0, row0 < n, row0 + 1 < n, v[t]);
    }
#pragma unroll
    for (int t = 0; t < kLenTiles; ++t) {
        const int64_t row0 = base + (int64_t)t * kFmtTile;
        const uint32_t sum = __reduce_add_sync(0xffffffffu, rows_len<F64>(row0 < n, row0 + 1 < n, v[t], fl));
        if ((tid & 31) == 0) s_warp[t][tid >> 5] = sum;
    }
    __syncthreads();
    const int64_t n256 = (n + kPcdTile - 1) / kPcdTile;
    if ((tid & 127) == 0) {
#pragma unroll
        for (int t = 0; t < kLenTiles; ++t) {
            const int64_t h = 2 * ((int64_t)blockIdx.x * kLenTiles + t) + (tid >> 7);
            const uint32_t* w = s_warp[t] + 4 * (tid >> 7);
            if (h < n256) tile_off[h + 1] = w[0] + w[1] + w[2] + w[3];
        }
    }
}

// sizes -> offsets, in place, without scratch memory: tile_off[0] = 0, tile_off[t + 1] = sum of sizes[0..t].
//   pass 1 (one CTA per chunk of 1024 entries): inclusive scan inside the chunk -> its last entry is the chunk total
//   pass 2 (one CTA): the chunk totals, which sit 1024 entries apart, become global offsets
//   pass 3 (one CTA per chunk): every other entry of chunk c > 0 gets the (now global) last entry of chunk c - 1 added
// All accesses coalesced; the single-CTA scan this replaces walked 137 consecutive entries per thread and took 149 us for 140 k tiles.
constexpr int kScanChunk = 1024;
__device__ __forceinline__ int64_t cta_scan_incl(int64_t x, int64_t* s_warp) {          // 1024 threads
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int64_t t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += t; }
    if (lane == 31) s_warp[w] = x;
    __syncthreads();
    if (w == 0) {
        int64_t y = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int64_t t = __shfl_up_sync(0xffffffffu, y, o); if (lane >= o) y += t; }
        s_warp[lane] = y;
    }
    __syncthreads();
    return x + (w ? s_warp[w - 1] : 0);
}
__global__ void __launch_bounds__(kScanChunk) k_pcd_scan_chunks(int64_t* __restrict__ tile_off, int64_t n_tiles) {
    __shared__ int64_t s_warp[32];
    const int64_t k = (int64_t)blockIdx.x * kScanChunk + threadIdx.x;
    const int64_t x = cta_scan_incl(k < n_tiles ? tile_off[k + 1] : 0, s_warp);
    if (k < n_tiles) tile_off[k + 1] = x;
    if (k == 0) tile_off[0] = 0;
}
__global__ void __launch_bounds__(kScanChunk) k_pcd_scan_totals(int64_t* __restrict__ tile_off, int64_t n_tiles, int64_t n_chunks) {
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int64_t c0 = 0; c0 < n_chunks; c0 += kScanChunk) {
        const int64_t c = c0 + threadIdx.x;
        const int64_t last = (c + 1) * kScanChunk < n_tiles ? (c + 1) * kScanChunk : n_tiles;      // index of chunk c's last entry
        const int64_t x = cta_scan_incl(c < n_chunks ? tile_off[last] : 0, s_warp) + s_carry;
        __syncthreads();
        if (c < n_chunks) tile_off[last] = x;
        if (threadIdx.x == kScanChunk - 1) s_carry = x;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(kScanChunk) k_pcd_scan_add(int64_t* __restrict__ tile_off, int64_t n_tiles) {
    const int64_t c = (int64_t)blockIdx.x + 1, k = c * kScanChunk + threadIdx.x;
    const int64_t last = (c + 1) * kScanChunk < n_tiles ? (c + 1) * kScanChunk : n_tiles;
    if (k + 1 < last) tile_off[k + 1] += tile_off[c * kScanChunk];      // (entry `last` is already global)
}
static cudaError_t launch_tile_scan(int64_t* tile_off, int64_t tiles, cudaStream_t st) {
    if (tiles <= 0) return cudaMemsetAsync(tile_off, 0, sizeof(int64_t), st);
    const int64_t chunks = (tiles + kScanChunk - 1) / kScanChunk;
    k_pcd_scan_chunks<<<(unsigned)chunks, kScanChunk, 0, st>>>(tile_off, tiles);
    if (chunks > 1) {
        k_pcd_scan_totals<<<1, kScanChunk, 0, st>>>(tile_off, tiles, chunks);
        k_pcd_scan_add<<<(unsigned)(chunks - 1), kScanChunk, 0, st>>>(tile_off, tiles);
    }
    return cudaGetLastError();
}

// one 512-point tile per CTA: digits in registers, block scan of the line lengths, word stream into the image (laid out at the
// destination's 16-byte phase), one TMA bulk store
template <bool F64>
__global__ void __launch_bounds__(kFmtThreads, F64 ? 3 : 4) k_pcd_write(const void* __restrict__ pts, int64_t n, const int64_t* __restrict__ tile_off,
                                                                        uint8_t* __restrict__ out, uint32_t* __restrict__ status) {
    extern __shared__ __align__(16) uint8_t s_img[];
    __shared__ uint32_t s_warp[kFmtThreads / 32], s_edge[kFmtThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int64_t dst0 = __ldg(tile_off + 2 * (int64_t)blockIdx.x);
    const int64_t row0 = (int64_t)blockIdx.x * kFmtTile + 2 * tid;
    const int64_t rest = n - (int64_t)blockIdx.x * kFmtTile;
    const int m = (int)(rest < kFmtTile ? rest : kFmtTile);
    const bool v0 = 2 * tid < m, v1 = 2 * tid + 1 < m;
    typename RowT<F64>::T v[8];
    rows_load<F64>(pts, row0, v0, v1, v);
    Piece pc[8];
    uint32_t fl = 0;
    bool special;
    const uint32_t len = rows_pieces<F64>(v0, v1, v, pc, special, fl);
    uint32_t inc = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    uint32_t prev_t1 = __shfl_up_sync(0xffffffffu, pc[7].T1, 1);         // the last four bytes of the previous thread's text
    if (lane == 31) { s_warp[w] = inc; s_edge[w] = pc[7].T1; }
    __syncthreads();
    uint32_t base = 0, total = 0;
#pragma unroll
    for (int k = 0; k < kFmtThreads / 32; ++k) { const uint32_t t = s_warp[k]; if (k < w) base += t; total += t; }
    if (lane == 0) prev_t1 = w ? s_edge[w - 1] : 0u;
    const int phase = (int)(dst0 & 15);
    rows_stream<F64>(smem_u32(s_img), (uint32_t)phase + base + inc - len, prev_t1, v0, v1, 2 * tid + 2 >= m, special, pc, pts, row0);
    cta_image_out(out + (dst0 - phase), s_img, phase, phase + (int)total, tid, kFmtThreads);     // TMA bulk store of the aligned body
    if (fl != 0 && status != nullptr) atomicOr(status, fl);
}

// Byte offset of the text of arbitrary rows (frame boundaries): one warp per query sums the line lengths of
// the rows of its tile that precede the row.  With these offsets ONE formatting pass over the frame-major
// buffer yields every per-frame file body of save_results (LMC:870-884) as a slice of the same text.
template <bool F64>
__global__ void __launch_bounds__(256) k_pcd_row_off(const void* __restrict__ pts, int64_t n, const int64_t* __restrict__ tile_off,
                                                     const int64_t* __restrict__ rows, int32_t n_rows, int64_t* __restrict__ byte_off) {
    const int lane = threadIdx.x & 31;
    const int64_t qi = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qi >= n_rows) return;
    int64_t r = rows[qi];
    r = r < 0 ? 0 : (r > n ? n : r);
    const int64_t tile = r / kPcdTile, first = tile * kPcdTile;
    uint32_t sum = 0, fl = 0;
    for (int64_t i = first + lane; i < r; i += 32) {
        typename RowT<F64>::T v[4];
        load_row_native<F64>(pts, i, v);
        sum += 4;
#pragma unroll
        for (int c = 0; c < 4; ++c) sum += fmt_len(v[c], fl);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) byte_off[qi] = tile_off[tile] + sum;
}

// ---- generic delimited text rows: CS:1643-1716 (_export_pcd '%.6f %.6f %.6f %.0f %.0f', _export_xyz, _export_csv) ----
// "%.{d}f" with d = 0..9 per column and the full integer range a timestamp column needs (ns since the epoch ~ 1.7e18):
// every number through the core's fmtg_prepare, except the compiled formats' fast '%.6f' numbers (piece_fast).
constexpr int kTextCols   = 6;                      // LMC_TEXT_MAX_COLS

struct TextFmt { int32_t n_cols, row_stride; int32_t col[kTextCols]; int32_t dec[kTextCols]; uint8_t sep; };

// text length of "%.{d}f" % v: no digits, one table compare
__device__ __noinline__ uint2 text_len_slow_eval(double v, int d) { uint32_t fl = 0; const uint32_t len = fmtg_prepare(v, d, fl).len; return make_uint2(len, fl); }
__device__ __forceinline__ uint32_t text_len(double v, int d, uint32_t& fl) {
    const double a = fabs(v);
    if (!(a < 18446744073709551616.0)) { const uint2 r = text_len_slow_eval(v, d); fl |= r.y; return r.x; }     // nan, inf, >= 2^64
    return ((uint32_t)__double2hiint(v) >> 31) + text_nd(a, d) + (d ? 1u + (uint32_t)d : 0u);
}

// The format is a launch parameter (TextFmt), but every runtime test on it sits inside the per-number code: the three formats the
// second simulator writes -- pcd '%.6f %.6f %.6f %.0f %.0f', xyz '%.6f' x 3, csv '%.6f' x 5, identity column pick (CS:1664 / 1703 /
// 1711) -- are compiled with the column count and the decimals as template constants (NC > 0, DP = 4 bits per column); anything
// else runs the same code with NC = 0 and reads them from F.
template <int NC, uint32_t DP> struct TextSpec {
    static __device__ __forceinline__ int ncols(const TextFmt& F) { return NC ? NC : F.n_cols; }
    static __device__ __forceinline__ int dec(const TextFmt& F, int c) { return NC ? (int)((DP >> (4 * c)) & 15u) : F.dec[c]; }
    static __device__ __forceinline__ int64_t cell(const TextFmt& F, int64_t i, int c) { return NC ? i * F.row_stride + c : i * F.row_stride + F.col[c]; }
};

// size pass: the rows' text lengths summed per 256-row tile (warp redux, no scan)
template <bool F64, int NC, uint32_t DP>
__global__ void __launch_bounds__(kPcdTile) k_text_len(const void* __restrict__ rows, int64_t n, const __grid_constant__ TextFmt F, int64_t* __restrict__ tile_off) {
    using S = TextSpec<NC, DP>;
    __shared__ uint32_t s_warp[kPcdTile / 32];
    const int64_t i = (int64_t)blockIdx.x * kPcdTile + threadIdx.x;
    uint32_t len = 0, fl = 0;
    if (i < n) {
        len = (uint32_t)S::ncols(F);                                 // separators + newline
#pragma unroll
        for (int c = 0; c < kTextCols; ++c) if (c < S::ncols(F)) len += text_len(load_cell<F64>(rows, S::cell(F, i, c)), S::dec(F, c), fl);
    }
    const uint32_t sum = __reduce_add_sync(0xffffffffu, len);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
#pragma unroll
        for (int k = 0; k < kPcdTile / 32; ++k) total += s_warp[k];
        tile_off[blockIdx.x + 1] = total;
    }
}

// write pass: one row per thread, 256 rows per tile; exact (ip, fq) per number by fmtg_prepare, digits by SWAR groups, word stream
template <bool F64, int NC, uint32_t DP>
__global__ void __launch_bounds__(kPcdTile) k_text_write(const void* __restrict__ rows, int64_t n, const __grid_constant__ TextFmt F,
                                                         const int64_t* __restrict__ tile_off, uint8_t* __restrict__ out, uint32_t* __restrict__ status) {
    using S = TextSpec<NC, DP>;
    extern __shared__ __align__(16) uint8_t s_dyn[];                 // the tile's text image, sized by the host from the format
    __shared__ uint32_t s_warp[kPcdTile / 32];
    uint8_t* s_img = s_dyn;
    const int tid = threadIdx.x;
    const int64_t i = (int64_t)blockIdx.x * kPcdTile + tid;
    const int64_t dst0 = tile_off[blockIdx.x];
    const int phase = (int)(dst0 & 15);
    // zero the part of the image this tile can reach (row edges are OR-ed in)
    const int img_words = (int)((phase + (tile_off[blockIdx.x + 1] - dst0) + 3 + 15) / 16) * 4;
    for (int k = tid * 4; k < img_words; k += kPcdTile * 4) *reinterpret_cast<uint4*>(s_img + 4 * k) = make_uint4(0, 0, 0, 0);
    Num t[kTextCols];
    [[maybe_unused]] Piece pc[kTextCols];
    [[maybe_unused]] bool slow6 = false;                             // compiled formats: some '%.6f' column of the row is not a fast number
    uint32_t len = 0, fl = 0;
    if (i < n) {
        len = (uint32_t)S::ncols(F);
        if constexpr (NC > 0) {
            // compiled formats: '%.6f' columns take the PCD writer's three-register pieces (|v| < 10^4 after rounding: every coordinate a
            // LiDAR produces; 63 instead of ~150 instructions per number), the other columns the generic exact split
            double v[NC];
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                v[c] = load_cell<F64>(rows, S::cell(F, i, c));
                if (S::dec(F, c) == 6) slow6 |= piece_fast(pc[c], v[c], c == NC - 1 ? 0x0au : (uint32_t)F.sep);
                else { t[c] = fmtg_prepare(v[c], S::dec(F, c), fl); len += t[c].len; }
            }
            if (slow6) {
#pragma unroll
                for (int c = 0; c < NC; ++c) if (S::dec(F, c) == 6) { t[c] = fmtg_prepare(v[c], 6, fl); len += t[c].len; }
            } else {
#pragma unroll
                for (int c = 0; c < NC; ++c) if (S::dec(F, c) == 6) len += piece_ll(pc[c]) + 7u;      // lead + ".dddddd" (separators counted above)
            }
        } else {
#pragma unroll
            for (int c = 0; c < kTextCols; ++c) if (c < S::ncols(F)) {
                t[c] = fmtg_prepare(load_cell<F64>(rows, S::cell(F, i, c)), S::dec(F, c), fl);
                len += t[c].len;
            }
        }
    }
    uint32_t total;
    const uint32_t off = block_scan_excl(len, s_warp, total);       // (its barrier also orders the zero fill before the ORs)
    if (i < n) {
        TextStream ts;
        ts.start(smem_u32(s_img), (uint32_t)phase + off);
        const uint32_t sep = (uint32_t)F.sep;
        if constexpr (NC > 0) {
            // (compiled formats start with a '%.6f' column, >= 9 bytes: the word shared with the previous row completes inside it)
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                constexpr int kFirst = 1, kRest = 0;
                if (S::dec(F, c) == 6 && !slow6) {
                    const uint32_t ll = piece_ll(pc[c]);
                    if (c == 0) {
                        if (ll > 4u) { ts.put<kFirst>(0x2du, 1u); ts.put<kFirst>(pc[c].L0, 4u); } else ts.put<kFirst>(pc[c].L0, ll);
                        ts.put4<kFirst>((pc[c].T0 & 0xffffff00u) | 0x2eu); ts.put4<kFirst>(pc[c].T1);
                    } else {
                        if (ll > 4u) { ts.put<kRest>(0x2du, 1u); ts.put<kRest>(pc[c].L0, 4u); } else ts.put<kRest>(pc[c].L0, ll);
                        ts.put4<kRest>((pc[c].T0 & 0xffffff00u) | 0x2eu); ts.put4<kRest>(pc[c].T1);
                    }
                } else if (c == 0) emit_number<kFirst>(ts, t[c], S::dec(F, c), c == NC - 1 ? 0x0au : sep);
                else emit_number<kRest>(ts, t[c], S::dec(F, c), c == NC - 1 ? 0x0au : sep);
            }
        } else {
            if (S::ncols(F) > 0) emit_number<2>(ts, t[0], S::dec(F, 0), S::ncols(F) == 1 ? 0x0au : sep);
#pragma unroll
            for (int c = 1; c < kTextCols; ++c) if (c < S::ncols(F)) emit_number<2>(ts, t[c], S::dec(F, c), c == S::ncols(F) - 1 ? 0x0au : sep);
        }
        ts.finish();
    }
    cta_image_out(out + (dst0 - phase), s_img, phase, phase + (int)total, tid, kPcdTile);
    if (fl != 0 && status != nullptr) atomicOr(status, fl);
}

// the compiled formats (TextSpec): decimals 4 bits per column, identity column pick
constexpr uint32_t kDpPcd = 0x00666u, kDpXyz = 0x666u, kDpCsv = 0x66666u;
static int text_spec_of(int32_t n_cols, const int32_t* col, const int32_t* dec) {      // 0 generic, 1 pcd, 2 xyz, 3 csv
    uint32_t dp = 0;
    for (int c = 0; c < n_cols; ++c) { if (col[c] != c) return 0; dp |= (uint32_t)dec[c] << (4 * c); }
    if (n_cols == 5 && dp == kDpPcd) return 1;
    if (n_cols == 3 && dp == kDpXyz) return 2;
    if (n_cols == 5 && dp == kDpCsv) return 3;
    return 0;
}

static TextFmt make_fmt(int32_t n_cols, int32_t row_stride, const int32_t* col, const int32_t* dec, uint8_t sep, int& img_bytes) {
    TextFmt F{};
    F.n_cols = n_cols; F.row_stride = row_stride; F.sep = sep;
    int row = n_cols;
    for (int c = 0; c < n_cols; ++c) { F.col[c] = col[c]; F.dec[c] = dec[c]; row += 1 + 20 + (dec[c] ? 1 + dec[c] : 0); }
    img_bytes = ((kPcdTile * row + 32 + 15) / 16) * 16;
    return F;
}

cudaError_t launch_text_size(bool f64, const void* rows, int64_t n, int32_t n_cols, int32_t row_stride, const int32_t* col, const int32_t* dec,
                             uint8_t sep, int64_t* tile_off, cudaStream_t st) {
    const int64_t tiles = (n + kPcdTile - 1) / kPcdTile;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    int img;
    const TextFmt F = make_fmt(n_cols, row_stride, col, dec, sep, img);
    if (tiles > 0) {
        const unsigned g = (unsigned)tiles;
#define LMC_TEXT_LEN(NC, DP) do { if (f64) k_text_len<true, NC, DP><<<g, kPcdTile, 0, st>>>(rows, n, F, tile_off); \
                                  else     k_text_len<false, NC, DP><<<g, kPcdTile, 0, st>>>(rows, n, F, tile_off); } while (0)
        switch (text_spec_of(n_cols, col, dec)) {
        case 1:  LMC_TEXT_LEN(5, kDpPcd); break;
        case 2:  LMC_TEXT_LEN(3, kDpXyz); break;
        case 3:  LMC_TEXT_LEN(5, kDpCsv); break;
        default: LMC_TEXT_LEN(0, 0u); break;
        }
#undef LMC_TEXT_LEN
    }
    return launch_tile_scan(tile_off, tiles, st);
}

template <bool F64, int NC, uint32_t DP>
static cudaError_t launch_text_write_as(const void* rows, int64_t n, const TextFmt& F, int img, const int64_t* tile_off, uint8_t* out,
                                        uint32_t* status, unsigned tiles, cudaStream_t st) {
    if (img > 48 * 1024) {                                           // widest formats only (6 columns x 9 decimals = 49 KB)
        cudaError_t e = cudaFuncSetAttribute(k_text_write<F64, NC, DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, img);
        if (e != cudaSuccess) return e;
    }
    k_text_write<F64, NC, DP><<<tiles, kPcdTile, img, st>>>(rows, n, F, tile_off, out, status);
    return cudaGetLastError();
}
cudaError_t launch_text_write(bool f64, const void* rows, int64_t n, int32_t n_cols, int32_t row_stride, const int32_t* col, const int32_t* dec,
                              uint8_t sep, const int64_t* tile_off, uint8_t* out, uint32_t* status, cudaStream_t st) {
    const int64_t tiles = (n + kPcdTile - 1) / kPcdTile;
    if (tiles == 0) return cudaSuccess;
    int img;
    const TextFmt F = make_fmt(n_cols, row_stride, col, dec, sep, img);
    const unsigned g = (unsigned)tiles;
#define LMC_TEXT_WRITE(NC, DP) (f64 ? launch_text_write_as<true, NC, DP>(rows, n, F, img, tile_off, out, status, g, st) \
                                    : launch_text_write_as<false, NC, DP>(rows, n, F, img, tile_off, out, status, g, st))
    switch (text_spec_of(n_cols, col, dec)) {
    case 1:  return LMC_TEXT_WRITE(5, kDpPcd);
    case 2:  return LMC_TEXT_WRITE(3, kDpXyz);
    case 3:  return LMC_TEXT_WRITE(5, kDpCsv);
    default: return LMC_TEXT_WRITE(0, 0u);
    }
#undef LMC_TEXT_WRITE
}

cudaError_t launch_pcd_size(bool f64, const void* pts, int64_t n, int64_t* tile_off, cudaStream_t st) {
    const int64_t per = (int64_t)kLenTiles * kFmtTile;
    const int64_t tiles = (n + kPcdTile - 1) / kPcdTile, ctas = (n + per - 1) / per;
    if (tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    if (ctas > 0) {
        if (f64) k_pcd_len<true><<<(unsigned)ctas, kFmtThreads, 0, st>>>(pts, n, tile_off);
        else     k_pcd_len<false><<<(unsigned)ctas, kFmtThreads, 0, st>>>(pts, n, tile_off);
    }
    return launch_tile_scan(tile_off, tiles, st);
}

cudaError_t launch_pcd_row_off(bool f64, const void* pts, int64_t n, const int64_t* tile_off, const int64_t* rows, int32_t n_rows,
                               int64_t* byte_off, cudaStream_t st) {
    if (n_rows <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((n_rows + 7) / 8);
    if (f64) k_pcd_row_off<true><<<grid, 256, 0, st>>>(pts, n, tile_off, rows, n_rows, byte_off);
    else     k_pcd_row_off<false><<<grid, 256, 0, st>>>(pts, n, tile_off, rows, n_rows, byte_off);
    return cudaGetLastError();
}

cudaError_t launch_pcd_write(bool f64, const void* pts, int64_t n, const int64_t* tile_off, uint8_t* out, uint32_t* status, cudaStream_t st) {
    const int64_t ctas = (n + kFmtTile - 1) / kFmtTile;
    if (ctas == 0) return cudaSuccess;
    if (ctas > 0x7fffffffLL) return cudaErrorInvalidValue;
    static thread_local int attr_dev = -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (attr_dev != dev) {
        if ((e = cudaFuncSetAttribute(k_pcd_write<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFmtImg)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(k_pcd_write<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFmtImg)) != cudaSuccess) return e;
        attr_dev = dev;
    }
    if (f64) k_pcd_write<true><<<(unsigned)ctas, kFmtThreads, kFmtImg, st>>>(pts, n, tile_off, out, status);
    else     k_pcd_write<false><<<(unsigned)ctas, kFmtThreads, kFmtImg, st>>>(pts, n, tile_off, out, status);
    return cudaGetLastError();
}

}  // namespace lmc
