"""Which point kernel serves an aligned-cloud call: csrc/lmc_plan.h (plan_point_launch) compiled with g++ and driven over
the cross product of layout, mode, path, size, alignment, exports, peers / multicast and the Mode B / C inputs, against
the routing rules written out below.  A call routed to the generic streaming kernel instead of its lean one still
computes the same bytes, only slower, so no parity test would notice."""
import itertools
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "livox_motion_compensation_sim_b200", "csrc")

RIGID, GYRO, SLERP, QUANT = 0, 1, 2, 3
OUT, LVX, LAS, GEN, LVX2, MC, PB = 1, 2, 4, 8, 16, 32, 64
OK, ERR_INVALID = 0, -1
LVX_TYPE2_OF_INPUT, LVX2_OF_OUTPUT = 0, 1
SMS = 148

# one case per line: f64 mode path sm_count p_begin p_end | ts tag out lvx14 las_x las_int | lvx_mode n_peers mc hold_idx
# frame_start n_samp.  A pointer column is 0 (NULL), 1 (16-byte aligned) or 2 (8-byte aligned only); the plan never
# dereferences them.  Output per case: rc stream ex grid tile0 n_tiles.
DRIVER = r'''
#include <cstdio>
#include <cstring>
#include "lmc_plan.h"
static void* ptr(long v) { return v == 0 ? nullptr : reinterpret_cast<void*>(v == 1 ? 0x10000 : 0x10008); }
int main() {
    long f64, mode, path, sms, pb, pe, ts, tag, out, lvx, lx, li, lm, np, mc, hold, fs, ns;
    while (std::scanf("%ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld %ld",
                      &f64, &mode, &path, &sms, &pb, &pe, &ts, &tag, &out, &lvx, &lx, &li, &lm, &np, &mc, &hold, &fs, &ns) == 18) {
        lmc::Params P;
        std::memset(&P, 0, sizeof P);
        P.p_begin = pb; P.p_end = pe; P.n_points = pe;
        P.ts = ptr(ts); P.tag = static_cast<const uint8_t*>(ptr(tag)); P.out = ptr(out);
        P.lvx14 = static_cast<uint8_t*>(ptr(lvx)); P.las_x = static_cast<int32_t*>(ptr(lx)); P.las_int = static_cast<uint16_t*>(ptr(li));
        P.las_y = P.las_z = P.las_x;
        P.lvx_mode = (int32_t)lm; P.n_peers = (int32_t)np;
        for (long r = 0; r < np; ++r) { P.peer_out[r] = ptr(1); P.peer_lvx[r] = static_cast<uint8_t*>(ptr(1)); }
        P.mc_out = ptr(mc); P.mc_lvx = static_cast<uint8_t*>(ptr(mc));
        P.hold_idx = static_cast<const int32_t*>(ptr(hold)); P.frame_start = static_cast<const int64_t*>(ptr(fs)); P.n_samp = ns;
        const lmc::Plan pl = lmc::plan_point_launch(f64 != 0, (int)mode, P, (int)path, (int)sms);
        std::printf("%d %d %d %d %lld %lld\n", pl.rc, pl.stream ? 1 : 0, pl.ex, pl.grid, (long long)pl.tile0, (long long)pl.n_tiles);
    }
    return 0;
}
'''


def tile_points(f64, mode):
    return 960 if f64 else (2880 if mode == SLERP else 1920)


def expected(c):
    """The routing rules (rc, streaming?, export variant)."""
    f64, mode, path = c["f64"], c["mode"], c["path"]
    peers, mc = c["n_peers"] > 0, c["mc"] != 0
    tp = tile_points(f64, mode)
    n_tiles = -(-(c["p_end"] - c["p_begin"] // tp * tp) // tp)
    # family
    if c["ts"] == 2 or c["tag"] == 2:                       # TMA needs 16-byte aligned timestamp / tag arrays
        return (ERR_INVALID, 0, 0) if peers else (OK, 0, 0)
    if not peers and (path == 0 or (path == 1 and n_tiles < 2 * SMS)):
        return OK, 0, 0
    # variant
    if mode == QUANT:
        return OK, 1, GEN
    mask = (OUT if c["out"] else 0) | (LVX if c["lvx14"] else 0) | (LAS if c["las_x"] or c["las_int"] else 0)
    lvx2 = c["lvx14"] and c["lvx_mode"] == LVX2_OF_OUTPUT
    samples_ok = 2 <= c["n_samp"] < 2 ** 31 - 1
    merge_kernel = not f64 and mode in (RIGID, SLERP) and mask == OUT | LVX and not lvx2
    lean = ((not peers or mc or merge_kernel)
            and (not lvx2 or mode == GYRO)
            and (not mask & LAS or (c["las_x"] and c["las_int"])))
    if mode == SLERP:
        lean = lean and not c["hold_idx"] and c["ts"] and samples_ok and (f64 or c["frame_start"])
    if mode == GYRO:
        lean = lean and c["ts"] and c["frame_start"] and samples_ok
    if mc and not (lean and merge_kernel):
        return ERR_INVALID, 0, 0
    if not lean:
        return OK, 1, GEN
    if mc:
        return OK, 1, OUT | LVX | MC
    if peers:
        return OK, 1, OUT | LVX | PB
    lean_kernels = {OUT: OUT, OUT | LVX: OUT | LVX | LVX2 if lvx2 else OUT | LVX, OUT | LAS: OUT | LAS}
    return OK, 1, lean_kernels.get(mask, GEN)


EXPORTS = {                                              # out, lvx14, lvx_mode, las_x, las_int
    "out": (1, 0, 0, 0, 0),
    "out+lvx": (1, 1, LVX_TYPE2_OF_INPUT, 0, 0),
    "out+lvx2": (1, 1, LVX2_OF_OUTPUT, 0, 0),
    "out+las": (1, 0, 0, 1, 1),
    "out+las_xyz": (1, 0, 0, 1, 0),                      # LAS incomplete: no intensity
    "out+las_int": (1, 0, 0, 0, 1),                      # LAS incomplete: no x / y / z
    "out+lvx+las": (1, 1, LVX_TYPE2_OF_INPUT, 1, 1),
    "lvx": (0, 1, LVX_TYPE2_OF_INPUT, 0, 0),
    "lvx+las": (0, 1, LVX_TYPE2_OF_INPUT, 1, 1),
}
MERGE = {"local": (0, 0), "peer": (1, 0), "peer+mc": (1, 1)}    # n_peers, multicast
SAMPLES = {                                              # ts, frame_start, hold_idx, n_samp (Mode B / C inputs)
    "plain": (1, 1, 0, 720_001),
    "hold_idx": (1, 1, 1, 720_001),
    "no_ts": (0, 1, 1, 720_001),                         # (Mode C hold-next needs no timestamps)
    "no_frame_start": (1, 0, 0, 720_001),
    "n_samp_1": (1, 1, 0, 1),
    "n_samp_2": (1, 1, 0, 2),
    "n_samp_2^31-1": (1, 1, 0, 2 ** 31 - 1),
}


def cases():
    for f64, mode, path, below, align, ex, merge, samp in itertools.product(
            (True, False), (RIGID, GYRO, SLERP, QUANT), (0, 1, 2), (True, False), ("aligned", "ts", "tag"),
            EXPORTS, MERGE, SAMPLES):
        out, lvx14, lvx_mode, las_x, las_int = EXPORTS[ex]
        n_peers, mc = MERGE[merge]
        ts, fs, hold, n_samp = SAMPLES[samp]
        if mode in (RIGID, QUANT):
            if samp != "plain" or align == "ts":
                continue
            ts, fs, hold, n_samp = 0, 0, 0, 0           # what lmc_align_rigid_* / lmc_quantize_* pass
        if mode == QUANT:
            out = 0                                      # lmc_quantize_* has no aligned cloud
            if not (lvx14 or las_x or las_int):
                continue
        if mode == GYRO and samp == "hold_idx":
            continue
        if align == "ts":
            if not ts:
                continue
            ts = 2
        tp = tile_points(f64, mode)
        n_tiles = 2 * SMS - 1 if below else 2 * SMS      # just below / at the size threshold of path 1
        p_begin = tp + 7                                 # a shard starting inside its first tile
        c = dict(f64=f64, mode=mode, path=path, p_begin=p_begin, p_end=tp + (n_tiles - 1) * tp + 1,
                 ts=ts, tag=2 if align == "tag" else (1 if lvx14 and lvx_mode == LVX2_OF_OUTPUT else 0),
                 out=out, lvx14=lvx14, las_x=las_x, las_int=las_int, lvx_mode=lvx_mode, n_peers=n_peers, mc=mc,
                 hold_idx=hold, frame_start=fs, n_samp=n_samp)
        yield c, n_tiles


def row(c, sms=SMS):
    return " ".join(str(int(v)) for v in (c["f64"], c["mode"], c["path"], sms, c["p_begin"], c["p_end"], c["ts"], c["tag"],
                                          c["out"], c["lvx14"], c["las_x"], c["las_int"], c["lvx_mode"], c["n_peers"], c["mc"],
                                          c["hold_idx"], c["frame_start"], c["n_samp"]))


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    d = tmp_path_factory.mktemp("plan")
    src, exe = d / "plan_driver.cpp", d / "plan_driver"
    src.write_text(DRIVER)
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", CSRC, "-o", str(exe), str(src)], check=True)

    def run(rows):
        r = subprocess.run([str(exe)], input="\n".join(rows) + "\n", capture_output=True, text=True, check=True, timeout=120)
        return [tuple(int(x) for x in ln.split()) for ln in r.stdout.splitlines()]
    return run


def test_routing_table(plan):
    table = list(cases())
    got = plan([row(c) for c, _ in table])
    assert len(got) == len(table)
    seen = set()
    for (c, n_tiles), (rc, stream, ex, grid, tile0, n) in zip(table, got):
        want = expected(c)
        assert (rc, stream, ex if stream else 0) == want, (c, (rc, stream, ex))
        if stream:
            assert (tile0, n, grid) == (tile_points(c["f64"], c["mode"]), n_tiles, SMS), c
        seen.add(want)
    # every family / variant / refusal the rules name is reached by the table
    assert {s[2] for s in seen if s[1]} == {GEN, OUT, OUT | LVX, OUT | LAS, OUT | LVX | LVX2, OUT | LVX | MC, OUT | LVX | PB}
    assert (OK, 0, 0) in seen and (ERR_INVALID, 0, 0) in seen


def test_bench_headline_kernel(plan):
    """bench.py V5 (f32 Mode C, 3.6e8 points of a 1 h stream, aligned cloud + type-2 LVX) runs k_stream<false, kSlerp, Out|Lvx>
    on the automatic path, over one CTA per SM; a one-tile call takes the direct kernel."""
    v5 = dict(f64=False, mode=SLERP, path=1, p_begin=0, p_end=360_000_000, ts=1, tag=0, out=1, lvx14=1, las_x=0, las_int=0,
              lvx_mode=LVX_TYPE2_OF_INPUT, n_peers=0, mc=0, hold_idx=0, frame_start=1, n_samp=720_001)
    small = dict(v5, p_end=2880)
    (rc, stream, ex, grid, tile0, n), (rc2, stream2, *_) = plan([row(v5), row(small)])
    assert (rc, stream, ex, grid, tile0, n) == (OK, 1, OUT | LVX, SMS, 0, 125_000)
    assert (rc2, stream2) == (OK, 0)
    # the grid never exceeds the tiles: a forced streaming launch of 3 tiles on 148 SMs runs 3 CTAs
    assert plan([row(dict(small, path=2, p_end=3 * 2880))])[0][3] == 3
