"""torchrun worker (>= 2 GPUs): merged-cloud assembly fused into the kernel epilogue (peer stores over
NVLink, SymmetricMerged) == NCCL all-gather path == single-rank result, byte for byte.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_fused_merge.py
"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

from livox_motion_compensation_sim_b200 import ops, sharding, synth


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    F, P = int(os.environ.get("LMC_F", "4000")), 10_000
    rng = np.random.default_rng(3)
    counts = np.full(F, P); counts[rng.integers(0, F, 40)] = rng.integers(0, 3000, 40)      # ragged: unequal shards
    st = synth.make_stream(F, counts, 4242, device=dev, dtype=torch.float32)               # same stream on every rank
    N = st.n_points
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                        # noqa: E731
    off_d, fs_d, sts_d, seg_d = d(st.frame_off), d(st.frame_start), d(st.sample_ts), d(st.seg)
    fcuts, pcuts = sharding.shard_ranges(st.frame_off, world)
    b, e = int(pcuts[rank]), int(pcuts[rank + 1])

    # reference: the whole stream on this rank
    whole, wb = ops.deskew_slerp(st.pts, st.ts_off, off_d, fs_d, sts_d, seg_d, export=ops.ExportSpec(lvx=True))

    # (1) NCCL path: shard kernel into the merged buffer, then all-gather(v)
    m_out = torch.zeros_like(whole); m_lvx = torch.zeros_like(wb.lvx14)
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    ops.deskew_slerp(st.pts, st.ts_off, off_d, fs_d, sts_d, seg_d, out=m_out,
                     export=ops.ExportSpec(lvx=True, into=ops.ExportBuffers(lvx14=m_lvx)), p_range=(b, e))
    sharding.all_gather_merged([m_out, m_lvx], pcuts)
    torch.cuda.synchronize(); dist.barrier()
    t_nccl = time.perf_counter() - t0
    assert torch.equal(m_out, whole) and torch.equal(m_lvx, wb.lvx14), "NCCL merge differs from the single-rank result"

    # (2) fused path: the epilogue stores into every rank's symmetric copy
    sm = sharding.SymmetricMerged(N, dev, lvx=True)
    sm.out.zero_(); sm.lvx14.zero_()
    po, pl = sm.peer_ptrs()
    spec = lambda: ops.ExportSpec(lvx=True, into=ops.ExportBuffers(lvx14=sm.lvx14), peer_out=po, peer_lvx14=pl)  # noqa: E731
    sm.barrier()
    for it in range(2):                                                                     # second pass is the timed one
        torch.cuda.synchronize(); dist.barrier()
        t0 = time.perf_counter()
        ops.deskew_slerp(st.pts, st.ts_off, off_d, fs_d, sts_d, seg_d, out=sm.out, export=spec(), p_range=(b, e))
        sm.barrier()
        torch.cuda.synchronize(); dist.barrier()
        t_fused = time.perf_counter() - t0
    assert torch.equal(sm.out, whole), "fused merge: aligned cloud differs"
    assert torch.equal(sm.lvx14, wb.lvx14), "fused merge: LVX records differ"

    # (3) the same through the NVSwitch multicast mapping (multimem.st), where the box offers one
    mo, ml = sm.mc_ptrs()
    t_mc = None
    if mo:
        sm.out.zero_(); sm.lvx14.zero_()
        sm.barrier()
        spec_mc = lambda: ops.ExportSpec(lvx=True, into=ops.ExportBuffers(lvx14=sm.lvx14), peer_out=po, peer_lvx14=pl, mc_out=mo, mc_lvx14=ml)  # noqa: E731
        for it in range(2):
            torch.cuda.synchronize(); dist.barrier()
            t0 = time.perf_counter()
            ops.deskew_slerp(st.pts, st.ts_off, off_d, fs_d, sts_d, seg_d, out=sm.out, export=spec_mc(), p_range=(b, e))
            sm.barrier()
            torch.cuda.synchronize(); dist.barrier()
            t_mc = time.perf_counter() - t0
        assert torch.equal(sm.out, whole), "multicast merge: aligned cloud differs"
        assert torch.equal(sm.lvx14, wb.lvx14), "multicast merge: LVX records differ"
    # (4) replication-free file production: every rank builds ITS byte range of each output file from ITS frames and
    #     pwrite()s it at its offset; the file on disk equals the single-GPU image
    import tempfile
    from livox_motion_compensation_sim_b200.lvx import frame_layout
    from livox_motion_compensation_sim_b200.simulator import LiDARMotionSimulator
    fa, fb = int(fcuts[rank]), int(fcuts[rank + 1])
    ids = np.arange(F, dtype=np.int64)
    _, fpos = frame_layout(st.frame_off)
    lvx_whole, _ = ops.build_lvx_v11(st.pts, off_d, d(fpos), d(st.frame_t), d(ids), int(np.diff(st.frame_off).max()))
    las_whole, _ = ops.build_las_pf3(whole, scale=(0.001,) * 3, year=2026, day_of_year=7)
    txt_whole, _ = ops.pcd_ascii_body(whole)
    hdr = LiDARMotionSimulator._pcd_header(N)
    tmp = os.environ.get("LMC_OUT") or os.path.join(tempfile.gettempdir(), "lmc_sharded_files")
    if rank == 0:
        os.makedirs(tmp, exist_ok=True)
        for f in ("a.lvx", "a.las", "a.pcd"):
            if os.path.exists(os.path.join(tmp, f)):
                os.remove(os.path.join(tmp, f))
    dist.barrier()
    sh, pos0, stat = sharding.lvx_v11_shard(st.pts, st.frame_off, st.frame_t, ids, fa, fb)
    assert torch.equal(sh, lvx_whole[pos0:pos0 + sh.numel()]), "sharded LVX range differs"
    sharding.pwrite_range(os.path.join(tmp, "a.lvx"), pos0, sh.cpu().numpy())
    sh, pos0, stat = sharding.las_pf3_shard(whole, b, e, rank, scale=(0.001,) * 3, year=2026, day_of_year=7)
    assert torch.equal(sh, las_whole[pos0:pos0 + sh.numel()]), "sharded LAS range differs"
    sharding.pwrite_range(os.path.join(tmp, "a.las"), pos0, sh.cpu().numpy())
    sh, pos0, h0, stat = sharding.pcd_ascii_shard(whole[b:e], N, rank)
    assert torch.equal(sh, txt_whole[pos0 - len(hdr):pos0 - len(hdr) + sh.numel()]), "sharded PCD text differs"
    if rank == 0:
        assert h0 == hdr
        sharding.pwrite_range(os.path.join(tmp, "a.pcd"), 0, h0)
    sharding.pwrite_range(os.path.join(tmp, "a.pcd"), pos0, sh.cpu().numpy())
    dist.barrier()
    if rank == 0:
        assert open(os.path.join(tmp, "a.lvx"), "rb").read() == lvx_whole.cpu().numpy().tobytes()
        assert open(os.path.join(tmp, "a.las"), "rb").read() == las_whole.cpu().numpy().tobytes()
        assert open(os.path.join(tmp, "a.pcd"), "rb").read() == hdr + txt_whole.cpu().numpy().tobytes()
    if rank == 0:
        print(f"OK world={world} points={N} shard={e - b}  kernel+NCCL all-gather {t_nccl * 1e3:.2f} ms (first call)  "
              f"fused peer-store epilogue {t_fused * 1e3:.2f} ms  multicast epilogue " + (f"{t_mc * 1e3:.2f} ms" if t_mc else "unavailable"))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
