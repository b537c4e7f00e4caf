"""World-size-2 gloo tests (CPU) of the N > 1 path's host logic: contiguous keyframe blocks, per-pass flag union,
rank-ordered variable all-gather.  The arithmetic engine here is the oracle (no GPU in this container); what is under
test is the sharding/collective logic that lt_mapper_b200.removert.TorchDistComm implements for the real library."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    # the buffers below are host memory: hide any GPU (before CUDA initialises) so that TorchDistComm takes its host path
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import ctypes
        import oracle
        import synth
        from lt_mapper_b200 import removert
        K = 4
        full = synth.make_session(0, K, beams=12, az_steps=300)
        blk = K // world
        mine = synth.make_session(0, blk, beams=12, az_steps=300, k0=rank * blk)   # this rank's contiguous keyframe block
        assert np.array_equal(mine.xyzi, full.subset(rank * blk, (rank + 1) * blk).xyzi)
        comm = removert.TorchDistComm()
        assert (comm.rank, comm.world) == (rank, world)
        # (1) rank-ordered variable all-gather of the merged clouds == keyframe-order concatenation
        local = np.concatenate([oracle.transform(mine.scan(k), mine.poses[k]) for k in range(blk)])
        counts = (ctypes.c_int64 * world)()
        assert comm._allgather_i64(None, len(local), counts) == 0
        cnt = [int(c) for c in counts]
        displs = (ctypes.c_int64 * world)(*np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.int64))
        gathered = np.empty((sum(cnt), 4), np.float32)
        for comp in range(4):
            src = np.ascontiguousarray(local[:, comp]); dst = np.empty(sum(cnt), np.float32)
            assert comm._allgatherv(None, src.ctypes.data, len(src), dst.ctypes.data, counts, displs) == 0
            gathered[:, comp] = dst
        expect = np.concatenate([oracle.transform(full.scan(k), full.poses[k]) for k in range(K)])
        assert np.array_equal(gathered, expect)
        # (2) per-pass flag union: OR of per-rank flags over keyframe blocks == flags of the single-process pass
        m = oracle.voxel(expect, 0.05)
        inv = oracle.inverse_poses(full.poses)
        f_local = oracle.remove_pass(m, mine.xyzi, mine.offsets, inv[rank * blk:(rank + 1) * blk], oracle.MODE_HD, 2.5, threads=1)
        buf = f_local.copy()
        assert comm._allreduce(None, buf.ctypes.data, len(buf)) == 0
        f_full = oracle.remove_pass(m, full.xyzi, full.offsets, inv, oracle.MODE_HD, 2.5, threads=1)
        assert np.array_equal(buf, f_full)
        assert f_local.sum() < f_full.sum()   # the union really needed both ranks
        q.put((rank, "ok"))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, "FAIL " + repr(e) + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_sharding_and_collectives():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res


@pytest.mark.parametrize("world,split", [(1, False), (2, True), (2, False), (4, True), (8, True), (3, False), (8, False)])
def test_owned_blocks_partition_the_sessions_in_rank_order(world, split):
    """bench.owned_blocks: per session the blocks of the owning ranks are contiguous, disjoint, in rank order and cover [0, K) --
    rank-order concatenation must equal keyframe order (utility.cpp:177-189 concatenates in keyframe order)."""
    sys.path.insert(0, ROOT)
    import bench
    for K in (1000, 7, 2000):
        for s in (0, 1):
            nxt = 0
            owners = 0
            for r in range(world):
                k0, n = bench.owned_blocks(r, world, K, split)[s]
                if n == 0:
                    continue
                owners += 1
                assert k0 == nxt
                nxt = k0 + n
            assert nxt == K
            assert owners == (world // 2 if split else min(world, K))
        if split:   # a rank owns keyframes of exactly one session: ranks < world/2 the central one
            for r in range(world):
                b = bench.owned_blocks(r, world, K, split)
                assert (b[0][1] > 0) == (r < world // 2) and (b[1][1] > 0) == (r >= world // 2)
