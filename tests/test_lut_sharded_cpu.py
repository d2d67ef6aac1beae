"""CPU check of the min-reduction of `lut.nearest_sharded` over gloo (world size 2): a rank whose search found no
finite-cost entry for an observation (all-NaN shard, padding shard) must not win the reduction.  The CUDA search is
replaced by a NumPy stand-in that reports such an observation with the kernels' all-ones "no entry" word."""
import os
import socket
import sys

import numpy as np
import torch

from conftest import ROOT

NB, M = 4, 9
NO_ENTRY = 2 ** 32 - 1


def _tables():
    rng = np.random.default_rng(21)
    shards = [rng.random((13, NB)).astype(np.float32), rng.random((20, NB)).astype(np.float32)]
    shards[0][:] = np.nan                      # rank 0: every entry NaN (e.g. rows of an invalid soil index)
    obs = rng.random((M, NB)).astype(np.float32)
    obs[4] = np.nan                            # an observation no entry can match
    return shards, obs


def _search(l, o, w, off):
    """NumPy stand-in of spart_lut_nearest with packed output: FP32 costs, ties to the lowest index, entries whose
    cost is NaN or not below 3e38 never chosen, all-ones word (-1 as int64) where nothing was found."""
    with np.errstate(invalid="ignore"):
        d = ((o.numpy()[:, None, :] - l.numpy()[None, :, :]) ** 2).sum(-1).astype(np.float32)
        ok = d < np.float32(3e38)
    words = np.full(d.shape[0], -1, dtype=np.int64)
    for i in range(d.shape[0]):
        if ok[i].any():
            j = int(np.argmin(np.where(ok[i], d[i], np.inf)))
            words[i] = (int(d[i, j].view(np.uint32)) << 32) | (j + off)
    return torch.from_numpy(words)


def _unpack(words):
    w = words.numpy()
    return torch.from_numpy(w & 0xffffffff), torch.from_numpy((w >> 32).astype(np.uint32).view(np.float32))


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    from spart_b200 import lut
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        shards, obs = _tables()
        idx, cost = lut.nearest_sharded(torch.from_numpy(shards[rank]), torch.from_numpy(obs), search=_search,
                                        unpack_words=_unpack)
        # a rank whose shard is empty contributes the identity; the all-NaN rank must behave the same
        idx2, cost2 = lut.nearest_sharded(torch.from_numpy(shards[rank][:0] if rank == 0 else shards[rank]),
                                          torch.from_numpy(obs), index_offset=0 if rank == 0 else 13,
                                          search=_search, unpack_words=_unpack)
        q.put((rank, idx.numpy(), cost.numpy(), idx2.numpy(), cost2.numpy()))
    finally:
        dist.destroy_process_group()


def test_no_entry_shard_loses_the_min_reduction_gloo_world2():
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        rank, *r = q.get(timeout=120)
        res[rank] = r
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    shards, obs = _tables()
    d = ((obs[:, None, :] - shards[1][None, :, :]) ** 2).sum(-1).astype(np.float32)
    want_idx = d.argmin(1) + 13                 # global index: rank 1's slice starts after rank 0's 13 entries
    want_cost = d.min(1)
    live = ~np.isnan(obs).any(1)
    for r in range(world):
        idx, cost, idx2, cost2 = res[r]
        assert np.array_equal(idx[live], want_idx[live]) and np.array_equal(cost[live], want_cost[live])
        # the observation nothing matches gets the documented "no entry" result on every rank
        assert (idx[~live] == NO_ENTRY).all() and np.isnan(cost[~live]).all()
        assert np.array_equal(idx, idx2) and np.array_equal(cost, cost2, equal_nan=True)


def test_search_stand_in_matches_the_kernel_convention():
    """The stand-in's "nothing found" word is the all-ones word the kernels leave (unpacked: index 2^32 - 1, NaN)."""
    l = torch.from_numpy(np.full((3, NB), np.nan, dtype=np.float32))
    o = torch.from_numpy(np.zeros((2, NB), dtype=np.float32))
    w = _search(l, o, None, 0)
    assert (w == -1).all()
    idx, cost = _unpack(w)
    assert (idx == NO_ENTRY).all() and torch.isnan(cost).all()
