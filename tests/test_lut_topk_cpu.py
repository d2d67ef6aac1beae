"""CPU check of the reductions of `lut.nearest_k_sharded` and `lut.estimate(group=...)` over gloo (world size 2).
The CUDA search, merge and moments are replaced by NumPy stand-ins with the kernels' conventions (packed words
cost bits << 32 | global index, the all-ones "no entry" word sorting last), so what is checked is the
gather / all-reduce logic: global indices across ranks, an empty rank, an all-NaN rank and one result on every rank."""
import os
import socket
import sys

import numpy as np
import torch

from conftest import ROOT

NB, M, K, P = 3, 7, 5, 4
NO_ENTRY = 2 ** 32 - 1


def _tables():
    rng = np.random.default_rng(5)
    table = rng.random((30, NB)).astype(np.float32)
    table[17:23] = np.nan                           # an invalid block, split over both ranks in the uneven split
    params = rng.random((30, P))
    params[:, 2] = 7.25                             # a constant parameter: std must be 0
    obs = rng.random((M, NB)).astype(np.float32)
    obs[3] = np.nan                                 # an observation no entry can match
    return table, params, obs


def _costs(l, o):
    with np.errstate(invalid="ignore"):
        return ((o[:, None, :] - l[None, :, :]) ** 2).sum(-1).astype(np.float32)


def _words(d, off, k):
    """The k smallest words per row of the cost matrix d (local index + off), "no entry" (-1) beyond the valid ones."""
    out = np.full((d.shape[0], k), -1, dtype=np.int64)
    for i in range(d.shape[0]):
        ok = np.flatnonzero(d[i] < np.float32(3e38))
        w = np.sort((d[i, ok].view(np.uint32).astype(np.uint64) << np.uint64(32)) | (ok + off).astype(np.uint64))[:k]
        out[i, :len(w)] = w.view(np.int64)
    return out


def _search(l, o, k, w, off):
    return torch.from_numpy(_words(_costs(l.numpy(), o.numpy()), off, k))


def _merge(lists):
    a = lists.numpy().view(np.uint64)
    L, m, k = a.shape
    w = np.sort(a.transpose(1, 0, 2).reshape(m, L * k), axis=1)[:, :k].view(np.int64)
    return torch.from_numpy(w & 0xffffffff), torch.from_numpy((w >> 32).astype(np.uint32).view(np.float32))


def _accumulate(params, index, off, centre, acc):
    x, idx = params.numpy(), index.numpy()
    for o in range(idx.shape[0]):
        for j in idx[o]:
            e = j - off
            if 0 <= e < x.shape[1]:
                acc[o, :-1] += torch.from_numpy(x[:, e] if centre is None else (x[:, e] - centre[o].numpy()) ** 2)
                acc[o, -1] += 1


def _finish(acc, sq):
    with np.errstate(invalid="ignore", divide="ignore"):
        a = acc.numpy()
        mean = a[:, :-1] / a[:, -1:]
        std = None if sq is None else np.sqrt(sq.numpy()[:, :-1] / a[:, -1:])
    return torch.from_numpy(mean), None if std is None else torch.from_numpy(std), torch.from_numpy(
        a[:, -1].astype(np.int64))


# rank pieces of the 30-entry table: (rank 0, rank 1)
SPLITS = {"uneven": (12, 30), "empty_rank0": (0, 30), "all_nan_rank1": (17, 23)}


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    from spart_b200 import lut
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        table, params, obs = _tables()
        out = {}
        for name, (cut, end) in SPLITS.items():
            lo, hi = (0, cut) if rank == 0 else (cut, end)
            idx, cost = lut.nearest_k_sharded(torch.from_numpy(table[lo:hi]), torch.from_numpy(obs), K,
                                              search=_search, merge=_merge)
            # the parameter table is split like the LUT; layout [P, n] as a view of the [n, P] table
            mean, std, count = lut.estimate(torch.from_numpy(params[lo:hi]).T, idx, group=dist.group.WORLD,
                                            accumulate=_accumulate, finish=_finish)
            out[name] = [t.numpy() for t in (idx, cost, mean, std, count)]
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


def _run(world=2):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        rank, r = q.get(timeout=120)
        res[rank] = r
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    return res


def test_sharded_topk_and_estimate_gloo_world2():
    res = _run()
    table, params, obs = _tables()
    for name, (cut, end) in SPLITS.items():
        keep = np.r_[0:end]                                 # the entries some rank holds
        want = _words(_costs(table[keep], obs), 0, K)
        want_idx, want_cost = (t.numpy() for t in _merge(torch.from_numpy(want[None])))
        live = ~np.isnan(obs).any(1)
        for r in (0, 1):
            idx, cost, mean, std, count = res[r][name]
            assert np.array_equal(idx, want_idx), (name, r)
            assert np.array_equal(cost, want_cost, equal_nan=True), (name, r)
            assert (idx[~live] == NO_ENTRY).all() and np.isnan(cost[~live]).all()
            # global indices: the rows of rank 1 are offset by rank 0's slice
            valid = idx != NO_ENTRY
            assert np.array_equal(cost[valid], _costs(table, obs)[np.nonzero(valid)[0], idx[valid]])
            for o in range(M):
                sel = params[idx[o][valid[o]]]
                assert count[o] == len(sel)
                if len(sel):
                    np.testing.assert_allclose(mean[o], sel.mean(0), rtol=1e-14, atol=0)
                    np.testing.assert_allclose(std[o], sel.std(0), rtol=1e-12, atol=1e-15)
                    assert std[o, 2] == 0.0
                else:
                    assert np.isnan(mean[o]).all() and np.isnan(std[o]).all()
            for a, b in zip(res[r][name], res[0][name]):         # the same result on every rank
                assert np.array_equal(a, b, equal_nan=True)
    # with rank 1 all NaN, every observation with a finite cost still gets K entries, all from rank 0
    assert (res[0]["all_nan_rank1"][0][~np.isnan(obs).any(1)] != NO_ENTRY).all()


def test_stand_ins_match_the_kernel_conventions():
    """A search with fewer than k valid entries fills with the all-ones word, which unpacks to (NO_ENTRY, NaN)."""
    l = torch.from_numpy(np.vstack([np.zeros((2, NB)), np.full((3, NB), np.nan)]).astype(np.float32))
    o = torch.from_numpy(np.zeros((2, NB), dtype=np.float32))
    w = _search(l, o, 4, None, 10)
    assert (w[:, 2:] == -1).all()
    idx, cost = _merge(w[None])
    assert (idx[:, :2] == torch.tensor([10, 11])).all() and (cost[:, :2] == 0).all()
    assert (idx[:, 2:] == NO_ENTRY).all() and torch.isnan(cost[:, 2:]).all()


def test_sharded_refuses_k_before_any_collective():
    """A bad k is refused on every rank before the first collective, also on a rank with an empty slice (which
    launches no search): no rank can be left waiting for others that refused.  Here no process group exists, so
    reaching a collective would fail with another error."""
    import pytest
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    from spart_b200 import lut
    obs = torch.zeros((2, NB))
    for k in (0, 129):
        for table in (torch.zeros((0, NB)), torch.zeros((4, NB))):
            with pytest.raises(ValueError, match="1 <= k <= 128"):
                lut.nearest_k_sharded(table, obs, k, search=_search, merge=_merge)
