"""The k nearest LUT entries (`lut.nearest_k`, spart_lut_topk), their merge over table pieces
(spart_lut_topk_merge, `lut.nearest_k_sharded`) and the parameter moments over the chosen entries (`lut.estimate`).

The search must equal `nearest` bit for bit at k = 1, equal an exact brute-force (cost, index) sort on tables whose
FP32 costs are exact (ties at the k-th place included), not depend on the launch plan, and mark unfilled slots with
the "no entry" result.  The moments are compared with NumPy float64 on the chosen parameter rows."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NO_ENTRY = 2 ** 32 - 1


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    from spart_b200 import lut
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    yield torch, spart_b200, lut
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def cycles(env):
    """torch.cuda._sleep cycles of a delay of at least 100 ms, measured with CUDA events."""
    torch, _, _ = env
    c = 1 << 20
    for _ in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.cuda._sleep(c)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= 120.0:
            return c
        c = int(c * min(max(150.0 / max(ms, 1e-3), 1.5), 64.0))
    pytest.fail(f"torch.cuda._sleep({c}) lasted {ms:.1f} ms, not 100 ms")


def bits(torch, t):
    """The integer view of a tensor (NaN-aware bit comparison)."""
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def same(torch, a, b):
    return all(torch.equal(bits(torch, x), bits(torch, y)) for x, y in zip(a, b))


def grid_table(rng, n, nb, levels=6):
    """Values on a 2^-8 grid in [0, levels / 256): every FP32 cost of <= 8 bands is exact, and costs tie often."""
    return (rng.integers(0, levels, size=(n, nb)) / 256.0).astype(np.float32)


def brute_k(L, O, k):
    """Exact reference: per observation a stable (cost, index) sort of the FP64 costs (exact here), the first k
    entries with a cost below 3e38 (NaN excluded), NO_ENTRY / NaN beyond."""
    with np.errstate(invalid="ignore"):
        d = ((O[:, None, :].astype(np.float64) - L[None, :, :]) ** 2).sum(-1)
    idx = np.full((O.shape[0], k), NO_ENTRY, dtype=np.int64)
    cost = np.full((O.shape[0], k), np.nan, dtype=np.float32)
    for i in range(O.shape[0]):
        ok = np.flatnonzero(d[i] < 3e38)
        order = ok[np.argsort(d[i, ok], kind="stable")][:k]
        idx[i, :len(order)] = order
        cost[i, :len(order)] = d[i, order]
    return idx, cost, d


def test_k1_is_nearest_bit_for_bit(env):
    """k = 1 returns `nearest`'s index and cost bit for bit, for every band-group instance, with and without weights."""
    torch, _, lut = env
    g = torch.Generator(device="cuda").manual_seed(3)
    shapes = ((6000, 777), (5000, 300), (333, 1000), (100, 5))
    for i, nb in enumerate((1, 4, 5, 9, 13, 17, 21, 26, 32)):
        n, m = shapes[i % len(shapes)]
        L = torch.rand((n, nb), generator=g, device="cuda")
        O = torch.rand((m, nb), generator=g, device="cuda")
        w = torch.rand(nb, generator=g, device="cuda") + 0.1
        for weights in (None, w):
            i1, c1 = lut.nearest(L, O, weights)
            ik, ck = lut.nearest_k(L, O, 1, weights)
            assert ik.shape == (m, 1) and ck.shape == (m, 1)
            assert torch.equal(ik[:, 0], i1) and torch.equal(bits(torch, ck[:, 0]), bits(torch, c1)), (nb, weights)


@pytest.mark.parametrize("k", [1, 7, 32, 128])
def test_exact_table_matches_a_stable_sort(env, k):
    """Grid tables with many duplicate rows spread over the slices: the whole [m, k] result equals the exact stable
    (cost, index) sort bit for bit, ties at the k-th place included, and a row is the same whether the observation is
    searched alone (m = 1: many slices) or among 10^5 (few slices)."""
    torch, _, lut = env
    rng = np.random.default_rng(100 + k)
    n, nb = 120_000, 7
    L = grid_table(rng, n, nb)
    src = rng.integers(0, n, size=3000)
    L[rng.permutation(n)[:3000]] = L[src]                  # duplicates at random places, i.e. in other slices
    O = grid_table(rng, 100_000, nb)
    O[:40] = L[rng.integers(0, n, size=40)]                # observations with exact matches (cost 0 ties)
    Ld, Od = torch.from_numpy(L).cuda(), torch.from_numpy(O).cuda()
    idx, cost = lut.nearest_k(Ld, Od, k)
    want_idx, want_cost, d = brute_k(L, O[:64], k)
    assert np.array_equal(idx[:64].cpu().numpy(), want_idx)
    assert np.array_equal(cost[:64].cpu().numpy().view(np.uint32), want_cost.view(np.uint32))
    # the k-th place is tied with an entry that was left out in some rows: the lowest index won there
    kth = np.sort(d, axis=1)[:, k - 1:k + 1]
    assert (kth[:, 0] == kth[:, 1]).sum() > 0
    for o in (0, 1, 39, 50, 63, 77_777, 99_999):
        i1, c1 = lut.nearest_k(Ld, Od[o:o + 1].clone(), k)
        assert torch.equal(i1[0], idx[o]) and torch.equal(bits(torch, c1[0]), bits(torch, cost[o])), o


@pytest.mark.parametrize("k", [10, 50])
def test_random_float_table(env, k):
    """Costs ascend, indices are distinct, each cost is its entry's FP64 cost to 1e-5, and no entry left out is
    cheaper than the k-th by more than that rounding."""
    torch, _, lut = env
    g = torch.Generator(device="cuda").manual_seed(k)
    n, m, nb = 50_000, 400, 13
    L = torch.rand((n, nb), generator=g, device="cuda")
    O = torch.rand((m, nb), generator=g, device="cuda")
    w = torch.rand(nb, generator=g, device="cuda") + 0.1
    idx, cost = lut.nearest_k(L, O, k, w)
    d = ((O[:, None, :].double() - L[None, :, :].double()) ** 2 * w.double()).sum(-1)
    assert torch.all(cost[:, 1:] >= cost[:, :-1])
    assert torch.all(idx.sort(1).values[:, 1:] != idx.sort(1).values[:, :-1])
    mine = d.gather(1, idx)
    assert torch.all((cost.double() - mine).abs() <= 1e-5 * mine + 1e-12)
    left_out = d.scatter(1, idx, float("inf")).min(1).values
    assert torch.all(left_out >= mine[:, -1] * (1 - 1e-5) - 1e-12)


def test_edge_cases(env):
    """n < k, NaN entries, a NaN observation and an all-NaN table give trailing NO_ENTRY / NaN; m = 0 is empty."""
    torch, _, lut = env
    rng = np.random.default_rng(8)
    L = grid_table(rng, 5, 4)
    O = grid_table(rng, 3, 4)
    idx, cost = lut.nearest_k(torch.from_numpy(L).cuda(), torch.from_numpy(O).cuda(), 10)
    want_idx, want_cost, _ = brute_k(L, O, 10)
    assert np.array_equal(idx.cpu().numpy(), want_idx) and (idx[:, 5:] == NO_ENTRY).all()
    assert np.array_equal(cost.cpu().numpy(), want_cost, equal_nan=True) and torch.isnan(cost[:, 5:]).all()
    L = grid_table(rng, 3000, 6)
    L[rng.permutation(3000)[:2990]] = np.nan              # 10 valid entries
    O = grid_table(rng, 20, 6)
    O[7] = np.nan
    idx, cost = lut.nearest_k(torch.from_numpy(L).cuda(), torch.from_numpy(O).cuda(), 16)
    want_idx, want_cost, _ = brute_k(L, O, 16)
    assert np.array_equal(idx.cpu().numpy(), want_idx) and (idx[7] == NO_ENTRY).all()
    assert np.array_equal(cost.cpu().numpy(), want_cost, equal_nan=True)
    assert (idx[torch.tensor([i for i in range(20) if i != 7]), 10:] == NO_ENTRY).all()
    idx, cost = lut.nearest_k(torch.full((500, 6), float("nan"), device="cuda"), torch.from_numpy(O).cuda(), 3)
    assert (idx == NO_ENTRY).all() and torch.isnan(cost).all()
    idx, cost = lut.nearest_k(torch.from_numpy(L).cuda(), torch.zeros((0, 6), device="cuda"), 4)
    assert idx.shape == (0, 4) and cost.shape == (0, 4)


def test_refusals_python_and_c_abi(env):
    torch, sb, lut = env
    from spart_b200 import _lib
    lib = _lib.load()
    L, O = torch.rand((100, 8), device="cuda"), torch.rand((4, 8), device="cuda")
    for k in (0, 129):
        with pytest.raises(sb.SpartError, match="1 <= k <= 128"):
            lut.nearest_k(L, O, k)
    with pytest.raises(sb.SpartError, match="n_bands <= 32"):
        lut.nearest_k(torch.rand((100, 33), device="cuda"), torch.rand((4, 33), device="cuda"), 5)
    with pytest.raises(sb.SpartError, match="index_offset"):
        lut._search_k(L, O, 5, None, 2 ** 32 - 100, packed=False)
    ws = torch.empty(lib.spart_lut_topk_workspace_bytes(100, 4, 128) // 8, dtype=torch.int64, device="cuda")
    idx = torch.empty((4, 128), dtype=torch.int64, device="cuda")
    cost = torch.empty((4, 128), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(n=100, nb=8, k=5, off=0):
        return lib.spart_lut_topk(L.data_ptr(), n, nb, O.data_ptr(), 4, k, 0, off, ws.data_ptr(), idx.data_ptr(),
                                  cost.data_ptr(), 0, stream)

    assert call() == 0
    for kw in (dict(k=0), dict(k=129), dict(nb=33), dict(off=2 ** 32 - 100), dict(n=0)):
        assert call(**kw) == -1, kw                                    # SPART_EINVAL
    assert b"spart_lut_topk" in lib.spart_last_error()
    assert lib.spart_lut_topk_merge(ws.data_ptr(), 0, 4, 5, idx.data_ptr(), cost.data_ptr(), 0, stream) == -1
    assert lib.spart_lut_topk_merge(ws.data_ptr(), 1, 4, 129, idx.data_ptr(), cost.data_ptr(), 0, stream) == -1
    assert lib.spart_lut_topk_workspace_bytes(100, 4, 129) == 0 and lib.spart_lut_topk_workspace_bytes(0, 4, 5) == 0
    torch.cuda.synchronize()


def test_pieces_merge_to_the_whole_table(env, tmp_path):
    """Three uneven pieces, one all NaN, searched with their offsets and merged, equal the whole-table search bit for
    bit; `nearest_k_sharded` at world size 1 on NCCL equals `nearest_k`."""
    torch, _, lut = env
    rng = np.random.default_rng(12)
    n, nb, k = 70_001, 8, 32
    L = grid_table(rng, n, nb)
    L[rng.permutation(n)[:5000]] = L[rng.integers(0, n, size=5000)]
    L[40_000:52_000] = np.nan
    O = grid_table(rng, 3000, nb)
    Ld, Od = torch.from_numpy(L).cuda(), torch.from_numpy(O).cuda()
    whole = lut.nearest_k(Ld, Od, k)
    cuts = (0, 40_000, 52_000, n)
    lists = torch.stack([lut._search_k(Ld[a:b].contiguous(), Od, k, None, a, packed=True)
                         for a, b in zip(cuts[:-1], cuts[1:])])
    assert (lists[1] == -1).all()                                  # the all-NaN piece: only "no entry" words
    assert same(torch, lut.merge_k(lists), whole)
    assert same(torch, lut.merge_k(lists[[2, 1, 0]]), whole)       # list order does not matter
    import torch.distributed as dist
    dist.init_process_group("nccl", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1,
                            device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        w = torch.rand(nb, device="cuda") + 0.5
        assert same(torch, lut.nearest_k_sharded(Ld, Od, k), whole)
        assert same(torch, lut.nearest_k_sharded(Ld, Od, 5, w), lut.nearest_k(Ld, Od, 5, w))
    finally:
        dist.destroy_process_group()


def numpy_moments(params_np, idx):
    """float64 mean / population std / count over the valid neighbours of each row; params_np [n, P]."""
    m, P = idx.shape[0], params_np.shape[1]
    mean, std = np.full((m, P), np.nan), np.full((m, P), np.nan)
    count = np.zeros(m, dtype=np.int64)
    for o in range(m):
        sel = params_np[idx[o][idx[o] != NO_ENTRY]]
        count[o] = len(sel)
        if len(sel):
            mean[o], std[o] = sel.mean(0), sel.std(0)
    return mean, std, count


def test_estimate_layouts_types_and_pieces(env):
    torch, _, lut = env
    rng = np.random.default_rng(27)
    n, P, k = 5000, 27, 20
    table = rng.random((n, P)) * np.logspace(-3, 3, P)
    table[:, 5] = 183.0                                            # a constant row (e.g. a fixed DOY)
    L = torch.rand((n, 6), device="cuda")
    L[rng.permutation(n)[:4990]] = float("nan")                    # 10 valid entries: NO_ENTRY slots beyond
    O = torch.rand((300, 6), device="cuda")
    idx_few, _ = lut.nearest_k(L, O, k)
    idx_full, _ = lut.nearest_k(torch.rand((n, 6), device="cuda"), O, k)
    for idx in (idx_few, idx_full):
        idx_np = idx.cpu().numpy()
        for dtype in (torch.float64, torch.float32):
            t = torch.from_numpy(table).to("cuda", dtype)
            ref = t.double().cpu().numpy()
            want_mean, want_std, want_count = numpy_moments(ref, idx_np)
            for params in (t.T.contiguous(), t.T):                 # [P, n] batch layout, and an [n, P] table's view
                mean, std, count = lut.estimate(params, idx)
                assert np.array_equal(count.cpu().numpy(), want_count)
                np.testing.assert_allclose(mean.cpu().numpy(), want_mean, rtol=1e-14, atol=0)
                np.testing.assert_allclose(std.cpu().numpy(), want_std, rtol=1e-12,
                                           atol=1e-14 * np.abs(want_mean).max())
                assert torch.all(std[:, 5] <= 1e-14 * mean[:, 5].abs())
        # pieces of the table accumulated with their offsets equal one call
        t = torch.from_numpy(table).cuda()
        one = torch.zeros((300, P + 1), dtype=torch.float64, device="cuda")
        lut._accumulate(t.T, idx, 0, None, one)
        parts = torch.zeros_like(one)
        for a, b in ((0, 1234), (1234, 1240), (1240, n)):
            lut._accumulate(t[a:b].T, idx, a, None, parts)
        assert torch.allclose(parts, one, rtol=1e-14, atol=0)


def test_estimate_of_index_views(env):
    """`estimate` on views of a neighbour index (the first / last neighbours, every other row or column, a transposed
    layout) uses exactly the neighbours the view shows."""
    torch, _, lut = env
    rng = np.random.default_rng(31)
    n, P = 4000, 27
    table = rng.random((n, P)) * np.logspace(-2, 2, P)
    idx, _ = lut.nearest_k(torch.rand((n, 5), device="cuda"), torch.rand((200, 5), device="cuda"), 50)
    params = torch.from_numpy(table).cuda().T
    for view in (idx[:, :10], idx[:, 5:], idx[::2], idx[:, ::3], idx.T.contiguous().T):
        assert not view.is_contiguous()
        mean, std, count = lut.estimate(params, view)
        want_mean, want_std, want_count = numpy_moments(table, view.cpu().numpy())
        assert np.array_equal(count.cpu().numpy(), want_count)
        np.testing.assert_allclose(mean.cpu().numpy(), want_mean, rtol=1e-14, atol=0)
        np.testing.assert_allclose(std.cpu().numpy(), want_std, rtol=1e-12, atol=1e-14 * np.abs(want_mean).max())


def test_estimate_refuses_params_on_another_gpu(env):
    torch, _, lut = env
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    idx = torch.zeros((4, 3), dtype=torch.int64, device="cuda:0")
    with pytest.raises(ValueError, match="same CUDA device"):
        lut.estimate(torch.rand((27, 10), dtype=torch.float64, device="cuda:1"), idx)


def test_end_to_end_sentinel2a(env):
    """A Sentinel-2A table from synthetic parameters: table rows find themselves first at cost 0, and the estimate
    over the k = 20 entries of simulated observations is the NumPy mean / std of those parameter rows."""
    torch, sb, lut = env
    import spart_oracle as so
    P = so.synthetic_params(20_000, 2, seed=91)
    table = lut.generate(P.T, "Sentinel2A-MSI", column=0, uniform_geometry=True)
    idx, cost = lut.nearest_k(table, table[100:164].clone(), 5)
    assert torch.equal(idx[:, 0].cpu(), torch.arange(100, 164)) and float(cost[:, 0].abs().max()) == 0.0
    held = so.synthetic_params(50, 2, seed=92)
    obs = lut.generate(held.T, "Sentinel2A-MSI", column=0, uniform_geometry=True)
    idx, cost = lut.nearest_k(table, obs, 20)
    assert (idx != NO_ENTRY).all()
    params = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    mean, std, count = lut.estimate(params, idx)
    want_mean, want_std, _ = numpy_moments(P, idx.cpu().numpy())
    assert (count == 20).all()
    np.testing.assert_allclose(mean.cpu().numpy(), want_mean, rtol=1e-14, atol=0)
    np.testing.assert_allclose(std.cpu().numpy(), want_std, rtol=1e-12, atol=1e-13 * np.abs(want_mean).max())


def _retrieve(torch, lut, L, O, lists, params, k=32):
    idx, cost = lut.nearest_k(L, O, k)
    merged = lut.merge_k(lists)
    return [idx, cost, *merged, *lut.estimate(params, idx)]


def test_stream_and_thread_contract(env, cycles):
    """Search, merge and moments enqueued on a side stream behind a GPU delay, and on two host threads with two
    streams (k = 32 and k = 10: different heap sizes of the same kernel), give the same bits as on the default
    stream."""
    torch, _, lut = env
    rng = np.random.default_rng(4)
    L = torch.from_numpy(grid_table(rng, 200_000, 8)).cuda()
    O = torch.from_numpy(grid_table(rng, 2000, 8)).cuda()
    lists = torch.stack([lut._search_k(L[a:a + 50_000].contiguous(), O, 32, None, a, packed=True)
                         for a in range(0, 200_000, 50_000)])
    params = torch.rand((27, 200_000), dtype=torch.float64, device="cuda")
    want = _retrieve(torch, lut, L, O, lists, params)
    want10 = _retrieve(torch, lut, L, O, lists, params, k=10)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(cycles)
        got = _retrieve(torch, lut, L, O, lists, params)
    side.synchronize()
    assert same(torch, got, want)
    out, errs = [None, None], []

    def work(i):
        try:
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                torch.cuda._sleep(cycles // 4)
                out[i] = _retrieve(torch, lut, L, O, lists, params, k=(32, 10)[i])
            s.synchronize()
        except Exception as e:                                     # noqa: BLE001 -- reported below
            errs.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs
    assert same(torch, out[0], want) and same(torch, out[1], want10)
