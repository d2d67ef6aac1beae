"""Look-up-table helpers: generation in chunks and nearest-entry retrieval on the GPU.

`generate` runs a parameter block through the forward model chunk by chunk (bounded device
memory) and returns / stores the band outputs; `nearest` is the retrieval step: the LUT entry with
the smallest weighted squared distance to each observed band vector (spart_lut_nearest).  `nearest_k`
returns the k best entries (spart_lut_topk) and `estimate` the mean and spread of their parameters, the
usual answer to an ill-posed inversion; both have sharded forms that never gather the table.
"""
import numpy as np
import torch

from . import _lib
from .engine import default_engine

NO_ENTRY = 2 ** 32 - 1      # index `nearest` returns (with cost NaN) for an observation without a finite-cost entry


def generate(params, sensor, precision="fp64", chunk=1 << 20, out_dtype=torch.float32, column=None, path=None,
             uniform_geometry=False, soil_library=None):
    """params: [27, n] (NumPy or torch, host or device).  Evaluates the batch in chunks of `chunk`
    samples and returns a CUDA tensor [n, nb, 3] (or [n, nb] when `column` selects 0 = R_TOC,
    1 = R_TOA, 2 = L_TOA) in `out_dtype`.  With `path` the table is also written as a compressed
    .npz holding `params` [n, 27] float32 and `lut`.  soil_library: a SoilLibrary; row 9 of params then
    holds each entry's index into it, so the stored params tell which soil the nearest entry of a
    retrieval used."""
    eng = default_engine()
    p = params if isinstance(params, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(params))
    n = p.shape[1]
    _, st = eng.sensor(sensor, soil_library=soil_library)
    shape = (n, st.n_bands) if column is not None else (n, st.n_bands, 3)
    lut = torch.empty(shape, dtype=out_dtype, device=eng.device)
    for s0 in range(0, n, chunk):
        blk = p[:, s0:s0 + chunk].to(eng.device, dtype=torch.float64).contiguous()
        res = eng.forward_bands(blk, sensor, precision=precision, uniform_geometry=uniform_geometry,
                                soil_library=soil_library)
        lut[s0:s0 + chunk] = (res[..., column] if column is not None else res).to(out_dtype)
    if path is not None:
        np.savez_compressed(path, params=p.T.to(torch.float32).cpu().numpy(), lut=lut.cpu().numpy(),
                            sensor=np.array(sensor if isinstance(sensor, str) else "custom"))
    return lut


def _check(lut, obs):
    if not (lut.is_cuda and obs.is_cuda and lut.dtype == torch.float32 and obs.dtype == torch.float32
            and lut.dim() == 2 and obs.dim() == 2 and lut.shape[1] == obs.shape[1]):
        raise ValueError("lut [n, nb] and obs [m, nb] must be CUDA float32 tensors with the same band count")


def _sqrt_weights(weights, nb, device):
    if weights is None:
        return None
    return torch.as_tensor(weights, dtype=torch.float32, device=device).reshape(nb).clamp_min(0).sqrt().contiguous()


def _search(lut, obs, weights, index_offset, packed, method="exact"):
    """spart_lut_nearest (method="exact": FP32 SIMT) or spart_lut_nearest_tc (method="tensor": 3xTF32 tensor-core
    search + exact re-costing of the winner) on the current stream.  packed=True: returns the int64 words
    (cost bits << 32 | global index) instead of (index, cost)."""
    if method not in ("exact", "tensor"):
        raise ValueError("method must be 'exact' or 'tensor'")
    lib = _lib.load()
    fn = lib.spart_lut_nearest if method == "exact" else lib.spart_lut_nearest_tc
    lut, obs = lut.contiguous(), obs.contiguous()
    n, nb = lut.shape
    m = obs.shape[0]
    w = _sqrt_weights(weights, nb, lut.device)
    ws = torch.empty(max(lib.spart_lut_workspace_bytes(m) // 8, 1), dtype=torch.int64, device=lut.device)
    words = torch.empty(m, dtype=torch.int64, device=lut.device) if packed else None
    idx = None if packed else torch.empty(m, dtype=torch.int64, device=lut.device)
    cost = None if packed else torch.empty(m, dtype=torch.float32, device=lut.device)
    with torch.cuda.device(lut.device):
        stream = torch.cuda.current_stream(lut.device).cuda_stream
        _lib.check(fn(lut.data_ptr(), n, nb, obs.data_ptr(), m, 0 if w is None else w.data_ptr(),
                                         int(index_offset), ws.data_ptr(), 0 if packed else idx.data_ptr(),
                                         0 if packed else cost.data_ptr(), words.data_ptr() if packed else 0,
                                         stream), "spart_lut_nearest")
    return words if packed else (idx, cost)


def unpack(words):
    """int64 words (cost bits << 32 | index) -> (index int64 [m], cost float32 [m])."""
    lib = _lib.load()
    m = words.shape[0]
    idx = torch.empty(m, dtype=torch.int64, device=words.device)
    cost = torch.empty(m, dtype=torch.float32, device=words.device)
    with torch.cuda.device(words.device):
        stream = torch.cuda.current_stream(words.device).cuda_stream
        _lib.check(lib.spart_lut_unpack(words.data_ptr(), m, idx.data_ptr(), cost.data_ptr(), stream),
                   "spart_lut_unpack")
    return idx, cost


def nearest(lut, obs, weights=None, method="exact"):
    """lut: CUDA float32 [n, nb]; obs: CUDA float32 [m, nb]; weights: optional per-band weights [nb].
    Returns (index int64 [m], cost float32 [m]) of the entry minimising sum_b w_b (obs_b - lut_b)^2, ties to the
    lowest index.  Entries whose cost is NaN (a NaN value in the entry or in the observation) or not below 3e38 are
    never chosen; an observation without any other entry gets the "no entry" result: index 2^32 - 1
    (NO_ENTRY) and cost NaN.
    method="tensor": the comparison runs on the tensor cores in 3xTF32 (the entry is optimal up to ~1e-6 of
    |obs||entry|, its cost is exact)."""
    _check(lut, obs)
    return _search(lut, obs, weights, 0, packed=False, method=method)


def for_min_reduction(words):
    """Packed words of a search piece, ready for a signed 64-bit min-reduction with other pieces: the all-ones
    "no entry" word is -1 as int64 and would win, so it becomes the reduction's identity 2^63 - 1 (which unpacks
    to the same "no entry" result, index NO_ENTRY and cost NaN)."""
    return words.masked_fill(words == -1, 2 ** 63 - 1)


def nearest_sharded(lut_local, obs, weights=None, group=None, index_offset=None, search=None, unpack_words=None,
                    method="exact"):
    """Retrieval against a table that stays sharded over the ranks of `group` (each rank holds
    `lut_local` [n_r, nb], rank order = table order; every rank passes the same `obs`).  Each GPU
    searches its own slice, the per-observation words (cost bits << 32 | global index) are
    min-reduced with one NCCL all-reduce of 8 bytes per observation, and every rank returns the
    global (index, cost); an observation that finds no entry on any rank gets `nearest`'s "no entry"
    result.  The table itself is never gathered.  `search` / `unpack_words` default to the
    CUDA kernels; CPU tests inject stand-ins to exercise the reduction logic with gloo."""
    import torch.distributed as dist
    if index_offset is None:
        sizes = [None] * dist.get_world_size(group)
        dist.all_gather_object(sizes, int(lut_local.shape[0]), group=group)
        index_offset = sum(sizes[:dist.get_rank(group)])
        if sum(sizes) >= 2 ** 32:
            raise ValueError("nearest_sharded: the table has 2^32 entries or more")
    if search is None:
        _check(lut_local, obs)
        search = lambda l, o, w, off: _search(l, o, w, off, packed=True, method=method)
    if lut_local.shape[0] == 0:       # a rank without entries contributes the identity of the min-reduction
        words = torch.full((obs.shape[0],), 2 ** 63 - 1, dtype=torch.int64, device=obs.device)
    else:
        words = for_min_reduction(search(lut_local, obs, weights, index_offset))
    # costs are >= 0, so the signed 64-bit order of the words is the (cost, index) order
    dist.all_reduce(words, op=dist.ReduceOp.MIN, group=group)
    return (unpack_words or unpack)(words)


def _search_k(lut, obs, k, weights, index_offset, packed):
    """spart_lut_topk on the current stream: (index int64 [m, k], cost float32 [m, k]), or with packed=True the
    sorted int64 words [m, k] (cost bits << 32 | global index)."""
    lib = _lib.load()
    lut, obs = lut.contiguous(), obs.contiguous()
    n, nb = lut.shape
    m = obs.shape[0]
    if m == 0 and 1 <= k <= 128:      # an empty tensor may have no data pointer, which the C ABI refuses
        return torch.empty((0, k), dtype=torch.int64, device=lut.device) if packed else (
            torch.empty((0, k), dtype=torch.int64, device=lut.device),
            torch.empty((0, k), dtype=torch.float32, device=lut.device))
    w = _sqrt_weights(weights, nb, lut.device)
    ws = torch.empty(max(lib.spart_lut_topk_workspace_bytes(n, m, k) // 8, 1), dtype=torch.int64, device=lut.device)
    shape = (m, max(int(k), 0))
    words = torch.empty(shape, dtype=torch.int64, device=lut.device) if packed else None
    idx = None if packed else torch.empty(shape, dtype=torch.int64, device=lut.device)
    cost = None if packed else torch.empty(shape, dtype=torch.float32, device=lut.device)
    with torch.cuda.device(lut.device):
        stream = torch.cuda.current_stream(lut.device).cuda_stream
        _lib.check(lib.spart_lut_topk(lut.data_ptr(), n, nb, obs.data_ptr(), m, int(k), 0 if w is None else w.data_ptr(),
                                      int(index_offset), ws.data_ptr(), 0 if packed else idx.data_ptr(),
                                      0 if packed else cost.data_ptr(), words.data_ptr() if packed else 0, stream),
                   "spart_lut_topk")
    return words if packed else (idx, cost)


def nearest_k(lut, obs, k, weights=None):
    """lut: CUDA float32 [n, nb]; obs: CUDA float32 [m, nb]; 1 <= k <= 128; weights: optional per-band weights [nb].
    Returns (index int64 [m, k], cost float32 [m, k]): per observation the k entries with the smallest
    sum_b w_b (obs_b - lut_b)^2, ascending by cost, ties to the lowest index (also at the k-th place).  The cost is
    `nearest`'s bit for bit, so k = 1 gives `nearest`'s result.  Entries whose cost is NaN or not below 3e38 are
    never chosen; slots beyond the qualifying entries get index NO_ENTRY and cost NaN."""
    _check(lut, obs)
    return _search_k(lut, obs, k, weights, 0, packed=False)


def merge_k(lists):
    """lists: CUDA int64 [L, m, k], L ascending lists of packed words per observation (e.g. the `nearest_k` words
    of L table pieces).  Returns the (index [m, k], cost [m, k]) of the k smallest words (spart_lut_topk_merge)."""
    lib = _lib.load()
    lists = lists.contiguous()
    L, m, k = lists.shape
    idx = torch.empty((m, k), dtype=torch.int64, device=lists.device)
    cost = torch.empty((m, k), dtype=torch.float32, device=lists.device)
    with torch.cuda.device(lists.device):
        stream = torch.cuda.current_stream(lists.device).cuda_stream
        _lib.check(lib.spart_lut_topk_merge(lists.data_ptr(), L, m, k, idx.data_ptr(), cost.data_ptr(), 0, stream),
                   "spart_lut_topk_merge")
    return idx, cost


def _table_offset(n_local, group, who):
    """First global entry of this rank's piece (rank order = table order); refuses a table of 2^32 entries or more."""
    import torch.distributed as dist
    sizes = [None] * dist.get_world_size(group)
    dist.all_gather_object(sizes, int(n_local), group=group)
    if sum(sizes) >= 2 ** 32:
        raise ValueError(f"{who}: the table has 2^32 entries or more")
    return sum(sizes[:dist.get_rank(group)])


def nearest_k_sharded(lut_local, obs, k, weights=None, group=None, index_offset=None, search=None, merge=None):
    """`nearest_k` against a table that stays sharded over the ranks of `group` (each rank holds `lut_local`
    [n_r, nb], rank order = table order; every rank passes the same `obs`).  Each GPU finds the k best words of
    its slice, one all-gather of m * k * 8 bytes per rank collects the W lists and spart_lut_topk_merge reduces
    them, so every rank returns the same global (index [m, k], cost [m, k]) as `nearest_k` on the whole table.
    A rank without entries contributes a list of "no entry" words.  `search` (lut, obs, k, weights, offset ->
    words [m, k]) and `merge` (lists [W, m, k] -> (index, cost)) default to the CUDA kernels; CPU tests inject
    stand-ins to exercise the reduction with gloo."""
    import torch.distributed as dist
    if not 1 <= k <= 128:             # before any collective: a rank must not wait for others that refused
        raise ValueError("nearest_k_sharded: need 1 <= k <= 128")
    if index_offset is None:
        index_offset = _table_offset(lut_local.shape[0], group, "nearest_k_sharded")
    if search is None:
        _check(lut_local, obs)
        search = lambda l, o, kk, w, off: _search_k(l, o, kk, w, off, packed=True)
    if lut_local.shape[0] == 0:
        words = torch.full((obs.shape[0], k), -1, dtype=torch.int64, device=obs.device)
    else:
        words = search(lut_local, obs, k, weights, index_offset)
    lists = [torch.empty_like(words) for _ in range(dist.get_world_size(group))]
    dist.all_gather(lists, words, group=group)
    return (merge or merge_k)(torch.stack(lists))


def _accumulate(params, index, index_offset, centre, acc):
    """spart_lut_moments_accumulate: adds this table piece's sums (centre None) or squared deviations from
    centre [m, P] to acc [m, P + 1] (last column: the count)."""
    lib = _lib.load()
    if not (params.is_cuda and params.dim() == 2 and params.dtype in (torch.float64, torch.float32)):
        raise ValueError("params must be a CUDA float64 or float32 tensor [P, n] (or the view .T of an [n, P] table)")
    if not (index.is_cuda and index.dtype == torch.int64 and index.dim() == 2):
        raise ValueError("index must be a CUDA int64 tensor [m, k]")
    if any(t is not None and t.device != index.device for t in (params, centre, acc)):
        raise ValueError("params, index, centre and acc must be on the same CUDA device")
    index = index.contiguous()        # the kernel reads a dense [m][k]; a view such as idx[:, :10] is copied
    P, n_local = params.shape
    m, k = index.shape
    flags = _lib.FLAG_F32_IO if params.dtype == torch.float32 else 0
    with torch.cuda.device(index.device):
        stream = torch.cuda.current_stream(index.device).cuda_stream
        _lib.check(lib.spart_lut_moments_accumulate(params.data_ptr(), P, params.stride(0), params.stride(1), flags,
                                                    int(index_offset), n_local, index.data_ptr(), m, k,
                                                    0 if centre is None else centre.data_ptr(), acc.data_ptr(), stream),
                   "spart_lut_moments_accumulate")


def _finish(acc, sq):
    """spart_lut_moments_finish: (mean [m, P], std [m, P] or None without sq, count int64 [m])."""
    lib = _lib.load()
    m, P = acc.shape[0], acc.shape[1] - 1
    mean = torch.empty((m, P), dtype=torch.float64, device=acc.device)
    std = None if sq is None else torch.empty((m, P), dtype=torch.float64, device=acc.device)
    count = torch.empty(m, dtype=torch.int64, device=acc.device)
    with torch.cuda.device(acc.device):
        stream = torch.cuda.current_stream(acc.device).cuda_stream
        _lib.check(lib.spart_lut_moments_finish(acc.data_ptr(), 0 if sq is None else sq.data_ptr(), m, P,
                                                mean.data_ptr(), 0 if std is None else std.data_ptr(),
                                                count.data_ptr(), stream), "spart_lut_moments_finish")
    return mean, std, count


def estimate(params, index, index_offset=None, group=None, accumulate=None, finish=None):
    """Mean and spread of the parameters of the entries `index` (CUDA int64 [m, k], e.g. from `nearest_k`; NO_ENTRY
    slots and indices outside this table piece are skipped).  params: the parameter table of the LUT, or of this
    rank's slice of it, as a CUDA float64 or float32 tensor [P, n] -- the [27, n] batch layout of `generate`'s input,
    or the transposed view `table.T` of an [n, P] table such as the `params` of a `generate` .npz; it is read
    through its strides, without a copy.  Returns (mean float64 [m, P], std float64 [m, P], count int64 [m]): the
    population standard deviation over the count neighbours found; count 0 gives NaN.  Two passes, each a plain
    FP64 sum in neighbour order (sums and count, then squared deviations from that mean), so a parameter that is
    the same in every neighbour gets std 0, not rounding noise of the mean.
    With `group` the table is sharded over its ranks (rank order = table order, every rank passes the same
    `index`): each pass ends in one SUM all-reduce of m * (P + 1) doubles, and index_offset (default: found from the
    slice sizes) is the first global entry of this rank's slice.  Without `group` there is no communication and
    index_offset defaults to 0.  `accumulate` / `finish` default to the CUDA kernels; CPU tests inject stand-ins."""
    accumulate, finish = accumulate or _accumulate, finish or _finish
    index = index.contiguous()        # once for both passes
    if index_offset is None:
        index_offset = 0 if group is None else _table_offset(params.shape[1], group, "estimate")
    m, P = index.shape[0], params.shape[0]

    def pass_(centre):
        acc = torch.zeros((m, P + 1), dtype=torch.float64, device=index.device)
        accumulate(params, index, index_offset, centre, acc)
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
        return acc

    acc = pass_(None)
    mean, _, _ = finish(acc, None)
    return finish(acc, pass_(mean))
