"""Look-up-table helpers: generation in chunks and nearest-entry retrieval on the GPU.

`generate` runs a parameter block through the forward model chunk by chunk (bounded device
memory) and returns / stores the band outputs; `nearest` is the retrieval step: the LUT entry with
the smallest weighted squared distance to each observed band vector (spart_lut_nearest).
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
    w = None
    if weights is not None:
        w = torch.as_tensor(weights, dtype=torch.float32, device=lut.device).reshape(nb).clamp_min(0).sqrt().contiguous()
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
