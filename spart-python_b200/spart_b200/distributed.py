"""Data-parallel sharding of a parameter batch over the GPUs of one node.

Samples are independent, so the batch is split into contiguous slices, one per rank, with no
data-path collective; the only collective is the final gather of the [n, nb, 3] results
(NCCL over NVLink when the tensors are on GPUs, gloo in the CPU tests).  `gather_pipelined` issues that
gather chunk by chunk on a side stream so that it hides behind the next chunk's kernels.
"""
import torch
import torch.distributed as dist


def shard_bounds(n, world_size, rank):
    """Contiguous slice [lo, hi) of rank `rank`: sizes differ by at most one sample."""
    if world_size <= 0 or not (0 <= rank < world_size):
        raise ValueError("bad rank / world_size")
    base, rem = divmod(int(n), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_results(local, n_total, group=None, dst=None):
    """Concatenate per-rank [n_r, nb, 3] results in rank order.

    dst=None: every rank gets the full [n_total, nb, 3] tensor (all_gather);
    dst=r:    only rank r gets it (others get None).
    Shard sizes differ by at most one sample, so each rank contributes a buffer padded to the
    largest shard and the padding row is dropped after the collective."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    tail = tuple(local.shape[1:])
    bounds = [shard_bounds(n_total, world, r) for r in range(world)]
    mine = bounds[rank][1] - bounds[rank][0]
    if local.shape[0] != mine:
        raise ValueError("local shard has the wrong number of samples for this rank")
    cap = max(hi - lo for lo, hi in bounds)
    if mine == cap:
        send = local.contiguous()
    else:
        send = torch.zeros((cap,) + tail, dtype=local.dtype, device=local.device)
        send[:mine] = local
    even = all(hi - lo == cap for lo, hi in bounds)
    want = dst is None or rank == dst
    recv = torch.empty((world * cap,) + tail, dtype=local.dtype, device=local.device) if want else None
    if dst is None:
        dist.all_gather_into_tensor(recv, send, group=group)
    else:
        parts = list(recv.chunk(world, dim=0)) if want else None
        dist.gather(send, gather_list=parts, dst=dst, group=group)
    if not want:
        return None
    if even:
        return recv
    return torch.cat([recv[r * cap:r * cap + (hi - lo)] for r, (lo, hi) in enumerate(bounds)], dim=0)


def run_batch_sharded(params, sensor, precision="fp64", group=None, dst=None, compute=None):
    """Every rank holds (or can index) the full [27, n] block; each computes its slice and
    the results are gathered.  `compute(params_slice, sensor, precision)` defaults to the
    CUDA path; tests inject a stand-in to exercise the sharding/gather logic without a GPU."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n = params.shape[1]
    lo, hi = shard_bounds(n, world, rank)
    if compute is None:
        from .batch import run_batch_params
        compute = lambda p, s, pr: run_batch_params(p, s, pr)
    local = compute(params[:, lo:hi].contiguous(), sensor, precision)
    return gather_results(local, n, group=group, dst=dst)


# ---- gather pipelined behind the computation -----------------------------------------------------
def chunk_bounds(n, chunk):
    """[(lo, hi), ...] covering [0, n) in pieces of at most `chunk` samples."""
    chunk = max(int(chunk), 1)
    return [(lo, min(lo + chunk, n)) for lo in range(0, n, chunk)] or [(0, 0)]


def gather_pipelined(compute_chunk, block_elems, dtype, device, group=None, dst=0, local=None, recv=None):
    """Run a sharded computation chunk by chunk and gather every finished chunk on rank `dst` WHILE the
    next chunk is being computed (the only collective of the path, SURVEY.md section 8(e)).

    compute_chunk(c, view): enqueue on the current stream the computation of local chunk c into `view`, a
    flat tensor of block_elems[c] elements (all ranks use the same block sizes; pad the last chunk).
    The gather of chunk c is issued on a side stream that waits for chunk c's kernels only, so it overlaps
    chunk c + 1's kernels; the caller's stream waits for the last gather before the function returns
    (stream-ordered, no host synchronisation).  On CPU tensors (gloo, tests) the same steps run in order.
    Returns (local, recv): the rank's flat result and, on `dst`, recv [world, sum(block_elems)] in rank
    order (None elsewhere).  `local` / `recv` may be passed in to reuse buffers between steps."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    total = int(sum(block_elems))
    device = torch.device(device)
    if local is None:
        local = torch.empty(total, dtype=dtype, device=device)
    if rank == dst and recv is None:
        recv = torch.empty((world, total), dtype=dtype, device=device)
    cuda = device.type == "cuda"
    if cuda:
        main = torch.cuda.current_stream(device)
        side = _side_stream(device)
        side.wait_stream(main)           # buffers handed in by the caller are ready before the side stream touches them
    off = 0
    for c, elems in enumerate(block_elems):
        view = local[off:off + elems]
        compute_chunk(c, view)
        parts = [recv[r, off:off + elems] for r in range(world)] if rank == dst else None
        if cuda:
            done = torch.cuda.Event()
            done.record(main)
            side.wait_event(done)
            with torch.cuda.stream(side):
                dist.gather(view, gather_list=parts, dst=dst, group=group)
        else:
            dist.gather(view, gather_list=parts, dst=dst, group=group)
        off += elems
    if cuda:
        main.wait_stream(side)
    return local, (recv if rank == dst else None)


_side = {}


def _side_stream(device):
    key = (device.type, device.index)
    if key not in _side:
        _side[key] = torch.cuda.Stream(device)
    return _side[key]


def run_batch_sharded_pipelined(params_local, sensor, precision="fp64", chunk=1 << 18, group=None, dst=0,
                                broadcast_rows=0, compact=False, compute=None, local=None, recv=None):
    """Each rank holds ITS shard `params_local` [27, n_local] (same n_local on every rank); the shard is
    evaluated in chunks of `chunk` samples and chunk c's results travel to rank `dst` while chunk c + 1 is
    computed.  Returns on `dst` a list over ranks of per-chunk results (tensors [m, nb, 3], or CompactBands
    when compact -- two thirds of the bytes over NVLink, float32 parameters with precision="fp32" half of
    that again), None elsewhere.  `compute(params_chunk, view)` defaults to the CUDA path; tests inject a
    stand-in to exercise the chunking / gather logic with gloo."""
    from .engine import NOUT, CompactBands, default_engine, out_elems
    n = params_local.shape[1]
    bounds = chunk_bounds(n, chunk)
    if compute is None:
        eng = default_engine(params_local.device)
        _, st = eng.sensor(sensor)
        nb, conv_ea = st.n_bands, st.conv_ea

        def compute(p, view):
            # p is a column slice of params_local: the broadcast rows' values sit in params_local's column 0
            eng.forward_bands(p, sensor, out=view if compact else view.view(p.shape[1], nb, NOUT), precision=precision,
                              broadcast_rows=broadcast_rows, compact=compact, broadcast_base=params_local)
    else:
        nb, conv_ea = compute.n_bands, getattr(compute, "conv_ea", None)
    blocks = [out_elems(hi - lo, nb, compact) for lo, hi in bounds]
    local, recv = gather_pipelined(lambda c, view: compute(params_local[:, bounds[c][0]:bounds[c][1]], view), blocks,
                                   params_local.dtype, params_local.device, group=group, dst=dst, local=local, recv=recv)
    if recv is None:
        return None
    res = []
    for r in range(recv.shape[0]):
        off, per = 0, []
        for (lo, hi), e in zip(bounds, blocks):
            blk = recv[r, off:off + e]
            per.append(CompactBands(blk, hi - lo, nb, conv_ea, precision in ("fp32", 32)) if compact
                       else blk.view(hi - lo, nb, NOUT))
            off += e
        res.append(per)
    return res
