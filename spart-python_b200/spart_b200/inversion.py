"""Per-observation retrieval by bounded Levenberg-Marquardt on the GPU.

A look-up table answers an inversion only to the fineness of its grid.  `invert` refines each observation from a
few starts (typically the parameters of `lut.nearest_k`'s entries, turned into starts by `starts`) to the parameter
set of a `sensitivity.ParameterSpace` box that minimises C(x) = sum_b w_b (f_b(x) - y_b)^2, with a covariance-based
standard deviation.  The design of each iteration's forward batch, the Levenberg-Marquardt step of every track and
the pick of the best start run as CUDA kernels (spart_invert_design, spart_invert_step, spart_invert_finish); the
forward model is `Engine.forward_bands` in FP64.  The algorithm is pinned in include/spart_b200.h and DESIGN.md §8;
tests/test_invert_cpu.py restates it in NumPy.

A track (one start of one observation) is iterated in u in [0, 1]^P, x = lo + (hi - lo) u.  An iteration is one
forward call of P + 1 samples per active track: the trial point and one forward-difference sample per parameter
(step 2^-17 of the range).  The step accepts the trial if its cost is strictly lower (then lambda / 10, else
lambda x 10), solves (J^T W J + lambda diag(J^T W J)) delta = -J^T W r by Cholesky and clips u + delta to the box.
A stopped track costs no further forward runs: each iteration's batch covers the active tracks only.
"""
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .engine import default_engine
from .lut import NO_ENTRY
from .sensitivity import LIDFA, LIDFB, NPAR, ROW_NAMES, ParameterSpace

ACTIVE, CONVERGED_COST, CONVERGED_STEP, MAX_ITER, STALLED, INVALID = range(6)
STATUS_NAMES = ("ACTIVE", "CONVERGED_COST", "CONVERGED_STEP", "MAX_ITER", "STALLED", "INVALID")
MAX_VARY = 16
LAMBDA0 = 1e-3
COLUMNS = {"R_TOC": 0, "R_TOA": 1, "L_TOA": 2}
# defaults, chosen from a measured run (DESIGN.md §8)
FTOL, XTOL, MAX_ITERATIONS = 1e-12, 1e-10, 50


def layout(P):
    """Row offsets of the state array [rows][n_tracks] of spart_invert_*: u [P], trial [P], J^T W J [P (P + 1) / 2]
    (lower triangle, (i, j <= i) at i (i + 1) / 2 + j), J^T W r [P], C, lambda, status, forward calls."""
    na = P * (P + 1) // 2
    return dict(u=0, trial=P, A=2 * P, g=2 * P + na, C=3 * P + na, lam=3 * P + na + 1, status=3 * P + na + 2,
                calls=3 * P + na + 3, rows=3 * P + na + 4)


@dataclass
class InversionResult:
    """Per observation (tensors on the device of `obs`): x [m, P] float64, the best parameters in the order of
    `names`; cost [m] float64, sum_b w_b (f_b(x) - y_b)^2; std [m, P] float64, the standard deviations from
    (J^T W J)^-1 at x (scaled by cost / (nb - P) unless absolute_sigma); status [m] int32 (STATUS_NAMES); start [m]
    int32, the winning start (-1: none); iterations [m] int32, the forward calls of the winning track; n_forward
    [m] int64, the forward runs spent on the observation over all its starts."""
    names: tuple
    x: torch.Tensor
    cost: torch.Tensor
    std: torch.Tensor
    status: torch.Tensor
    start: torch.Tensor
    iterations: torch.Tensor
    n_forward: torch.Tensor


@dataclass
class Problem:
    """The constants of one chunk of observations, handed to `design`, `step` and `finish`: the box (rows, lo, hi),
    base [27] (the fixed rows), obs_rows / obs_values [len(obs_rows), mc] (rows given per observation, a view with
    any row stride), obs [mc, nb], weights [nb] or None, n_starts, column (0..2), ftol, xtol, max_iter,
    absolute_sigma, and bcast_mask (the broadcast rows of the forward call)."""
    rows: np.ndarray
    lo: np.ndarray
    hi: np.ndarray
    base: np.ndarray
    obs_rows: np.ndarray
    obs_values: torch.Tensor
    obs: torch.Tensor
    weights: object
    n_starts: int
    column: int
    ftol: float
    xtol: float
    max_iter: int
    absolute_sigma: bool
    bcast_mask: int

    @property
    def P(self):
        return len(self.rows)

    @property
    def n_tracks(self):
        return self.obs.shape[0] * self.n_starts


def init_state(prob, start):
    """The state array [rows][mc * S] of a chunk from its starts [mc, S, P] (x units): trial = start clipped into
    the box in u, C = NaN, lambda = 1e-3, status ACTIVE (INVALID for a start that is not finite), no calls."""
    P, lay = prob.P, layout(prob.P)
    lo = torch.as_tensor(prob.lo, dtype=torch.float64, device=start.device)
    hi = torch.as_tensor(prob.hi, dtype=torch.float64, device=start.device)
    x = start.reshape(-1, P)
    u = ((x - lo) / (hi - lo)).clamp(0.0, 1.0)
    state = torch.zeros((lay["rows"], x.shape[0]), dtype=torch.float64, device=start.device)
    state[lay["trial"]:lay["trial"] + P] = u.T
    state[lay["C"]] = float("nan")
    state[lay["lam"]] = LAMBDA0
    state[lay["status"]] = torch.where(torch.isfinite(x).all(1), float(ACTIVE), float(INVALID))
    return state


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _design(prob, state, active, buf):
    """spart_invert_design into buf [27, >= n_active (P + 1)]; returns the batch view [27, n_active (P + 1)]."""
    lib = _lib.load()
    n = active.numel() * (prob.P + 1)
    ov = prob.obs_values
    with torch.cuda.device(state.device):
        _lib.check(lib.spart_invert_design(
            _lib.as_int32_ptr(prob.rows), _lib.as_double_ptr(prob.lo), _lib.as_double_ptr(prob.hi), prob.P,
            _lib.as_int32_ptr(prob.obs_rows), len(prob.obs_rows), ov.data_ptr() if ov.numel() else 0,
            ov.stride(0) if ov.numel() else 0, _lib.as_double_ptr(prob.base), prob.n_starts, state.data_ptr(),
            state.shape[1], active.data_ptr(), active.numel(), buf.data_ptr(), buf.stride(0), _stream(state)),
            "spart_invert_design")
    return buf[:, :n]


def _step(prob, f, state, active):
    """spart_invert_step on the forward outputs f [n_active (P + 1), nb, 3]; updates state in place."""
    lib = _lib.load()
    w = prob.weights
    with torch.cuda.device(state.device):
        _lib.check(lib.spart_invert_step(
            _lib.as_double_ptr(prob.lo), _lib.as_double_ptr(prob.hi), prob.P, prob.n_starts, f.data_ptr(),
            f.shape[1], prob.column, prob.obs.data_ptr(), 0 if w is None else w.data_ptr(), prob.ftol, prob.xtol,
            prob.max_iter, state.data_ptr(), state.shape[1], active.data_ptr(), active.numel(), _stream(state)),
            "spart_invert_step")


def _finish(prob, state):
    """spart_invert_finish: (x, cost, std, status, start, iterations, n_forward) of the chunk's observations."""
    lib = _lib.load()
    m, P, dev = prob.obs.shape[0], prob.P, state.device
    outs = [torch.empty((m, P), dtype=torch.float64, device=dev), torch.empty(m, dtype=torch.float64, device=dev),
            torch.empty((m, P), dtype=torch.float64, device=dev)]
    outs += [torch.empty(m, dtype=torch.int32, device=dev) for _ in range(3)]
    outs.append(torch.empty(m, dtype=torch.int64, device=dev))
    with torch.cuda.device(dev):
        _lib.check(lib.spart_invert_finish(
            _lib.as_double_ptr(prob.lo), _lib.as_double_ptr(prob.hi), P, prob.n_starts, prob.obs.shape[1],
            int(prob.absolute_sigma), state.data_ptr(), m, *(o.data_ptr() for o in outs), _stream(state)),
            "spart_invert_finish")
    return tuple(outs)


def _row_index(key, what):
    if isinstance(key, str) and key in ROW_NAMES:
        return ROW_NAMES.index(key)
    if isinstance(key, (int, np.integer)) and 0 <= int(key) < NPAR:
        return int(key)
    raise ValueError(f"{what}: unknown parameter row {key!r}")


def _empty(names, P, device):
    z = lambda shape, dt: torch.empty(shape, dtype=dt, device=device)
    return InversionResult(names, z((0, P), torch.float64), z(0, torch.float64), z((0, P), torch.float64),
                           z(0, torch.int32), z(0, torch.int32), z(0, torch.int32), z(0, torch.int64))


def invert(obs, sensor, space, start, column="R_TOC", weights=None, absolute_sigma=False, per_obs=None, ftol=FTOL,
           xtol=XTOL, max_iter=MAX_ITERATIONS, chunk=2 ** 16, precision="fp64", band_mode="interp",
           soil_spectrum=None, soil_library=None, lidf=None, group=None, design=None, forward=None, step=None,
           finish=None):
    """Fit the varied rows of `space` (1 <= P <= 16) to every observation by bounded Levenberg-Marquardt.

    obs: CUDA float64 [m, nb], the observed `column` ("R_TOC", "R_TOA" or "L_TOA") of `sensor`'s bands.
    start: [m, S, P] starts in x units (e.g. `starts(...)` from `lut.nearest_k`); starts outside the box are clipped
    into it, and a start that is not finite (a NO_ENTRY neighbour) is skipped.  weights: [nb] band weights >= 0
    (default 1); with absolute_sigma=True they are read as 1 / sigma_b^2 and the covariance is not scaled by
    cost / (nb - P).  per_obs: {row name or index: [m] values} for rows given per observation (e.g. sun and view
    angles, aot550, or the soil-library index in row 9); the other fixed rows are `space.base` and go in as
    broadcast rows.  ftol, xtol, max_iter: the stop tests (DESIGN.md §8).  Tracks are iterated chunk by chunk,
    `chunk` tracks (whole observations, at least one) at a time, so device memory stays bounded.
    band_mode, soil_spectrum, soil_library: as in `Engine.forward_bands`.  Returns an InversionResult.
    Each observation's result is bit-identical whatever the other observations, the chunk size or the stream.
    Refused: precision "fp32" (forward differences need FP64), lidf=, a varied row 9 with soil_library, and
    per-observation LIDFa / LIDFb values for which the box would allow |LIDFa| + |LIDFb| > 1.
    With `group` (torch.distributed), each rank takes a contiguous slice of the observations and one all-gather
    returns the whole result on every rank.  `design` (prob, state, active -> batch [27, n]), `forward` (batch ->
    [n, nb, 3]), `step` (prob, f, state, active) and `finish` (prob, state -> the seven result tensors) default to
    the CUDA library; CPU tests inject stand-ins."""
    # every argument check comes before the first collective and the first GPU call
    if precision != "fp64":
        raise ValueError("invert: precision must be 'fp64' (forward-difference Jacobians need FP64)")
    if lidf is not None:
        raise ValueError("invert: lidf= is not supported (the leaf angles follow LIDFa / LIDFb)")
    if not isinstance(space, ParameterSpace):
        raise ValueError("invert: space must be a ParameterSpace")
    P = space.d
    if P > MAX_VARY:
        raise ValueError("invert: at most 16 varied rows")
    if soil_library is not None and 9 in space.rows:
        raise ValueError("invert: row 9 is the soil-library index with soil_library; it cannot be varied")
    if column not in COLUMNS:
        raise ValueError("invert: column must be 'R_TOC', 'R_TOA' or 'L_TOA'")
    if band_mode not in ("interp", "srf"):
        raise ValueError("invert: band_mode must be 'interp' or 'srf'")
    if not (isinstance(obs, torch.Tensor) and obs.dim() == 2 and obs.dtype == torch.float64):
        raise ValueError("invert: obs must be a float64 tensor [m, nb]")
    m, nb = obs.shape
    dev = obs.device
    start = torch.as_tensor(start, dtype=torch.float64).to(dev)
    if start.dim() != 3 or start.shape[0] != m or start.shape[2] != P or start.shape[1] < 1:
        raise ValueError("invert: start must be [m, S, P] with S >= 1")
    S = start.shape[1]
    if weights is not None:
        weights = torch.as_tensor(weights, dtype=torch.float64).to(dev).reshape(-1).contiguous()
        if weights.shape[0] != nb or not bool((torch.isfinite(weights) & (weights >= 0)).all()):
            raise ValueError("invert: weights must be [nb] finite values >= 0")
    if not (0 <= ftol < np.inf and 0 <= xtol < np.inf and int(max_iter) >= 1 and int(chunk) >= 1):
        raise ValueError("invert: need finite ftol, xtol >= 0, max_iter >= 1 and chunk >= 1")
    obs_rows, obs_cols = [], []
    for key, vals in (per_obs or {}).items():
        r = _row_index(key, "invert: per_obs")
        if r in space.rows or r in obs_rows:
            raise ValueError(f"invert: per_obs row {ROW_NAMES[r]} is varied or given twice")
        v = torch.as_tensor(vals, dtype=torch.float64).reshape(-1)
        if v.shape[0] != m:
            raise ValueError(f"invert: per_obs row {ROW_NAMES[r]} needs one value per observation ({m})")
        obs_rows.append(r)
        obs_cols.append(v)
    if LIDFA in obs_rows or LIDFB in obs_rows:
        rows = list(space.rows)

        def max_abs(row):
            if row in obs_rows:
                return obs_cols[obs_rows.index(row)].abs().cpu().numpy()
            if row in rows:
                return max(abs(space.lo[rows.index(row)]), abs(space.hi[rows.index(row)]))
            return abs(space.base[row])
        if (max_abs(LIDFA) + max_abs(LIDFB) > 1.0).any():
            raise ValueError("invert: per-observation LIDFa / LIDFb: the box must keep |LIDFa| + |LIDFb| <= 1 for "
                             "every observation (the reference's domain)")
    defaults = design is None or step is None or finish is None
    if defaults and not obs.is_cuda:
        raise ValueError("invert: obs must be a CUDA tensor")

    r0, r1 = 0, m
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        r0, r1 = m * rank // world, m * (rank + 1) // world
    # the rows may arrive on different devices (host arrays and CUDA tensors mixed): each is moved to `dev`
    obs_values = (torch.stack([c.to(dev) for c in obs_cols]) if obs_cols
                  else torch.empty((0, m), dtype=torch.float64, device=dev))
    obs_rows = np.asarray(obs_rows, dtype=np.int32)
    bcast = sum(1 << r for r in range(NPAR) if r not in space.rows and r not in obs_rows)
    mc = max(1, int(chunk) // S)
    buf = {}
    if design is None:
        def design(prob, state, active):
            n = prob.n_tracks * (P + 1)
            if "b" not in buf or buf["b"].shape[1] < n:
                buf["b"] = torch.empty((NPAR, n), dtype=torch.float64, device=dev)
            return _design(prob, state, active, buf["b"])
    if forward is None:
        eng = default_engine()
        forward = lambda p: eng.forward_bands(p, sensor, band_mode=band_mode, soil_spectrum=soil_spectrum,
                                              soil_library=soil_library, broadcast_rows=bcast)
    step, finish = step or _step, finish or _finish
    obs_c = obs.contiguous()
    parts = []
    for o0 in range(r0, r1, mc):
        o1 = min(o0 + mc, r1)
        prob = Problem(space.rows, space.lo, space.hi, space.base, obs_rows, obs_values[:, o0:o1], obs_c[o0:o1],
                       weights, S, COLUMNS[column], float(ftol), float(xtol), int(max_iter), bool(absolute_sigma),
                       bcast)
        state = init_state(prob, start[o0:o1])
        status = state[layout(P)["status"]]
        while True:
            active = torch.nonzero(status == ACTIVE).reshape(-1).to(torch.int32)     # the one sync per iteration
            if active.numel() == 0:
                break
            step(prob, forward(design(prob, state, active)), state, active)
        parts.append(finish(prob, state))
    if parts:
        local = [torch.cat([p[i] for p in parts]) for i in range(7)]
    else:
        e = _empty(space.names, P, dev)
        local = [e.x, e.cost, e.std, e.status, e.start, e.iterations, e.n_forward]
    if group is not None:
        local = _all_gather(local, m, P, group)
    return InversionResult(space.names, *local)


def _all_gather(local, m, P, group):
    """One all-gather of the ranks' results, packed as float64 [rows, 2 P + 5] (every field is exact in float64)
    and padded to the largest slice."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    sizes = [m * (r + 1) // world - m * r // world for r in range(world)]
    x, cost, std, status, start, iters, nfwd = local
    dev = x.device
    pack = torch.cat([x, std, cost[:, None], status[:, None].double(), start[:, None].double(),
                      iters[:, None].double(), nfwd[:, None].double()], dim=1)
    width = 2 * P + 5
    padded = torch.full((max(sizes), width), float("nan"), dtype=torch.float64, device=dev)
    padded[:pack.shape[0]] = pack
    lists = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(lists, padded, group=group)
    allp = torch.cat([l[:s] for l, s in zip(lists, sizes)])
    return [allp[:, :P].contiguous(), allp[:, 2 * P].contiguous(), allp[:, P:2 * P].contiguous(),
            allp[:, 2 * P + 1].to(torch.int32), allp[:, 2 * P + 2].to(torch.int32), allp[:, 2 * P + 3].to(torch.int32),
            allp[:, 2 * P + 4].to(torch.int64)]


def starts(table_params, index, space, index_offset=None, group=None):
    """Starts [m, k, P] (float64, x units, on the device of `index`) for `invert` from neighbour indices `index`
    [m, k] (int64, e.g. `lut.nearest_k`'s): the varied rows of `space` of each entry.  table_params: the parameter
    table of the LUT, or of this rank's slice of it, as a [27, n] batch or the transposed view `table.T` of an
    [n, 27] table such as the `params` of a `lut.generate` .npz; float64 or float32.  NO_ENTRY and indices outside
    the table become NaN, which `invert` skips.
    With `group` the table is sharded over its ranks as for `lut.estimate` (rank order = table order, every rank
    passes the same `index`): each rank fills the entries it holds and one SUM all-reduce of the m k P values and
    an m k found-mask assembles the starts on every rank.  index_offset (default: found from the slice sizes with
    `group`, else 0) is the first global entry of this rank's slice."""
    if not (isinstance(space, ParameterSpace) and isinstance(index, torch.Tensor) and index.dim() == 2):
        raise ValueError("starts: need a ParameterSpace and an index tensor [m, k]")
    tp = torch.as_tensor(table_params)
    if tp.dim() != 2 or tp.shape[0] != NPAR:
        raise ValueError("starts: table_params must be [27, n] (or the view .T of an [n, 27] table)")
    if index_offset is None:
        if group is None:
            index_offset = 0
        else:
            from .lut import _table_offset
            index_offset = _table_offset(tp.shape[1], group, "starts")
    dev = index.device
    idx = index.to(torch.int64) - int(index_offset)
    found = (index != NO_ENTRY) & (idx >= 0) & (idx < tp.shape[1])
    rows = torch.as_tensor(space.rows.astype(np.int64), device=tp.device)
    sel = tp.index_select(0, rows).to(dev, torch.float64)                       # [P, n]
    if sel.shape[1] == 0:                                                        # a rank without entries
        sel = torch.zeros((space.d, 1), dtype=torch.float64, device=dev)
    vals = sel[:, torch.where(found, idx, 0).reshape(-1)].T.reshape(*index.shape, space.d)
    if group is not None:
        import torch.distributed as dist
        vals = torch.where(found[..., None], vals, 0.0)
        both = torch.cat([vals.reshape(-1), found.reshape(-1).to(torch.float64)])
        dist.all_reduce(both, op=dist.ReduceOp.SUM, group=group)
        vals = both[:vals.numel()].reshape(vals.shape)
        found = both[vals.numel():].reshape(found.shape) > 0
    return torch.where(found[..., None], vals, float("nan"))
