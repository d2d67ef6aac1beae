"""Variance-based global sensitivity analysis on the GPU: which parameters drive which band output.

`ParameterSpace` names the varied rows of a parameter batch and their ranges (uniform); `sample` is a scrambled
Sobol' design of the space (a quasi-random LUT design for `lut.generate`), `design` the Saltelli design of
N (d + 2) samples, and `sobol` the first-order and total Sobol' indices of every band output, with the design,
the forward model and the estimator all on the device (spart_sobol_design, spart_forward_bands,
spart_sobol_accumulate / spart_sobol_finish).  The estimators are those of scipy.stats.sobol_indices with
method "saltelli_2010" (which centres the outputs on their mean):
  V = population variance of f_A and f_B together,  S_i = mean(t) / V with t = (f_B - mean) (f_ABi - f_A),
  ST_i = mean(u) / (2 V) with u = (f_A - f_ABi)^2,
with standard errors std(t) / (sqrt(N) V) and std(u) / (2 sqrt(N) V) that ignore the uncertainty of V.
`indices` runs the estimator on outputs a caller computed, for example a vegetation index.
"""
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .engine import default_engine

ROW_NAMES = ("Cab", "Cdm", "Cw", "Cs", "Cca", "Cant", "N", "PROT", "CBC", "B", "lat", "lon", "SMp", "SMC", "film",
             "LAI", "LIDFa", "LIDFb", "q", "sol_angle", "obs_angle", "rel_angle", "aot550", "uo3", "uh2o", "Pa", "DOY")
NPAR = len(ROW_NAMES)
LIDFA, LIDFB = 16, 17
MAX_POINTS = 2 ** 32


class ParameterSpace:
    """A box of parameter space: `base` [27] (or the [27, 1] column of `pack_params`) holds the values of the fixed
    rows, `vary` maps row names (see ROW_NAMES) or row indices to ranges (lo, hi), sampled uniformly in [lo, hi).
    The order of `vary` is the order of the varied parameters in every result.  Refused: unknown names, a row named
    twice, non-finite bounds or lo >= hi, no or more than 27 varied rows, and a leaf-angle box the reference does
    not accept: max |LIDFa| + max |LIDFb| <= 1 over the ranges and fixed values."""

    def __init__(self, base, vary):
        if isinstance(base, torch.Tensor):
            base = base.detach().cpu().numpy()
        base = np.asarray(base, dtype=np.float64).reshape(-1)
        if base.shape != (NPAR,):
            raise ValueError("base must hold the 27 parameter rows ([27] or a [27, 1] column)")
        vary = dict(vary)
        if not 1 <= len(vary) <= NPAR:
            raise ValueError("vary must name 1 to 27 rows")
        rows, lo, hi = [], [], []
        for key, rng in vary.items():
            if isinstance(key, str):
                if key not in ROW_NAMES:
                    raise ValueError(f"unknown parameter row {key!r}; rows are {', '.join(ROW_NAMES)}")
                r = ROW_NAMES.index(key)
            elif isinstance(key, (int, np.integer)) and 0 <= int(key) < NPAR:
                r = int(key)
            else:
                raise ValueError(f"unknown parameter row {key!r}: row indices are 0..26")
            if r in rows:
                raise ValueError(f"parameter row {ROW_NAMES[r]} is varied twice")
            a, b = (float(x) for x in rng)
            if not (np.isfinite(a) and np.isfinite(b) and a < b):
                raise ValueError(f"{ROW_NAMES[r]}: need finite lo < hi, got ({a}, {b})")
            rows.append(r)
            lo.append(a)
            hi.append(b)
        self.base = base
        self._base_dev = {}
        self.rows = np.asarray(rows, dtype=np.int32)
        self.lo = np.asarray(lo, dtype=np.float64)
        self.hi = np.asarray(hi, dtype=np.float64)
        fixed = [r for r in range(NPAR) if r not in rows]
        if not np.isfinite(base[fixed]).all():
            raise ValueError("the fixed rows of base must be finite")

        def max_abs(r):
            return max(abs(self.lo[rows.index(r)]), abs(self.hi[rows.index(r)])) if r in rows else abs(base[r])
        if max_abs(LIDFA) + max_abs(LIDFB) > 1.0:
            raise ValueError("LIDFa / LIDFb: the box must keep |LIDFa| + |LIDFb| <= 1 (the reference's domain)")

    @property
    def d(self):
        return len(self.rows)

    @property
    def names(self):
        return tuple(ROW_NAMES[r] for r in self.rows)

    @property
    def broadcast_rows(self):
        """Bit mask of the fixed rows, for `broadcast_rows=` of the forward entry points."""
        return sum(1 << r for r in range(NPAR) if r not in self.rows)

    def _fixed(self):
        return [r for r in range(NPAR) if r not in self.rows]

    def _write(self, out, count, seed, first, scramble, saltelli):
        if not (isinstance(seed, (int, np.integer)) and 0 <= int(seed) < 2 ** 64):
            raise ValueError("seed must be an integer in [0, 2^64)")
        lib = _lib.load()
        with torch.cuda.device(out.device):
            stream = torch.cuda.current_stream(out.device).cuda_stream
            _lib.check(lib.spart_sobol_design(_lib.as_int32_ptr(self.rows), _lib.as_double_ptr(self.lo),
                                              _lib.as_double_ptr(self.hi), self.d, int(seed), int(bool(scramble)),
                                              int(first), int(count), int(saltelli),
                                              out.data_ptr() if out.numel() else 0, out.stride(0), stream),
                       "spart_sobol_design")
        return out

    def sample(self, n, seed=0, first=0, scramble=True, device=None):
        """Points first .. first + n - 1 of the (scrambled, with `seed`) Sobol' sequence of the space as a CUDA
        float64 batch [27, n] with every row filled: a quasi-random design for `lut.generate` or
        `run_batch_params(..., broadcast_rows=space.broadcast_rows)`.  first + n <= 2^32; any index range can be
        produced on its own (e.g. one per GPU)."""
        dev = torch.device(device) if device is not None else default_engine().device
        out = torch.empty((NPAR, int(n)), dtype=torch.float64, device=dev)
        fixed = self._fixed()
        out[fixed] = torch.from_numpy(self.base[fixed]).to(dev)[:, None]
        return self._write(out, n, seed, first, scramble, saltelli=0)

    def design(self, count, seed=0, first=0, device=None):
        """The Saltelli design of base points first .. first + count - 1 (count >= 1): a CUDA float64 batch
        [27, (d + 2) count] of blocks A, B, AB_1 .. AB_d of `count` samples (sample block * count + j).  A is
        `sample(count, seed, first)`'s varied rows, B uses Sobol' dimensions d .. 2d - 1 and AB_i is A with varied
        parameter i from B.  The fixed rows are set at element 0 only: pass `broadcast_rows=space.broadcast_rows`
        (fixed sun / view angles then select the folded-geometry kernels)."""
        if count < 1:
            raise ValueError("design: need count >= 1")
        dev = torch.device(device) if device is not None else default_engine().device
        out = torch.empty((NPAR, (self.d + 2) * int(count)), dtype=torch.float64, device=dev)
        if dev not in self._base_dev:      # one host-to-device copy per device, not one per chunk
            self._base_dev[dev] = torch.from_numpy(self.base).to(dev)
        out[:, 0] = self._base_dev[dev]
        return self._write(out, count, seed, first, True, saltelli=1)


@dataclass
class SobolResult:
    """Host NumPy results.  names: the varied parameters (d); mean, var: mean and population variance of each
    output over f_A and f_B; first, total: S_i and ST_i; first_se, total_se: their standard errors (ignoring the
    uncertainty of var); n: base points.  Shapes: [nb, 3] and [nb, 3, d] from `sobol` (columns R_TOC, R_TOA,
    L_TOA), [s] and [s, d] from `indices`."""
    names: tuple
    mean: np.ndarray
    var: np.ndarray
    first: np.ndarray
    total: np.ndarray
    first_se: np.ndarray
    total_se: np.ndarray
    n: int


def _accumulate(f, n, n_vary, ref, acc):
    """spart_sobol_accumulate: f [(n_vary + 2) n, n_out] (any shape with that element order), ref [n_vary + 2,
    n_out], acc from _new_acc."""
    lib = _lib.load()
    n_out = ref.shape[-1]
    if not (f.is_cuda and f.dtype == torch.float64 and f.is_contiguous() and f.numel() == (n_vary + 2) * n * n_out):
        raise ValueError("outputs must be a contiguous CUDA float64 tensor of (d + 2) * n * n_out elements")
    with torch.cuda.device(f.device):
        stream = torch.cuda.current_stream(f.device).cuda_stream
        _lib.check(lib.spart_sobol_accumulate(f.data_ptr(), n, n_out, n_vary, ref.data_ptr(), acc.data_ptr(), stream),
                   "spart_sobol_accumulate")


def _finish(acc, ref, n_total, n_vary):
    """spart_sobol_finish: (mean [n_out], var [n_out], first, total, first_se, total_se [n_out, n_vary])."""
    lib = _lib.load()
    n_out = ref.shape[-1]
    outs = [torch.empty(n_out, dtype=torch.float64, device=acc.device) for _ in range(2)]
    outs += [torch.empty((n_out, n_vary), dtype=torch.float64, device=acc.device) for _ in range(4)]
    with torch.cuda.device(acc.device):
        stream = torch.cuda.current_stream(acc.device).cuda_stream
        _lib.check(lib.spart_sobol_finish(acc.data_ptr(), ref.data_ptr(), int(n_total), n_out, n_vary,
                                          *(o.data_ptr() for o in outs), stream), "spart_sobol_finish")
    return outs


def _new_acc(n_out, n_vary, device):
    return torch.zeros(_lib.load().spart_sobol_acc_elems(n_out, n_vary), dtype=torch.float64, device=device)


def sobol(space, sensor, n, seed=0, chunk=2 ** 15, precision="fp64", band_mode="interp", soil_spectrum=None,
          group=None, soil_library=None, design=None, forward=None, accumulate=None, finish=None):
    """First-order and total Sobol' indices of every band output (R_TOC, R_TOA, L_TOA of each band of `sensor`)
    with respect to the varied parameters of `space`, from N = n base points (n (d + 2) forward runs) of the
    scrambled design `space.design(..., seed)`.  Runs design -> Engine.forward_bands -> accumulate chunk by chunk
    (`chunk` base points, (d + 2) chunk samples, at a time) on the current stream and returns a SobolResult.
    Every sum is FP64 in a fixed order, so the same arguments give the same bits; results for different `chunk`
    agree to rounding.
    With `group` (torch.distributed), each rank takes a contiguous range of base points, evaluates base point 0
    itself for the shift, and the ranks sum their accumulators with one all-reduce; every rank returns the result.
    soil_library is not supported (a discrete parameter).  `design` (space, count, seed, first -> [27, (d+2)
    count]), `forward` (params -> [samples, nb, 3]), `accumulate` (f, n, d, ref, acc) and `finish` (acc, ref,
    n_total, d -> mean, var, first, total, first_se, total_se) default to the CUDA library; CPU tests inject
    stand-ins."""
    # every argument check comes before the first collective: no rank may wait for ranks that refused
    if soil_library is not None:
        raise ValueError("sobol: soil_library is not supported (a soil index is a discrete parameter)")
    if not isinstance(space, ParameterSpace):
        raise ValueError("sobol: space must be a ParameterSpace")
    if not 1 <= n <= MAX_POINTS:
        raise ValueError("sobol: need 1 <= n <= 2^32 base points")
    if chunk < 1:
        raise ValueError("sobol: need chunk >= 1")
    if precision not in ("fp64", "fp32") or band_mode not in ("interp", "srf"):
        raise ValueError("sobol: precision is 'fp64' or 'fp32', band_mode 'interp' or 'srf'")
    if not (isinstance(seed, (int, np.integer)) and 0 <= int(seed) < 2 ** 64):
        raise ValueError("sobol: seed must be an integer in [0, 2^64)")
    d = space.d
    design = design or (lambda sp, count, sd, first: sp.design(count, seed=sd, first=first))
    if forward is None:
        eng = default_engine()
        forward = lambda p: eng.forward_bands(p, sensor, precision=precision, band_mode=band_mode,
                                              soil_spectrum=soil_spectrum, broadcast_rows=space.broadcast_rows)
    accumulate, finish = accumulate or _accumulate, finish or _finish
    j0, j1 = 0, n
    if group is not None:
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        j0, j1 = n * rank // world, n * (rank + 1) // world
    f_ref = forward(design(space, 1, seed, 0))
    nb = f_ref.shape[1]
    ref = f_ref.reshape(d + 2, -1)
    acc = _new_acc(ref.shape[1], d, ref.device)
    for c0 in range(j0, j1, chunk):
        m = min(chunk, j1 - c0)
        accumulate(forward(design(space, m, seed, c0)), m, d, ref, acc)
    if group is not None:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
    res = [t.cpu().numpy() for t in finish(acc, ref, n, d)]
    return SobolResult(space.names, res[0].reshape(nb, 3), res[1].reshape(nb, 3),
                       *(r.reshape(nb, 3, d) for r in res[2:]), n=int(n))


def indices(f_A, f_B, f_AB):
    """The estimator of `sobol` on outputs a caller computed (e.g. a vegetation index of `run_batch_params` outputs,
    or planes of `forward_spectrum` over a design): CUDA float64 arrays in the shapes of scipy.stats.sobol_indices'
    dict input, f_A, f_B [s, N] and f_AB [d, s, N] (d <= 27), base point 0 serving as the shift.  Returns a
    SobolResult with mean, var [s] and first, total, first_se, total_se [s, d] (names: 0 .. d - 1)."""
    if not all(isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64 for t in (f_A, f_B, f_AB)):
        raise ValueError("indices: f_A, f_B, f_AB must be CUDA float64 tensors")
    if not (f_A.dim() == 2 and f_B.shape == f_A.shape and f_AB.dim() == 3 and f_AB.shape[1:] == f_A.shape
            and f_A.shape[1] >= 1 and 1 <= f_AB.shape[0] <= NPAR and f_A.shape[0] >= 1):
        raise ValueError("indices: need f_A, f_B [s, N] and f_AB [d, s, N] with 1 <= d <= 27, N, s >= 1")
    d, (s, n) = f_AB.shape[0], f_A.shape
    f = torch.cat([f_A[None], f_B[None], f_AB]).transpose(1, 2).contiguous()       # [(d + 2), N, s]
    ref = f[:, 0, :].contiguous()
    acc = _new_acc(s, d, f.device)
    _accumulate(f, n, d, ref, acc)
    res = [t.cpu().numpy() for t in _finish(acc, ref, n, d)]
    return SobolResult(tuple(range(d)), *res, n=int(n))
