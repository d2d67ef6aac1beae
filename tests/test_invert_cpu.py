"""CPU checks of the retrieval by bounded Levenberg-Marquardt: the kernels restated in NumPy (`init_np`,
`design_np`, `step_np`, `finish_np`; the GPU tests import them as their reference), driven by the oracle to recover
noise-free Sentinel-2A observations; the forward-difference Jacobian against central differences; every refusal of
`invert` before any GPU call; the C-ABI symbols; and `invert(group=)` / `starts(group=)` over gloo at world size 2
with stand-ins for the kernels."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

sys.path.insert(0, str(ROOT / "spart-python_b200"))

from spart_b200 import inversion  # noqa: E402
from spart_b200.inversion import (ACTIVE, CONVERGED_COST, CONVERGED_STEP, INVALID, MAX_ITER, STALLED,  # noqa: E402
                                  layout)
from spart_b200.sensitivity import NPAR, ParameterSpace  # noqa: E402

S2A = "Sentinel2A-MSI"
H = 2.0 ** -17
BASE = np.array([40, 0.01, 0.02, 0.1, 10, 1, 1.5, 0, 0, 0.5, 10, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                 40, 0, 0, 0.3, 0.35, 1.5, 1013, 180], dtype=np.float64)
VARY6 = {"Cab": (5, 80), "Cw": (0.005, 0.05), "Cdm": (0.002, 0.02), "N": (1, 3), "LAI": (0.1, 8), "SMp": (5, 55)}
VARY7 = dict(VARY6, LIDFa=(-0.5, 0.5))


def tri(i):
    return i * (i + 1) // 2


# ---- the kernels restated in NumPy -------------------------------------------------------------------------------

def x_of(lo, hi, u):
    """x = lo + (hi - lo) u, each operation rounded once (the kernels use no FMA here)."""
    return lo + (hi - lo) * u


def moved(u):
    """u_p of sample p + 1: u + h if that is <= 1, else u - h."""
    up = u + H
    return np.where(up <= 1.0, up, u - H)


def init_np(lo, hi, start):
    """inversion.init_state: state [rows, T] from starts [.., P] in x units."""
    P = len(lo)
    lay = layout(P)
    x = np.asarray(start, dtype=np.float64).reshape(-1, P)
    with np.errstate(invalid="ignore"):
        u = np.clip((x - lo) / (hi - lo), 0.0, 1.0)
    state = np.zeros((lay["rows"], x.shape[0]))
    state[lay["trial"]:lay["trial"] + P] = u.T
    state[lay["C"]] = np.nan
    state[lay["lam"]] = 1e-3
    state[lay["status"]] = np.where(np.isfinite(x).all(1), ACTIVE, INVALID)
    return state


def design_np(rows, lo, hi, base, obs_rows, obs_values, n_starts, state, active, out):
    """invert_design_kernel: writes the P + 1 samples of each active track into out [27, >= n (P + 1)]; the rows
    neither varied nor given per observation only at element 0."""
    P = len(rows)
    t = np.asarray(active, dtype=np.int64)
    trial = state[P:2 * P][:, t]
    o = t // n_starts
    for s in range(P + 1):
        cols = np.arange(len(t)) * (P + 1) + s
        for p in range(P):
            u = moved(trial[p]) if s == p + 1 else trial[p]
            out[rows[p], cols] = x_of(lo[p], hi[p], u)
        for k, r in enumerate(obs_rows):
            out[r, cols] = obs_values[k][o]
    if len(t):
        for r in range(NPAR):
            if r not in rows and r not in obs_rows:
                out[r, 0] = base[r]
    return out


def cholesky_np(A, lam):
    """Packed lower Cholesky factor of A + lam diag(max(A_pp, 1e-30)) (lam None: of A) per column of A [NA, n];
    returns (L, ok) with ok False where a pivot is not > 0."""
    na, n = A.shape
    P = int(round((np.sqrt(8 * na + 1) - 1) / 2))
    L = np.zeros_like(A)
    ok = np.ones(n, dtype=bool)
    with np.errstate(invalid="ignore", divide="ignore"):
        for j in range(P):
            jj = tri(j)
            ajj = A[jj + j]
            s = ajj + lam * np.fmax(ajj, 1e-30) if lam is not None else ajj.copy()
            for k in range(j):
                s = s - L[jj + k] * L[jj + k]
            ok &= s > 0
            d = np.sqrt(np.where(s > 0, s, 1.0))
            L[jj + j] = d
            for i in range(j + 1, P):
                ii = tri(i)
                v = A[ii + j].copy()
                for k in range(j):
                    v = v - L[ii + k] * L[jj + k]
                L[ii + j] = v / d
    return L, ok


def step_np(lo, hi, n_starts, f, column, obs, weights, ftol, xtol, max_iter, state, active):
    """invert_step_kernel on the forward outputs f [n (P + 1), nb, 3] of a design_np batch; updates state."""
    P = len(lo)
    lay = layout(P)
    NA = tri(P)
    t = np.asarray(active, dtype=np.int64)
    n = len(t)
    nb = f.shape[1]
    w = np.ones(nb) if weights is None else np.asarray(weights, dtype=np.float64)
    calls = state[lay["calls"], t] + 1
    state[lay["calls"], t] = calls
    f0 = f[np.arange(n) * (P + 1), :, column]
    y = obs[t // n_starts]
    c = np.zeros(n)
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(nb):
            d = f0[:, b] - y[:, b]
            c = c + w[b] * (d * d)
    first = calls == 1
    invalid = first & ~(np.isfinite(y).all(1) & np.isfinite(c))
    live = ~invalid
    c_old = state[lay["C"], t]
    lam = state[lay["lam"], t].copy()
    with np.errstate(invalid="ignore"):
        acc = live & (first | (c < c_old))
    ia = np.nonzero(acc)[0]
    ta = t[ia]
    utr = state[lay["trial"]:lay["trial"] + P][:, ta]
    state[lay["u"]:lay["u"] + P, ta] = utr
    du = (x_of(lo[:, None], hi[:, None], moved(utr)) - x_of(lo[:, None], hi[:, None], utr)) / (hi - lo)[:, None]
    A = np.zeros((NA, len(ia)))
    g = np.zeros((P, len(ia)))
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(nb):
            fb = f0[ia, b]
            d = fb - y[ia, b]
            J = [(f[ia * (P + 1) + p + 1, b, column] - fb) / du[p] for p in range(P)]
            for i in range(P):
                wj = w[b] * J[i]
                g[i] = g[i] + wj * d
                for j in range(i + 1):
                    A[tri(i) + j] = A[tri(i) + j] + wj * J[j]
    state[lay["A"]:lay["A"] + NA, ta] = A
    state[lay["g"]:lay["g"] + P, ta] = g
    state[lay["C"], ta] = c[ia]
    later = acc & ~first
    lam[later] = np.maximum(lam[later] / 10.0, 1e-15)
    with np.errstate(invalid="ignore"):
        conv_cost = later & (c_old - c <= ftol * c_old)
    rej = live & ~acc
    lam[rej] = lam[rej] * 10.0
    status = np.full(n, ACTIVE)
    status[invalid] = INVALID
    status[conv_cost] = CONVERGED_COST
    go = live & ~conv_cost
    stalled = go & (lam > 1e16)
    status[stalled] = STALLED
    maxit = go & ~stalled & (calls >= max_iter)
    status[maxit] = MAX_ITER
    pending = go & ~stalled & ~maxit
    L = np.zeros((NA, n))
    solved = np.zeros(n, dtype=bool)
    while pending.any():
        ip = np.nonzero(pending)[0]
        Lp, ok = cholesky_np(state[lay["A"]:lay["A"] + NA][:, t[ip]], lam[ip])
        L[:, ip[ok]] = Lp[:, ok]
        solved[ip[ok]] = True
        bad = ip[~ok]
        lam[bad] = lam[bad] * 10.0
        over = bad[lam[bad] > 1e16]
        status[over] = STALLED
        pending[ip[ok]] = False
        pending[over] = False
    i_s = np.nonzero(solved)[0]
    ts = t[i_s]
    Ls = L[:, i_s]
    gs = state[lay["g"]:lay["g"] + P][:, ts]
    z = np.zeros((P, len(i_s)))
    for i in range(P):
        v = -gs[i]
        for k in range(i):
            v = v - Ls[tri(i) + k] * z[k]
        z[i] = v / Ls[tri(i) + i]
    for i in range(P - 1, -1, -1):
        v = z[i].copy()
        for k in range(i + 1, P):
            v = v - Ls[tri(k) + i] * z[k]
        z[i] = v / Ls[tri(i) + i]
    u = state[lay["u"]:lay["u"] + P][:, ts]
    nxt = np.clip(u + z, 0.0, 1.0)
    state[lay["trial"]:lay["trial"] + P, ts] = nxt
    stepn = np.abs(nxt - u).max(0) if P else np.zeros(len(i_s))
    status[i_s[stepn <= xtol]] = CONVERGED_STEP
    state[lay["lam"], t[live]] = lam[live]
    state[lay["status"], t] = status


def finish_np(lo, hi, n_starts, nb, absolute_sigma, state):
    """invert_finish_kernel: (x, cost, std, status, start, iterations, n_forward) per observation."""
    P = len(lo)
    lay = layout(P)
    T = state.shape[1]
    m = T // n_starts
    C = state[lay["C"]].reshape(m, n_starts)
    calls = state[lay["calls"]].reshape(m, n_starts)
    n_forward = (calls * (P + 1)).sum(1).astype(np.int64)
    finite = np.isfinite(C)
    best = np.argmin(np.where(finite, C, np.inf), axis=1)          # ties to the lowest start
    any_ = finite.any(1)
    tb = np.arange(m) * n_starts + best
    x = x_of(lo[:, None], hi[:, None], state[lay["u"]:lay["u"] + P][:, tb]).T
    cost = C[np.arange(m), best]
    L, ok = cholesky_np(state[lay["A"]:lay["A"] + tri(P)][:, tb], None)
    var = np.zeros((P, m))
    with np.errstate(invalid="ignore", divide="ignore"):
        for p in range(P):
            z = {}
            for i in range(p, P):
                v = np.full(m, 1.0 if i == p else 0.0)
                for k in range(p, i):
                    v = v - L[tri(i) + k] * z[k]
                z[i] = v / L[tri(i) + i]
                var[p] = var[p] + z[i] * z[i]
        scale = np.ones(m) if absolute_sigma else (cost / (nb - P) if nb > P else np.full(m, np.nan))
        std = ((hi - lo)[:, None] * np.sqrt(scale * var)).T
    std[~ok] = np.nan
    status = state[lay["status"], tb].astype(np.int32)
    iters = calls[np.arange(m), best].astype(np.int32)
    start = best.astype(np.int32)
    x[~any_] = np.nan
    std[~any_] = np.nan
    cost = np.where(any_, cost, np.nan)
    status[~any_] = INVALID
    start[~any_] = -1
    iters[~any_] = 0
    return x, cost, std, status, start, iters, n_forward


def run_np(space, obs, start, forward, column=0, weights=None, obs_rows=(), obs_values=None, ftol=inversion.FTOL,
           xtol=inversion.XTOL, max_iter=inversion.MAX_ITERATIONS, absolute_sigma=False, return_state=False):
    """The whole retrieval with the NumPy kernels; forward(batch [27, n] with every row filled) -> [n, nb, 3]."""
    lo, hi = space.lo, space.hi
    P, (m, nb) = space.d, obs.shape
    S = start.shape[1]
    state = init_np(lo, hi, start)
    lay = layout(P)
    obs_values = np.zeros((0, m)) if obs_values is None else obs_values
    while True:
        active = np.nonzero(state[lay["status"]] == ACTIVE)[0]
        if not len(active):
            break
        out = np.full((NPAR, len(active) * (P + 1)), np.nan)
        design_np(space.rows, lo, hi, space.base, list(obs_rows), obs_values, S, state, active, out)
        bc = [r for r in range(NPAR) if r not in space.rows and r not in obs_rows]
        out[bc] = out[bc, :1]
        step_np(lo, hi, S, forward(out), column, obs, weights, ftol, xtol, max_iter, state, active)
    res = finish_np(lo, hi, S, nb, absolute_sigma, state)
    return (res, state) if return_state else res


# ---- recovery with the oracle ------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def oracle(optical):
    import spart_oracle
    return lambda params: spart_oracle.spart_bands(np.ascontiguousarray(params.T), S2A, optical)


def test_noise_free_recovery_with_the_oracle(oracle):
    space = ParameterSpace(BASE, VARY6)
    rng = np.random.default_rng(1)
    m, P = 16, space.d
    truth = rng.uniform(0.05, 0.95, (m, P))
    X = np.tile(BASE, (m, 1))
    X[:, space.rows] = space.lo + (space.hi - space.lo) * truth
    obs = oracle(X.T)[..., 0]
    u0 = np.clip(truth + rng.uniform(-0.15, 0.15, (m, P)), 0, 1)
    start = (space.lo + (space.hi - space.lo) * u0)[:, None, :]
    x, cost, std, status, st, iters, nfwd = run_np(space, obs, start, oracle)
    u = (x - space.lo) / (space.hi - space.lo)
    assert np.abs(u - truth).max() <= 1e-9, np.abs(u - truth).max(1)
    assert np.isin(status, (CONVERGED_COST, CONVERGED_STEP)).all(), status
    assert (st == 0).all() and (iters <= 50).all() and (nfwd == iters * (P + 1)).all()
    assert (cost <= 1e-20).all()


def test_forward_difference_jacobian_against_central_differences(oracle):
    """The step 2^-17 of the range against central differences (2^-10), LIDFa included: within 2e-4 relative to
    each column's largest value (the GPU test re-measures this on the kernels' own design)."""
    space = ParameterSpace(BASE, VARY7)
    rng = np.random.default_rng(2)
    P, n = space.d, 64
    U = rng.uniform(0.05, 0.95, (n, P))

    def F(U):
        X = np.tile(BASE, (U.shape[0], 1))
        X[:, space.rows] = x_of(space.lo, space.hi, U)
        return oracle(X.T)[..., 0]
    f0 = F(U)
    worst = []
    for p in range(P):
        Up, Uc1, Uc2 = U.copy(), U.copy(), U.copy()
        Up[:, p] = moved(U[:, p])
        du = (x_of(space.lo[p], space.hi[p], Up[:, p]) - x_of(space.lo[p], space.hi[p], U[:, p])) / (
            space.hi[p] - space.lo[p])
        fd = (F(Up) - f0) / du[:, None]
        hc = 2.0 ** -10
        Uc1[:, p] += hc
        Uc2[:, p] -= hc
        cd = (F(Uc1) - F(Uc2)) / (2 * hc)
        worst.append(np.abs(fd - cd).max() / np.abs(cd).max())
    assert max(worst) <= 2e-4, worst


def test_step_branches_on_crafted_state():
    """The reject branch and the Cholesky retry on an indefinite stored J^T W J, the accept branch, and the stop
    tests, with hand-made forward outputs (P = 2, 3 bands)."""
    lo, hi = np.array([0.0, 0.0]), np.array([1.0, 1.0])
    lay = layout(2)
    state = init_np(lo, hi, np.array([[0.5, 0.5], [0.25, 0.75]]))
    obs = np.array([[1.0, 2.0, 3.0], [1.0, 2.0, 3.0]])
    f = np.zeros((6, 3, 3))
    f[:, :, 0] = np.arange(1.0, 4.0) + 0.5
    f[[1, 4], :, 0] += np.array([1.0, 0.0, 0.0]) * 2.0 ** -17
    f[[2, 5], :, 0] += np.array([0.0, 1.0, 1.0]) * 2.0 ** -17
    step_np(lo, hi, 1, f, 0, obs, None, 1e-12, 1e-12, 50, state, np.array([0, 1]))
    assert (state[lay["status"]] == ACTIVE).all() and (state[lay["C"]] == 0.75).all()
    # reject: a worse trial; the stored matrix is made indefinite so the first two retries fail
    state[lay["A"]:lay["A"] + 3, 0] = [1.0, 3.0, 1.0]
    f[:, :, 0] += 10.0
    step_np(lo, hi, 1, f, 0, obs, None, 1e-12, 1e-12, 50, state, np.array([0]))
    # 1e-3 x 10 for the rejection, then x 10 after each of the failed factorisations at 1e-2, 1e-1 and 1
    assert state[lay["C"], 0] == 0.75 and state[lay["lam"], 0] == pytest.approx(10.0)
    assert state[lay["status"], 0] == ACTIVE
    # max_iter reached
    step_np(lo, hi, 1, f, 0, obs, None, 1e-12, 1e-12, 3, state, np.array([0]))
    assert state[lay["status"], 0] == MAX_ITER


# ---- refusals, symbols ---------------------------------------------------------------------------------------------

def _args(m=3, S=2, space=None):
    space = space or ParameterSpace(BASE, VARY6)
    return torch.zeros((m, 13), dtype=torch.float64), space, torch.zeros((m, S, space.d), dtype=torch.float64)


def _no_gpu(*a, **k):
    raise AssertionError("a GPU stand-in was called before the refusal")


@pytest.mark.parametrize("kwargs, match", [
    (dict(precision="fp32"), "fp64"),
    (dict(lidf=np.ones(13) / 13), "lidf"),
    (dict(column="R_TOX"), "column"),
    (dict(band_mode="nearest"), "band_mode"),
    (dict(weights=np.ones(12)), "weights"),
    (dict(weights=-np.ones(13)), "weights"),
    (dict(max_iter=0), "max_iter"),
    (dict(chunk=0), "chunk"),
    (dict(per_obs={"Cab": np.zeros(3)}), "varied"),
    (dict(per_obs={"sol_angle": np.zeros(2)}), "one value per observation"),
    (dict(per_obs={"nope": np.zeros(3)}), "unknown"),
    (dict(per_obs={"LIDFa": np.array([0.2, 0.9, 0.1])}), "LIDFa"),
])
def test_refusals_before_any_gpu_call(kwargs, match):
    obs, space, start = _args()
    with pytest.raises(ValueError, match=match):
        inversion.invert(obs, S2A, space, start, design=_no_gpu, forward=_no_gpu, step=_no_gpu, finish=_no_gpu,
                         **kwargs)


def test_structural_refusals():
    obs, space, start = _args()
    stub = dict(design=_no_gpu, forward=_no_gpu, step=_no_gpu, finish=_no_gpu)
    with pytest.raises(ValueError, match="row 9"):
        inversion.invert(obs, S2A, ParameterSpace(BASE, dict(VARY6, B=(0, 3))), torch.zeros((3, 2, 7)),
                         soil_library=object(), **stub)
    big = ParameterSpace(BASE, {n: (0.0, 1.0) for n in ("Cab", "Cdm", "Cw", "Cs", "Cca", "Cant", "N", "PROT", "CBC",
                                                        "B", "lat", "lon", "SMp", "SMC", "film", "LAI", "q")})
    with pytest.raises(ValueError, match="16"):
        inversion.invert(obs, S2A, big, torch.zeros((3, 2, 17)), **stub)
    with pytest.raises(ValueError, match="start"):
        inversion.invert(obs, S2A, space, start[:, :, :5], **stub)
    with pytest.raises(ValueError, match="CUDA"):
        inversion.invert(obs, S2A, space, start)
    # a per-observation LIDFb that stays inside the domain with the varied LIDFa box is accepted
    sp7 = ParameterSpace(BASE, VARY7)
    ok = inversion.invert(obs, S2A, sp7, torch.full((3, 1, 7), float("nan")),
                          per_obs={"LIDFb": np.array([0.1, -0.5, 0.0])}, design=_no_gpu, forward=_no_gpu,
                          step=_no_gpu, finish=lambda prob, state: finish_torch(prob, state))
    assert (ok.status == INVALID).all() and (ok.start == -1).all()


def test_exports_declare_the_invert_entry_points():
    from spart_b200 import _lib
    header = (ROOT / "include" / "spart_b200.h").read_text()
    lib = _lib.load()
    for sym in ("spart_invert_state_rows", "spart_invert_design", "spart_invert_step", "spart_invert_finish"):
        assert sym in _lib.EXPORTS and re.search(rf"\b{sym}\s*\(", header) and hasattr(lib, sym)
    assert lib.spart_invert_state_rows(7) == layout(7)["rows"] == 3 * 7 + 28 + 4
    assert lib.spart_invert_state_rows(0) == 0 and lib.spart_invert_state_rows(17) == 0


def test_c_abi_refuses_bad_arguments_without_a_device():
    """Argument checks come before any CUDA call, so they answer SPART_EINVAL on a machine without a GPU too."""
    from spart_b200 import _lib
    lib = _lib.load()
    rows = np.array([0, 2], dtype=np.int32)
    lo, hi, base = np.zeros(2), np.ones(2), BASE.copy()
    P = _lib.as_int32_ptr
    D = _lib.as_double_ptr
    obs_rows = np.array([2], dtype=np.int32)
    assert lib.spart_invert_design(P(rows), D(lo), D(hi), 2, P(obs_rows), 1, 8, 4, D(base), 1, 8, 4, 8, 4, 8, 12,
                                   None) == -1
    assert b"not varied" in lib.spart_last_error()
    assert lib.spart_invert_design(P(rows), D(lo), D(hi), 17, None, 0, 0, 0, D(base), 1, 8, 4, 8, 4, 8, 80, None) == -1
    assert lib.spart_invert_design(P(rows), D(lo), D(hi), 2, None, 0, 0, 0, D(base), 1, 8, 4, 0, 4, 8, 12, None) == -1
    assert lib.spart_invert_step(D(lo), D(hi), 2, 1, 8, 13, 3, 8, None, 1e-12, 1e-12, 50, 8, 4, 8, 4, None) == -1
    assert lib.spart_invert_step(D(lo), D(hi), 2, 0, 8, 13, 0, 8, None, 1e-12, 1e-12, 50, 8, 4, 8, 4, None) == -1
    assert lib.spart_invert_step(D(lo), D(hi), 2, 1, 8, 13, 0, 8, None, 1e-12, 1e-12, 50, 8, 4, None, 4, None) == -1
    assert lib.spart_invert_finish(D(lo), D(hi), 2, 1, 13, 2, 8, 4, *([8] * 7), None) == -1
    assert lib.spart_invert_finish(D(lo), D(hi), 2, 1, 13, 0, 8, 4, *([8] * 6), None, None) == -1
    assert lib.spart_invert_finish(D(hi), D(lo), 2, 1, 13, 0, 8, 4, *([8] * 7), None) == -1
    assert b"lo < hi" in lib.spart_last_error()


# ---- stand-ins for the kernels, on torch CPU tensors ---------------------------------------------------------------

def design_torch(prob, state, active):
    n = active.numel() * (prob.P + 1)
    out = np.full((NPAR, n), np.nan)
    design_np(prob.rows, prob.lo, prob.hi, prob.base, list(prob.obs_rows), prob.obs_values.numpy(), prob.n_starts,
              state.numpy(), active.numpy(), out)
    return torch.from_numpy(out)


def step_torch(prob, f, state, active):
    step_np(prob.lo, prob.hi, prob.n_starts, f.numpy(), prob.column, prob.obs.numpy(),
            None if prob.weights is None else prob.weights.numpy(), prob.ftol, prob.xtol, prob.max_iter,
            state.numpy(), active.numpy().astype(np.int64))


def finish_torch(prob, state):
    return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in
                 finish_np(prob.lo, prob.hi, prob.n_starts, prob.obs.shape[1], prob.absolute_sigma, state.numpy()))


TOY_ROWS = {"Cab": (0.0, 2.0), "LAI": (0.5, 3.0)}


def toy_forward(params):
    """A smooth stand-in of the forward model: 5 bands of the varied rows Cab, LAI and the per-observation row q."""
    a, l, q = params[0], params[15], params[18]
    k = torch.arange(1.0, 6.0, dtype=torch.float64)
    r = torch.sin(a[:, None] * k / 3) + l[:, None] * l[:, None] / k + q[:, None] * k / 10
    return torch.stack([r, 2 * r, 3 * r], dim=-1)


def _toy_problem():
    space = ParameterSpace(BASE, TOY_ROWS)
    rng = np.random.default_rng(5)
    m = 7
    truth = np.column_stack([rng.uniform(0.2, 1.8, m), rng.uniform(0.7, 2.8, m)])
    q = rng.uniform(0.0, 0.1, m)
    X = np.tile(BASE, (m, 1))
    X[:, [0, 15]] = truth
    X[:, 18] = q
    obs = toy_forward(torch.from_numpy(X.T))[..., 0]
    obs[3, 2] = float("nan")                        # an observation that must come out INVALID
    start = torch.from_numpy(np.stack([truth * 0.9, truth * 1.1, np.full_like(truth, np.nan)], axis=1))
    return space, obs, start, torch.from_numpy(q)


def test_driver_with_stand_ins_matches_run_np():
    space, obs, start, q = _toy_problem()
    kw = dict(design=design_torch, forward=toy_forward, step=step_torch, finish=finish_torch, per_obs={"q": q})
    res = inversion.invert(obs, S2A, space, start, **kw)
    ref = run_np(space, obs.numpy(), start.numpy(), lambda p: toy_forward(torch.from_numpy(p)).numpy(),
                 obs_rows=(18,), obs_values=q.numpy()[None])
    for got, want in zip((res.x, res.cost, res.std, res.status, res.start, res.iterations, res.n_forward), ref):
        np.testing.assert_array_equal(got.numpy(), want)
    assert res.status[3] == INVALID and torch.isnan(res.x[3]).all()
    for chunk in (1, 2, 5):
        again = inversion.invert(obs, S2A, space, start, chunk=chunk, **kw)
        assert torch.equal(again.x.nan_to_num(-1), res.x.nan_to_num(-1)) and torch.equal(again.status, res.status)


# ---- gloo, world size 2 ----------------------------------------------------------------------------------------------

def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    sys.path.insert(0, str(ROOT / "tests"))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        space, obs, start, qv = _toy_problem()
        res = inversion.invert(obs, S2A, space, start, per_obs={"q": qv}, design=design_torch, forward=toy_forward,
                               step=step_torch, finish=finish_torch, group=dist.group.WORLD)
        table = torch.arange(27 * 10, dtype=torch.float64).reshape(27, 10)
        idx = torch.tensor([[0, 9, 2 ** 32 - 1], [5, 4, 3]], dtype=torch.int64)
        lo, hi = (0, 4) if rank == 0 else (4, 10)
        st = inversion.starts(table[:, lo:hi], idx, space, group=dist.group.WORLD)
        q.put((rank, [t.numpy() for t in (res.x, res.cost, res.std, res.status, res.start, res.iterations,
                                           res.n_forward)], st.numpy()))
    finally:
        dist.destroy_process_group()


def test_group_gives_the_single_process_answer():
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict((r, (res, st)) for r, res, st in (q.get(timeout=120) for _ in procs))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    space, obs, start, qv = _toy_problem()
    one = inversion.invert(obs, S2A, space, start, per_obs={"q": qv}, design=design_torch, forward=toy_forward,
                           step=step_torch, finish=finish_torch)
    table = torch.arange(27 * 10, dtype=torch.float64).reshape(27, 10)
    idx = torch.tensor([[0, 9, 2 ** 32 - 1], [5, 4, 3]], dtype=torch.int64)
    st1 = inversion.starts(table, idx, space)
    assert torch.isnan(st1[0, 2]).all() and st1[1, 0, 1] == table[15, 5]
    for r in range(2):
        res, st = out[r]
        for got, want in zip(res, (one.x, one.cost, one.std, one.status, one.start, one.iterations, one.n_forward)):
            np.testing.assert_array_equal(got, want.numpy())
        np.testing.assert_array_equal(st, st1.numpy())
