"""The retrieval by bounded Levenberg-Marquardt on the GPU: the design and step kernels against their NumPy
restatement (test_invert_cpu), the forward-difference Jacobian against oracle central differences, local
convergence, retrieval from a LUT's nearest entries, the invariants of every result, the covariance, bad input,
bit-identical results across calls, chunk sizes, batches, streams and threads, and the SRF and soil-library modes."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from test_invert_cpu import (BASE, VARY6, VARY7, design_np, finish_np, init_np, moved, step_np,  # noqa: E402
                             x_of)

S2A, L8 = "Sentinel2A-MSI", "LANDSAT8-OLI"
ANGLES = {"sol_angle": (20.0, 60.0), "obs_angle": (0.0, 30.0), "rel_angle": (0.0, 180.0)}


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    yield torch, spart_b200
    torch.cuda.synchronize()


def _space(sb, vary, base=BASE):
    return sb.sensitivity.ParameterSpace(base, vary)


def _truth_batch(torch, space, u, per_obs=None):
    """Full [27, m] batch of the points u [m, P] (x = lo + (hi - lo) u) with per-observation rows."""
    m = u.shape[0]
    X = np.tile(space.base, (m, 1))
    X[:, space.rows] = x_of(space.lo, space.hi, u)
    for r, v in (per_obs or {}).items():
        X[:, r] = v
    return torch.from_numpy(np.ascontiguousarray(X.T)).cuda()


def _forward(torch, sb, batch, sensor=S2A, **kw):
    return sb.default_engine().forward_bands(batch, sensor, **kw)


def _per_obs_rows(rng, m):
    names = sorted(ANGLES, key=lambda n: ["sol_angle", "obs_angle", "rel_angle"].index(n))
    return {19 + i: rng.uniform(*ANGLES[n], m) for i, n in enumerate(names)}


def _prob(torch, sb, space, obs, S, per_obs=None, weights=None, column=0, absolute_sigma=False):
    inv = sb.inversion
    ftol, xtol, max_iter = inv.FTOL, inv.XTOL, inv.MAX_ITERATIONS
    per_obs = per_obs or {}
    rows = np.array(sorted(per_obs), dtype=np.int32)
    vals = (torch.from_numpy(np.stack([per_obs[r] for r in rows])).cuda() if len(rows)
            else torch.empty((0, obs.shape[0]), dtype=torch.float64, device="cuda"))
    bc = sum(1 << r for r in range(27) if r not in space.rows and r not in rows)
    return inv.Problem(space.rows, space.lo, space.hi, space.base, rows, vals, obs.contiguous(), weights, S, column,
                       ftol, xtol, max_iter, absolute_sigma, bc)


# ---- kernels against the NumPy restatement -------------------------------------------------------------------------

def test_design_kernel_equals_design_np(env):
    torch, sb = env
    inv = sb.inversion
    space = _space(sb, VARY7)
    rng = np.random.default_rng(3)
    m, S, P = 50, 3, space.d
    u = rng.uniform(0, 1, (m * S, P))
    u[::7, 2] = 1.0                                  # moved downwards
    u[1::7, 4] = 1.0 - 2.0 ** -18                    # also downwards
    u[2::7, 1] = 0.0
    start = x_of(space.lo, space.hi, u).reshape(m, S, P)
    per = _per_obs_rows(rng, m)
    per[22] = rng.uniform(0.05, 0.5, m)
    obs = torch.zeros((m, 13), dtype=torch.float64, device="cuda")
    prob = _prob(torch, sb, space, obs, S, per)
    state = inv.init_state(prob, torch.from_numpy(start).cuda())
    active = torch.from_numpy(rng.permutation(m * S)[:101].astype(np.int32)).cuda()
    buf = torch.full((27, 101 * (P + 1) + 5), -7.0, dtype=torch.float64, device="cuda")
    got = inv._design(prob, state, active, buf)
    assert got.shape == (27, 101 * (P + 1))
    want = np.full(buf.shape, -7.0)
    design_np(space.rows, space.lo, space.hi, space.base, list(prob.obs_rows), prob.obs_values.cpu().numpy(), S,
              state.cpu().numpy(), active.cpu().numpy(), want)
    np.testing.assert_array_equal(buf.cpu().numpy(), want)
    np.testing.assert_array_equal(state.cpu().numpy(), init_np(space.lo, space.hi, start))


def _one_step_both(torch, sb, prob, state, active, sensor=S2A):
    """Design + forward on the GPU, then the step kernel and step_np on copies of the same state."""
    inv = sb.inversion
    P = prob.P
    buf = torch.empty((27, active.numel() * (P + 1)), dtype=torch.float64, device="cuda")
    f = _forward(torch, sb, inv._design(prob, state, active, buf), sensor, broadcast_rows=prob.bcast_mask)
    ref = state.cpu().numpy().copy()
    inv._step(prob, f, state, active)
    step_np(prob.lo, prob.hi, prob.n_starts, f.cpu().numpy(), prob.column, prob.obs.cpu().numpy(),
            None if prob.weights is None else prob.weights.cpu().numpy(), prob.ftol, prob.xtol, prob.max_iter, ref,
            active.cpu().numpy())
    return state.cpu().numpy(), ref


def _check_step(got, ref, L, P):
    """The step kernel's state against step_np's: status, C, lambda and u (the accepted point) within 1e-12
    relative, J^T W J and J^T W r within 1e-10 of each row's largest magnitude, and the next trial within 1e-8: it
    is the solution of a Marquardt system whose conditioning magnifies the rounding differences of its sums."""
    np.testing.assert_array_equal(got[L["status"]], ref[L["status"]])
    np.testing.assert_array_equal(np.isnan(got), np.isnan(ref))
    for name, n, tol, rel in (("u", P, 1e-12, True), ("C", 1, 1e-12, True), ("lam", 1, 1e-12, True),
                              ("A", P * (P + 1) // 2, 1e-10, False), ("g", P, 1e-10, False),
                              ("trial", P, 1e-8, False)):
        a, b = np.nan_to_num(got[L[name]:L[name] + n]), np.nan_to_num(ref[L[name]:L[name] + n])
        scale = np.maximum(np.abs(a), np.abs(b)) if rel else np.abs(np.concatenate([a, b], 1)).max(1, keepdims=True)
        err = np.abs(a - b) / np.where(scale > 0, scale, 1.0)
        assert err.max() <= tol, (name, err.max())


def test_one_step_equals_step_np_accept_reject_and_retry(env):
    torch, sb = env
    inv = sb.inversion
    lay = inv.layout
    space = _space(sb, VARY6)
    P = space.d
    L = lay(P)
    rng = np.random.default_rng(4)
    m, S = 64, 2
    truth = rng.uniform(0.1, 0.9, (m, P))
    obs = _forward(torch, sb, _truth_batch(torch, space, truth))[..., 0].contiguous()
    start = x_of(space.lo, space.hi, np.clip(truth[:, None] + rng.uniform(-0.15, 0.15, (m, S, P)), 0, 1))
    prob = _prob(torch, sb, space, obs, S)
    state = inv.init_state(prob, torch.from_numpy(start).cuda())
    active = torch.arange(m * S, dtype=torch.int32, device="cuda")
    got, ref = _one_step_both(torch, sb, prob, state, active)          # first call: every start accepted
    _check_step(got, ref, L, P)
    before = got.copy()
    got, ref = _one_step_both(torch, sb, prob, torch.from_numpy(before).cuda(), active)   # mostly accepted
    acc_gpu = got[L["lam"]] < before[L["lam"]]
    assert acc_gpu.sum() > m
    _check_step(got, ref, L, P)
    # rejections: trials moved far away; retries: an indefinite stored J^T W J on a quarter of the tracks
    st = got.copy()
    st[L["trial"]:L["trial"] + P] = np.where(st[L["u"]:L["u"] + P] < 0.5, 0.98, 0.02)
    k = np.arange(0, m * S, 4)
    st[L["A"]:L["A"] + 3, k] = np.array([1.0, 3.0, 1.0])[:, None] * st[L["A"], k]
    before = st.copy()
    state = torch.from_numpy(st).cuda()
    got, ref = _one_step_both(torch, sb, prob, state, active)
    rejected = got[L["C"]] == before[L["C"]]
    assert rejected.sum() >= m and (rejected == (ref[L["C"]] == before[L["C"]])).all()
    _check_step(got, ref, L, P)
    retried = rejected[k] & (got[L["lam"], k] > 10 * before[L["lam"], k] * 1.5)
    assert retried.sum() >= m // 8, "the Cholesky retry branch was not taken"


def test_uh2o_on_R_TOC_stays_at_its_start_with_nan_std(env):
    """uh2o does not reach R_TOC (DESIGN §8, "Exact zeros"): its Jacobian column is exactly zero, so its step is
    exactly 0 (the pivot lambda 1e-30 stays positive) and J^T W J is singular, so every std is NaN."""
    torch, sb = env
    space = _space(sb, dict(VARY6, uh2o=(0.5, 4.0)))
    rng = np.random.default_rng(5)
    m, P = 32, space.d
    truth = rng.uniform(0.1, 0.9, (m, P))
    obs = _forward(torch, sb, _truth_batch(torch, space, truth))[..., 0].contiguous()
    u0 = np.clip(truth + rng.uniform(-0.1, 0.1, (m, P)), 0, 1)
    start = x_of(space.lo, space.hi, u0)[:, None, :]
    res = sb.inversion.invert(obs, S2A, space, torch.from_numpy(start))
    x = res.x.cpu().numpy()
    u_init = init_np(space.lo, space.hi, start)[P:2 * P].T
    np.testing.assert_array_equal(x[:, -1], x_of(space.lo[-1], space.hi[-1], u_init[:, -1]))
    assert np.isnan(res.std.cpu().numpy()).all()
    assert np.abs((x[:, :-1] - space.lo[:-1]) / (space.hi - space.lo)[:-1] - truth[:, :-1]).max() <= 1e-9


def test_jacobian_against_oracle_central_differences(env, optical):
    """The forward-difference Jacobian of the kernels' own design (GPU forward outputs) against central differences
    of the oracle (step 2^-10), LIDFa included, 64 points: within 2e-4 of each column's largest value."""
    import spart_oracle
    torch, sb = env
    inv = sb.inversion
    space = _space(sb, VARY7)
    P = space.d
    rng = np.random.default_rng(6)
    n = 64
    U = rng.uniform(0.05, 0.95, (n, P))
    obs = torch.zeros((n, 13), dtype=torch.float64, device="cuda")
    prob = _prob(torch, sb, space, obs, 1)
    state = inv.init_state(prob, torch.from_numpy(x_of(space.lo, space.hi, U)[:, None]).cuda())
    active = torch.arange(n, dtype=torch.int32, device="cuda")
    buf = torch.empty((27, n * (P + 1)), dtype=torch.float64, device="cuda")
    f = _forward(torch, sb, inv._design(prob, state, active, buf), broadcast_rows=prob.bcast_mask)
    f = f[..., 0].cpu().numpy().reshape(n, P + 1, 13)
    u = state.cpu().numpy()[P:2 * P].T

    def F(V):
        X = np.tile(BASE, (V.shape[0], 1))
        X[:, space.rows] = x_of(space.lo, space.hi, V)
        return spart_oracle.spart_bands(X, S2A, optical)[..., 0]
    worst = []
    for p in range(P):
        du = (x_of(space.lo[p], space.hi[p], moved(u[:, p])) - x_of(space.lo[p], space.hi[p], u[:, p])) / (
            space.hi[p] - space.lo[p])
        fd = (f[:, p + 1] - f[:, 0]) / du[:, None]
        hc = 2.0 ** -10
        V1, V2 = u.copy(), u.copy()
        V1[:, p] += hc
        V2[:, p] -= hc
        cd = (F(V1) - F(V2)) / (2 * hc)
        worst.append(np.abs(fd - cd).max() / np.abs(cd).max())
    print("forward vs central differences, per column:", " ".join(f"{w:.1e}" for w in worst))
    assert max(worst) <= 2e-4, worst


# ---- convergence ---------------------------------------------------------------------------------------------------

def test_local_convergence_with_per_observation_geometry(env):
    """4096 observations, random truth and per-observation sun / view angles, one start at truth +- 0.15, run with
    max_iter = 500 so that the slow tail of the iteration is seen to converge rather than cut off.  Measured on a
    B200: 4094 of 4096 (0.99951) at the truth, all CONVERGED_STEP, the other two in another minimum; 8 tracks
    needed more than 50 forward calls (at most 369).  With the default max_iter = 50, 4088 (0.99805) converge and
    8 stop at MAX_ITER: the default trades that tail for bounded iteration counts per chunk (DESIGN §8)."""
    torch, sb = env
    space = _space(sb, VARY6)
    rng = np.random.default_rng(7)
    m, P = 4096, space.d
    truth = rng.uniform(0.05, 0.95, (m, P))
    per = _per_obs_rows(rng, m)
    bc = sum(1 << r for r in range(27) if r not in space.rows and r not in per)
    obs = _forward(torch, sb, _truth_batch(torch, space, truth, per), broadcast_rows=bc)[..., 0].contiguous()
    start = x_of(space.lo, space.hi, np.clip(truth + rng.uniform(-0.15, 0.15, (m, P)), 0, 1))[:, None]
    res = sb.inversion.invert(obs, S2A, space, torch.from_numpy(start), per_obs=per, max_iter=500)
    u = (res.x.cpu().numpy() - space.lo) / (space.hi - space.lo)
    status = res.status.cpu().numpy()
    iters = res.iterations.cpu().numpy()
    ok = np.isin(status, (1, 2)) & (np.abs(u - truth).max(1) <= 1e-9)
    print(f"local convergence: {ok.sum()} of {m} ({ok.mean():.5f}) recovered; statuses "
          f"{np.bincount(status, minlength=6)}; forward calls median {np.median(iters)}, over 50: "
          f"{(iters > 50).sum()}, max {iters.max()}; misses at |u - truth| {np.abs(u - truth).max(1)[~ok]}")
    assert ok.mean() >= 0.999


@pytest.fixture(scope="module")
def lut_run(env):
    """Starts from nearest_k(k=8) of a 2^16-entry space.sample LUT (Sentinel-2A R_TOC, fixed geometry), 2048
    observations of random truth."""
    torch, sb = env
    space = _space(sb, VARY6)
    table = space.sample(2 ** 16, seed=11)
    lut = sb.lut.generate(table, S2A, column=0)
    rng = np.random.default_rng(8)
    m = 2048
    truth = rng.uniform(0.02, 0.98, (m, space.d))
    obs = _forward(torch, sb, _truth_batch(torch, space, truth), broadcast_rows=space.broadcast_rows)[..., 0]
    obs = obs.contiguous()
    idx, _ = sb.lut.nearest_k(lut, obs.float(), 8)
    start = sb.inversion.starts(table, idx, space)
    res = sb.inversion.invert(obs, S2A, space, start)
    return space, truth, obs, start, res


def test_from_the_lut(env, lut_run):
    """Measured on a B200: every observation recovered to 1e-6 (2048 of 2048, all CONVERGED_STEP); asserted
    >= 0.995."""
    torch, sb = env
    space, truth, obs, start, res = lut_run
    u = (res.x.cpu().numpy() - space.lo) / (space.hi - space.lo)
    ok = np.abs(u - truth).max(1) <= 1e-6
    print(f"from the LUT: {ok.mean():.5f} recovered to 1e-6; statuses {np.bincount(res.status.cpu().numpy(), minlength=6)}"
          f"; forward runs per observation {res.n_forward.double().mean().item():.1f}")
    assert ok.mean() >= 0.995


def test_invariants_of_every_result(env, lut_run):
    torch, sb = env
    space, truth, obs, start, res = lut_run
    m, S, P = start.shape
    lo, hi = space.lo, space.hi
    x = res.x.cpu().numpy()
    assert ((x >= lo) & (x <= hi)).all()
    # the cost of every start, evaluated independently at the start clipped into the box
    u0 = init_np(lo, hi, start.cpu().numpy())[P:2 * P].T
    f0 = _forward(torch, sb, _truth_batch(torch, space, u0), broadcast_rows=space.broadcast_rows)[..., 0]
    c0 = ((f0.reshape(m, S, -1) - obs[:, None]) ** 2).sum(-1).cpu().numpy()
    best0 = np.nanmin(np.where(np.isfinite(c0), c0, np.nan), axis=1)
    cost = res.cost.cpu().numpy()
    assert (cost <= best0).all()
    batch = np.tile(BASE, (m, 1))
    batch[:, space.rows] = x
    f = _forward(torch, sb, torch.from_numpy(np.ascontiguousarray(batch.T)).cuda(),
                 broadcast_rows=space.broadcast_rows)[..., 0]
    d = (f - obs).cpu().numpy()
    again = np.zeros(m)
    for b in range(d.shape[1]):
        again = again + d[:, b] * d[:, b]
    np.testing.assert_allclose(cost, again, rtol=1e-13, atol=1e-300)


# ---- covariance ----------------------------------------------------------------------------------------------------

def test_std_equals_the_numpy_formula_on_the_final_state(env):
    torch, sb = env
    inv = sb.inversion
    space = _space(sb, VARY6)
    rng = np.random.default_rng(9)
    m, S, P = 128, 2, space.d
    truth = rng.uniform(0.1, 0.9, (m, P))
    obs = _forward(torch, sb, _truth_batch(torch, space, truth))[..., 0]
    obs = (obs + 1e-3 * torch.from_numpy(rng.standard_normal(obs.shape)).cuda()).contiguous()
    start = x_of(space.lo, space.hi, np.clip(truth[:, None] + rng.uniform(-0.1, 0.1, (m, S, P)), 0, 1))
    for absolute in (False, True):
        w = torch.from_numpy(rng.uniform(0.5, 2.0, 13)).cuda()
        prob = _prob(torch, sb, space, obs, S, weights=w, absolute_sigma=absolute)
        state = inv.init_state(prob, torch.from_numpy(start).cuda())
        buf = torch.empty((27, m * S * (P + 1)), dtype=torch.float64, device="cuda")
        while True:
            active = torch.nonzero(state[inv.layout(P)["status"]] == 0).reshape(-1).to(torch.int32)
            if not active.numel():
                break
            f = _forward(torch, sb, inv._design(prob, state, active, buf), broadcast_rows=prob.bcast_mask)
            inv._step(prob, f, state, active)
        got = [t.cpu().numpy() for t in inv._finish(prob, state)]
        want = finish_np(space.lo, space.hi, S, 13, absolute, state.cpu().numpy())
        np.testing.assert_allclose(got[2], want[2], rtol=1e-10)
        for g, wnt in zip(got[:2] + got[3:], want[:2] + want[3:]):
            np.testing.assert_array_equal(g, wnt)
        res = inv.invert(obs, S2A, space, torch.from_numpy(start), weights=w, absolute_sigma=absolute)
        np.testing.assert_array_equal(res.std.cpu().numpy(), got[2])


def test_std_matches_the_spread_of_noisy_estimates(env):
    """1024 noise draws (sigma 1e-4) of one truth, weights 1 / sigma^2, absolute_sigma: the empirical std of the
    estimates over the mean reported std lies in [0.85, 1.15] for every parameter."""
    torch, sb = env
    space = _space(sb, VARY6)
    P = space.d
    rng = np.random.default_rng(10)
    truth = np.full((1, P), 0.5)
    clean = _forward(torch, sb, _truth_batch(torch, space, truth))[..., 0]
    n, sigma = 1024, 1e-4
    obs = (clean + sigma * torch.from_numpy(rng.standard_normal((n, 13))).cuda()).contiguous()
    start = np.broadcast_to(x_of(space.lo, space.hi, truth)[:, None], (n, 1, P)).copy()
    res = sb.inversion.invert(obs, S2A, space, torch.from_numpy(start), weights=np.full(13, sigma ** -2),
                              absolute_sigma=True)
    x = res.x.cpu().numpy()
    ratio = x.std(0) / res.std.cpu().numpy().mean(0)
    print("empirical / reported std per parameter:", " ".join(f"{r:.3f}" for r in ratio))
    assert ((ratio >= 0.85) & (ratio <= 1.15)).all(), ratio


# ---- bad input, determinism, other modes ---------------------------------------------------------------------------

def _small(torch, sb, m=40, S=3, seed=12):
    space = _space(sb, VARY6)
    rng = np.random.default_rng(seed)
    truth = rng.uniform(0.1, 0.9, (m, space.d))
    per = _per_obs_rows(rng, m)
    bc = sum(1 << r for r in range(27) if r not in space.rows and r not in per)
    obs = _forward(torch, sb, _truth_batch(torch, space, truth, per), broadcast_rows=bc)[..., 0].contiguous()
    start = x_of(space.lo, space.hi, np.clip(truth[:, None] + rng.uniform(-0.2, 0.2, (m, S, space.d)), 0, 1))
    return space, obs, torch.from_numpy(start).cuda(), per, truth


def _fields(res):
    return [t.cpu().numpy() for t in (res.x, res.cost, res.std, res.status, res.start, res.iterations, res.n_forward)]


def _same(a, b):
    for u, v in zip(_fields(a), _fields(b)):
        np.testing.assert_array_equal(u, v)


def test_bad_input(env):
    torch, sb = env
    inv = sb.inversion
    space, obs, start, per, _ = _small(torch, sb)
    base = inv.invert(obs, S2A, space, start, per_obs=per)
    bad = obs.clone()
    bad[5, 3] = float("nan")
    start2 = start.clone()
    start2[9] = float("nan")                         # all starts NO_ENTRY
    res = inv.invert(bad, S2A, space, start2, per_obs=per)
    st = res.status.cpu().numpy()
    assert st[5] == inv.INVALID and st[9] == inv.INVALID and (res.start.cpu().numpy()[[5, 9]] == -1).all()
    for i in (5, 9):
        assert np.isnan(res.x[i].cpu().numpy()).all() and np.isnan(res.cost[i].item())
    keep = np.setdiff1d(np.arange(obs.shape[0]), [5, 9])
    for u, v in zip(_fields(res), _fields(base)):
        np.testing.assert_array_equal(u[keep], v[keep])
    empty = inv.invert(obs[:0], S2A, space, start[:0], per_obs={r: v[:0] for r, v in per.items()})
    assert empty.x.shape == (0, space.d) and empty.status.numel() == 0
    from spart_b200 import _lib
    lib = _lib.load()
    rows = space.rows
    r = lib.spart_invert_design(_lib.as_int32_ptr(rows), _lib.as_double_ptr(space.lo), _lib.as_double_ptr(space.hi),
                                space.d, _lib.as_int32_ptr(rows[:1].copy()), 1, obs.data_ptr(), obs.shape[0],
                                _lib.as_double_ptr(space.base), 1, obs.data_ptr(), 4, obs.data_ptr(), 1,
                                obs.data_ptr(), 64, torch.cuda.current_stream().cuda_stream)
    assert r == -1 and b"not varied" in lib.spart_last_error()
    r = lib.spart_invert_step(_lib.as_double_ptr(space.lo), _lib.as_double_ptr(space.hi), 17, 1, obs.data_ptr(), 13,
                              0, obs.data_ptr(), None, 1e-12, 1e-12, 50, obs.data_ptr(), 4, obs.data_ptr(), 1,
                              torch.cuda.current_stream().cuda_stream)
    assert r == -1


def test_bit_identical_results(env):
    torch, sb = env
    inv = sb.inversion
    space, obs, start, per, _ = _small(torch, sb)
    a = inv.invert(obs, S2A, space, start, per_obs=per)
    _same(a, inv.invert(obs, S2A, space, start, per_obs=per))
    _same(a, inv.invert(obs, S2A, space, start, per_obs=per, chunk=37))
    mixed = {r: (torch.from_numpy(v).cuda() if k % 2 else v) for k, (r, v) in enumerate(per.items())}
    _same(a, inv.invert(obs, S2A, space, start, per_obs=mixed))           # host arrays and CUDA tensors mixed
    i = 17
    alone = inv.invert(obs[i:i + 1], S2A, space, start[i:i + 1], per_obs={r: v[i:i + 1] for r, v in per.items()})
    for u, v in zip(_fields(alone), _fields(a)):
        np.testing.assert_array_equal(u, v[i:i + 1])
    space2, obs2, start2, per2, _ = _small(torch, sb, m=30, seed=13)
    b = inv.invert(obs2, S2A, space2, start2, per_obs=per2)
    results, errors = {}, []

    def job(name, o, sp, st, po):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                torch.cuda._sleep(1 << 24)
                results[name] = inv.invert(o, S2A, sp, st, per_obs=po)
                torch.cuda.current_stream().synchronize()
        except Exception as e:                       # reported below
            errors.append(e)
    threads = [threading.Thread(target=job, args=("a", obs, space, start, per)),
               threading.Thread(target=job, args=("b", obs2, space2, start2, per2))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    _same(results["a"], a)
    _same(results["b"], b)


def test_srf_and_soil_library_modes(env):
    torch, sb = env
    inv = sb.inversion
    rng = np.random.default_rng(14)
    space = _space(sb, {"Cab": (5, 80), "Cw": (0.005, 0.05), "LAI": (0.1, 8), "SMp": (5, 55)})
    m, P = 24, space.d
    truth = rng.uniform(0.1, 0.9, (m, P))
    obs = _forward(torch, sb, _truth_batch(torch, space, truth), L8, band_mode="srf",
                   broadcast_rows=space.broadcast_rows)[..., 1].contiguous()
    start = x_of(space.lo, space.hi, np.clip(truth + rng.uniform(-0.1, 0.1, (m, P)), 0, 1))[:, None]
    res = inv.invert(obs, L8, space, torch.from_numpy(start), column="R_TOA", band_mode="srf")
    u = (res.x.cpu().numpy() - space.lo) / (space.hi - space.lo)
    assert np.abs(u - truth).max() <= 1e-8, np.abs(u - truth).max(1)
    wl = np.linspace(0, 1, 2001)
    libr = sb.SoilLibrary(np.stack([0.1 + 0.2 * wl, 0.3 - 0.1 * wl, 0.2 + 0.05 * np.sin(6 * wl)]))
    soil = rng.integers(0, 3, m).astype(np.float64)
    bc = space.broadcast_rows & ~(1 << 9)
    obs = _forward(torch, sb, _truth_batch(torch, space, truth, {9: soil}), soil_library=libr,
                   broadcast_rows=bc)[..., 0].contiguous()
    res = inv.invert(obs, S2A, space, torch.from_numpy(start), per_obs={"B": soil}, soil_library=libr)
    u = (res.x.cpu().numpy() - space.lo) / (space.hi - space.lo)
    assert np.abs(u - truth).max() <= 1e-8, np.abs(u - truth).max(1)
