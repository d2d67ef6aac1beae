"""The sensitivity analysis on the GPU: the Sobol' design kernel against SciPy and against the NumPy restatement of
its scramble (test_sobol_cpu), its net property and Saltelli layout, the refusals, the estimator against
scipy.stats.sobol_indices on the Ishigami function and on forward-model outputs, exact zeros where an output reads
no varied row, determinism, sharding, FP32 and SRF modes, and the stream / thread contract."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from test_sobol_cpu import design_np  # noqa: E402

S2A, L8 = "Sentinel2A-MSI", "LANDSAT8-OLI"
BASE = np.array([40, 0.01, 0.02, 0.1, 10, 1, 1.5, 0, 0, 0.5, 10, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                 40, 0, 0, 0.3, 0.35, 1.5, 1013, 180], dtype=np.float64)
E2E = {"Cab": (5, 80), "Cw": (0.005, 0.05), "SMp": (5, 55), "LAI": (0.1, 8), "aot550": (0.05, 0.6),
       "uh2o": (0.5, 4)}


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    yield torch, spart_b200
    torch.cuda.synchronize()


def _raw_design(torch, rows, lo, hi, seed, scramble, first, count, saltelli, ld=None):
    from spart_b200 import _lib
    d = len(rows)
    n = (d + 2) * count if saltelli else count
    ld = n if ld is None else ld
    out = torch.full((27, max(ld, 1)), -1.0, dtype=torch.float64, device="cuda")
    r = np.asarray(rows, dtype=np.int32)
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    rc = _lib.load().spart_sobol_design(_lib.as_int32_ptr(r), _lib.as_double_ptr(lo), _lib.as_double_ptr(hi), d,
                                        seed, scramble, first, count, saltelli, out.data_ptr(), ld,
                                        torch.cuda.current_stream().cuda_stream)
    return rc, out


def _scipy_values(D, first, count, lo, hi):
    from scipy.stats import qmc
    eng = qmc.Sobol(D, scramble=False, bits=32)
    if first:
        eng.fast_forward(first)
    x = np.asarray(lo) + (np.asarray(hi) - np.asarray(lo)) * eng.random(count)
    return np.where(x < hi, x, np.nextafter(hi, lo))


@pytest.mark.parametrize("first", [0, 12345, 2 ** 32 - 70])
@pytest.mark.parametrize("D", [1, 7, 54])
def test_unscrambled_design_equals_scipy(env, D, first):
    torch, _ = env
    count = 70 if first == 2 ** 32 - 70 else 4096
    rng = np.random.default_rng(D)
    d = D // 2 if D == 54 else D
    rows = rng.permutation(27)[:d]
    lo = rng.uniform(-50, 50, d)
    hi = lo + rng.uniform(1e-3, 100, d)
    rc, out = _raw_design(torch, rows, lo, hi, 0, 0, first, count, int(D == 54))
    assert rc == 0
    got = out.cpu().numpy()
    if D == 54:
        want = _scipy_values(D, first, count, np.tile(lo, 2), np.tile(hi, 2))
        for p, r in enumerate(rows):
            assert np.array_equal(got[r, :count], want[:, p]) and np.array_equal(got[r, count:2 * count], want[:, d + p])
    else:
        want = _scipy_values(D, first, count, lo, hi)
        for p, r in enumerate(rows):
            assert np.array_equal(got[r], want[:, p])
    untouched = np.setdiff1d(np.arange(27), rows)
    assert (got[untouched] == -1.0).all()


@pytest.mark.parametrize("seed", [0, 0xDEADBEEFCAFEF00D])
@pytest.mark.parametrize("saltelli", [0, 1])
def test_scrambled_design_equals_numpy_restatement(env, seed, saltelli):
    torch, _ = env
    rows, lo, hi = [3, 22, 0, 26, 15], [0, 0.05, 5, 1, 0.1], [0.5, 0.6, 80, 366, 8]
    for first, count in ((0, 2048), (777, 1000)):
        rc, out = _raw_design(torch, rows, lo, hi, seed, 1, first, count, saltelli)
        assert rc == 0
        got = out.cpu().numpy()
        for r, x in design_np(rows, lo, hi, seed, True, first, count, saltelli).items():
            assert np.array_equal(got[r], x), (r, first)


def test_scrambled_design_keeps_the_net_property(env):
    torch, _ = env
    n = 2 ** 16
    rc, out = _raw_design(torch, list(range(27)), [0.0] * 27, [1.0] * 27, 5, 1, 0, n, 1)
    assert rc == 0
    x = out.cpu().numpy()
    rc, plain = _raw_design(torch, list(range(27)), [0.0] * 27, [1.0] * 27, 5, 0, 0, n, 1)
    assert not np.array_equal(x[:, :2 * n], plain.cpu().numpy()[:, :2 * n])
    for r in range(27):
        for blk in (0, 1):                           # A: dimension r, B: dimension 27 + r
            for m in range(17):
                cells = np.floor(x[r, blk * n:blk * n + 2 ** m] * 2 ** m).astype(np.int64)
                assert np.array_equal(np.bincount(cells, minlength=2 ** m), np.ones(2 ** m)), (r, blk, m)


def test_design_blocks(env):
    torch, spart_b200 = env
    sp = spart_b200.sensitivity.ParameterSpace(BASE, E2E)
    n, d = 1000, sp.d
    P = sp.design(n, seed=9, first=321).cpu().numpy()
    S = sp.sample(n, seed=9, first=321).cpu().numpy()
    rows = list(sp.rows)
    A, B = P[:, :n], P[:, n:2 * n]
    assert np.array_equal(A[rows], S[rows])
    fixed = np.setdiff1d(np.arange(27), rows)
    assert np.array_equal(P[fixed, 0], BASE[fixed]) and np.array_equal(S[fixed], np.repeat(BASE[fixed, None], n, 1))
    for i, r in enumerate(rows):
        AB = P[:, (2 + i) * n:(3 + i) * n]
        others = [q for q in rows if q != r]
        assert np.array_equal(AB[others], A[others]) and np.array_equal(AB[r], B[r])
        assert not np.array_equal(AB[r], A[r])
    for p, (lo, hi) in enumerate(E2E.values()):
        assert (P[rows[p]] >= lo).all() and (P[rows[p]] < hi).all()


def test_refusals(env):
    torch, spart_b200 = env
    from spart_b200 import _lib
    sens = spart_b200.sensitivity
    lib = _lib.load()
    ok = dict(rows=[0, 15], lo=[5, 0.1], hi=[80, 8], seed=0, scramble=1, first=0, count=16, saltelli=1)

    def call(**kw):
        a = ok | kw
        rc, _ = _raw_design(torch, a["rows"], a["lo"], a["hi"], a["seed"], a["scramble"], a["first"], a["count"],
                            a["saltelli"], kw.get("ld"))
        return rc, lib.spart_last_error().decode()

    assert call()[0] == 0
    for kw, text in [(dict(first=2 ** 32 - 15), "2^32"), (dict(first=-1), "2^32"), (dict(count=-1), "2^32"),
                     (dict(rows=[0, 27], lo=[0, 0], hi=[1, 1]), "distinct"), (dict(rows=[4, 4]), "distinct"),
                     (dict(rows=[-1, 3]), "distinct"), (dict(lo=[5, 8]), "lo < hi"), (dict(hi=[np.inf, 8]), "lo < hi"),
                     (dict(lo=[np.nan, 0]), "lo < hi"), (dict(ld=16 * 4 - 1), "ld"), (dict(saltelli=0, ld=15), "ld"),
                     (dict(scramble=2), "scramble"), (dict(saltelli=2), "saltelli")]:
        rc, msg = call(**kw)
        assert rc == -1 and text in msg, (kw, msg)
    assert call(first=2 ** 32 - 16)[0] == 0
    rc, msg = call(rows=list(range(27)) + [0], lo=[0] * 28, hi=[1] * 28)          # 28 rows: n_vary > 27
    assert rc == -1 and "n_vary" in msg
    st = torch.cuda.current_stream().cuda_stream
    r = np.array([0], dtype=np.int32)
    one = np.array([1.0])
    zero = np.array([0.0])
    out = torch.empty((27, 16), dtype=torch.float64, device="cuda")
    assert lib.spart_sobol_design(None, _lib.as_double_ptr(zero), _lib.as_double_ptr(one), 1, 0, 1, 0, 4, 0,
                                  out.data_ptr(), 16, st) == -1
    assert lib.spart_sobol_design(_lib.as_int32_ptr(r), _lib.as_double_ptr(zero), _lib.as_double_ptr(one), 1, 0, 1,
                                  0, 4, 0, None, 16, st) == -1
    assert lib.spart_sobol_design(_lib.as_int32_ptr(r), _lib.as_double_ptr(zero), _lib.as_double_ptr(one), 0, 0, 1,
                                  0, 4, 0, out.data_ptr(), 16, st) == -1
    acc = torch.zeros(lib.spart_sobol_acc_elems(3, 1), dtype=torch.float64, device="cuda")
    f = torch.zeros(9, dtype=torch.float64, device="cuda")
    assert lib.spart_sobol_accumulate(f.data_ptr(), 1, 3, 1, None, acc.data_ptr(), st) == -1
    assert lib.spart_sobol_accumulate(f.data_ptr(), 1, 3, 28, f.data_ptr(), acc.data_ptr(), st) == -1
    assert lib.spart_sobol_accumulate(f.data_ptr(), -1, 3, 1, f.data_ptr(), acc.data_ptr(), st) == -1
    outs = [f.data_ptr()] * 6
    assert lib.spart_sobol_finish(acc.data_ptr(), f.data_ptr(), 0, 3, 1, *outs, st) == -1
    assert lib.spart_sobol_finish(acc.data_ptr(), f.data_ptr(), 1, 3, 1, *outs[:5], None, st) == -1
    sp = sens.ParameterSpace(BASE, {"Cab": (5, 80)})
    with pytest.raises(_lib.SpartError, match="2\\^32"):
        sp.sample(16, first=2 ** 32 - 15)
    with pytest.raises(ValueError, match="seed"):
        sp.sample(16, seed=-1)
    with pytest.raises(ValueError, match="count"):
        sp.design(0)
    with pytest.raises(ValueError, match="indices"):
        sens.indices(f[:4].reshape(2, 2), f[:4].reshape(2, 2), f[:4].reshape(1, 2, 2).float())
    with pytest.raises(ValueError, match="1 <= d <= 27"):
        sens.indices(f[:4].reshape(2, 2), f[:4].reshape(2, 2), f[:4].reshape(1, 4, 1))


def _ishigami(x):
    return np.sin(x[0]) + 7 * np.sin(x[1]) ** 2 + 0.1 * x[2] ** 4 * np.sin(x[0])


def _scipy(f_A, f_B, f_AB):
    from scipy.stats import sobol_indices
    return sobol_indices(func={"f_A": f_A.copy(), "f_B": f_B.copy(), "f_AB": f_AB.copy()}, n=f_A.shape[1])


def _check_scipy(res, f_A, f_B, f_AB, first, total):
    """first, total [s, d] against NumPy's two-pass Saltelli estimator at |dS| <= 1e-12 mean|t| / V and
    |dST| <= 1e-12 mean(u) / V, and against scipy.stats.sobol_indices at that tolerance plus SciPy's own rounding:
    SciPy centres f_A and f_AB before it forms f_AB - f_A, which costs up to ~eps (|f_A| + |f_AB|) per difference."""
    want = _scipy(f_A, f_B, f_AB)
    mu = np.mean([f_A, f_B], axis=(0, -1))[:, None]
    V = np.var([f_A, f_B], axis=(0, -1))[:, None]
    D = f_AB - f_A
    t = np.abs((f_B - mu) * D).mean(-1).T
    u = (D ** 2).mean(-1).T
    eps = np.finfo(np.float64).eps
    mag = np.abs(f_A) + np.abs(f_AB)
    tol_s, tol_st = 1e-12 * t / V, 1e-12 * u / V
    assert (np.abs(first - np.mean((f_B - mu) * D, -1).T / V) <= tol_s).all()
    assert (np.abs(total - np.mean(D ** 2, -1).T / (2 * V)) <= tol_st).all()
    assert (np.abs(first - want.first_order) <= tol_s + 4 * eps * np.mean(np.abs(f_B - mu) * mag, -1).T / V).all()
    assert (np.abs(total - want.total_order) <= tol_st + 4 * eps * np.mean(np.abs(D) * mag, -1).T / V).all()
    np.testing.assert_allclose(np.reshape(res.var, -1), V[:, 0], rtol=1e-12)
    return want


def _ishigami_outputs(torch, spart_b200, n, offset=0.0):
    sp = spart_b200.sensitivity.ParameterSpace(BASE, {"Cab": (-np.pi, np.pi), "Cw": (-np.pi, np.pi),
                                                      "LAI": (-np.pi, np.pi)})
    P = sp.design(n, seed=2024).cpu().numpy()[sp.rows]
    f = (_ishigami(P) + offset).reshape(5, 1, n)
    return f[0], f[1], f[2:]


def test_ishigami_against_scipy_and_analytic(env):
    torch, spart_b200 = env
    f_A, f_B, f_AB = _ishigami_outputs(torch, spart_b200, 2 ** 16)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    res = spart_b200.sensitivity.indices(cuda(f_A), cuda(f_B), cuda(f_AB))
    _check_scipy(res, f_A, f_B, f_AB, res.first, res.total)
    S = np.array([0.3139, 0.4424, 0.0])
    ST = np.array([0.5576, 0.4424, 0.2437])
    assert (np.abs(res.first[0] - S) <= 4 * res.first_se[0]).all(), (res.first, res.first_se)
    assert (np.abs(res.total[0] - ST) <= 4 * res.total_se[0]).all(), (res.total, res.total_se)
    assert (res.first_se > 0).all() and (res.first_se < 0.02).all() and (res.total_se < 0.02).all()


def test_shift_keeps_the_variance_far_above_the_spread(env):
    torch, spart_b200 = env
    f_A, f_B, f_AB = _ishigami_outputs(torch, spart_b200, 2 ** 16, offset=1e4)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    res = spart_b200.sensitivity.indices(cuda(f_A), cuda(f_B), cuda(f_AB))
    both = np.concatenate([f_A, f_B], axis=1)
    V = np.mean((both - both.mean()) ** 2)
    assert abs(res.var[0] - V) <= 1e-9 * V
    m = both.size
    raw = np.cumsum(both.ravel() ** 2)[-1] / m - (np.cumsum(both.ravel())[-1] / m) ** 2   # raw power sums, in order
    assert abs(raw - V) > 1e-9 * V
    base = spart_b200.sensitivity.indices(cuda(f_A - 1e4), cuda(f_B - 1e4), cuda(f_AB - 1e4))
    np.testing.assert_allclose(res.first, base.first, rtol=0, atol=1e-9)
    np.testing.assert_allclose(res.total, base.total, rtol=0, atol=1e-9)


def _e2e_space(spart_b200, extra=None):
    return spart_b200.sensitivity.ParameterSpace(BASE, E2E | (extra or {}))


def _reference(torch, spart_b200, sp, sensor, n, seed=0, **kw):
    """f_A, f_B, f_AB [s, N] from run_batch_params on space.design (the outputs of sobol's forward pass)."""
    P = sp.design(n, seed=seed)
    F = spart_b200.run_batch_params(P, sensor, broadcast_rows=sp.broadcast_rows, **kw).cpu().numpy()
    F = F.reshape(sp.d + 2, n, -1).transpose(0, 2, 1)
    return F[0], F[1], F[2:]


@pytest.fixture(scope="module")
def s2a_fp64(env):
    torch, spart_b200 = env
    sp = _e2e_space(spart_b200)
    return sp, spart_b200.sensitivity.sobol(sp, S2A, 2 ** 12, chunk=2 ** 10)


def test_end_to_end_against_scipy_and_exact_zeros(env, s2a_fp64):
    torch, spart_b200 = env
    sp, res = s2a_fp64
    assert res.names == tuple(E2E) and res.first.shape == (13, 3, 6) and res.n == 2 ** 12
    f_A, f_B, f_AB = _reference(torch, spart_b200, sp, S2A, 2 ** 12)
    _check_scipy(res, f_A, f_B, f_AB, res.first.reshape(-1, 6), res.total.reshape(-1, 6))
    np.testing.assert_allclose(res.mean.reshape(-1), np.mean([f_A, f_B], axis=(0, -1)), rtol=1e-13)
    # water vapour enters only the gaseous transmittance of R_TOA, so R_TOC never reads uh2o; aerosols do reach
    # R_TOC, through the direct / diffuse weights of its band value (ta_ss rso + ta_sd rdo) / (ta_ss + ta_sd)
    i = res.names.index("uh2o")
    assert (res.first[:, 0, i] == 0.0).all() and (res.total[:, 0, i] == 0.0).all()
    assert (res.total[:, 1, i] != 0.0).any()
    assert (res.total[:, 0, res.names.index("aot550")] > 0).all()
    assert (res.total[:, 0, res.names.index("LAI")] > 0).all()
    doy = spart_b200.sensitivity.sobol(_e2e_space(spart_b200, {"DOY": (1, 366)}), S2A, 2 ** 10)
    for c in (0, 1):                                 # DOY scales L_TOA only
        assert (doy.first[:, c, -1] == 0.0).all() and (doy.total[:, c, -1] == 0.0).all()
    assert (doy.total[:, 2, -1] > 0).all()


def test_determinism_chunks_and_nccl(env, s2a_fp64, tmp_path):
    torch, spart_b200 = env
    sp, res = s2a_fp64
    again = spart_b200.sensitivity.sobol(sp, S2A, 2 ** 12, chunk=2 ** 10)
    big = spart_b200.sensitivity.sobol(sp, S2A, 2 ** 12, chunk=2 ** 12)
    for k in ("mean", "var", "first", "total", "first_se", "total_se"):
        assert np.array_equal(getattr(again, k), getattr(res, k)), k
        np.testing.assert_allclose(getattr(big, k), getattr(res, k), rtol=1e-12, atol=1e-12 * np.abs(getattr(res, k)).max())
    import torch.distributed as dist
    dist.init_process_group("nccl", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1,
                            device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        sh = spart_b200.sensitivity.sobol(sp, S2A, 2 ** 12, chunk=2 ** 10, group=dist.group.WORLD)
    finally:
        dist.destroy_process_group()
    for k in ("mean", "var", "first", "total", "first_se", "total_se"):
        assert np.array_equal(getattr(sh, k), getattr(res, k)), k


def test_fp32_and_srf_modes(env, s2a_fp64):
    torch, spart_b200 = env
    sp, res = s2a_fp64
    r32 = spart_b200.sensitivity.sobol(sp, S2A, 2 ** 12, chunk=2 ** 10, precision="fp32")
    assert np.abs(r32.first - res.first).max() <= 1e-3 and np.abs(r32.total - res.total).max() <= 1e-3
    i = r32.names.index("uh2o")
    assert (r32.first[:, 0, i] == 0.0).all() and (r32.total[:, 0, i] == 0.0).all()
    srf = spart_b200.sensitivity.sobol(sp, L8, 2 ** 10, band_mode="srf")
    f_A, f_B, f_AB = _reference(torch, spart_b200, sp, L8, 2 ** 10, band_mode="srf")
    _check_scipy(srf, f_A, f_B, f_AB, srf.first.reshape(-1, 6), srf.total.reshape(-1, 6))


def test_stream_and_threads(env, s2a_fp64):
    torch, spart_b200 = env
    sp, res = s2a_fp64
    sens = spart_b200.sensitivity
    l8 = sens.sobol(sp, L8, 2 ** 11, chunk=2 ** 9)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(1 << 26)                  # work queued ahead on the side stream
        side = sens.sobol(sp, S2A, 2 ** 12, chunk=2 ** 10)
    results, errors = {}, []

    def job(name, sensor, n, chunk):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                results[name] = sens.sobol(sp, sensor, n, chunk=chunk)
        except Exception as e:                       # reported below
            errors.append(e)
    threads = [threading.Thread(target=job, args=a) for a in (("s2a", S2A, 2 ** 12, 2 ** 10), ("l8", L8, 2 ** 11, 2 ** 9))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for got, want in ((side, res), (results["s2a"], res), (results["l8"], l8)):
        for k in ("mean", "var", "first", "total", "first_se", "total_se"):
            assert np.array_equal(getattr(got, k), getattr(want, k)), k
