"""The CUDA paths over the whole input domain of the model, against the oracle.

The other parity tests draw their batches from `spart_oracle.synthetic_params`, the benchmark
distributions, and the goldens were recorded from the same generator.  Here every input spans the
range a user may pass (BOUNDS below), with extra rows at each bound and at the corners where the
kernels switch branches: the last pieces of the plate-transmissivity table, the dry-soil branch, the
exact hot spot, nadir, RAA = 360.

FP64 gate: 1e-9 relative.  An output that is a difference of O(1) terms -- R_TOA near 0 or outside
SMAC's validity, canopy reflectances outside (0, 1) -- has no relative accuracy in any floating-point
evaluation; `check_close` compares those with |got - want| <= tol * s, s the largest magnitude among the
summands, and every test asserts how many outputs took that rule."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import spart_oracle as so  # noqa: E402

RTOL64 = 1e-9
RTOL32 = 1e-4
MAX_SCALED = 0.01       # largest share of outputs that may pass by the summand-scale rule

# (column, low, high, where the bound comes from)
BOUNDS = [
    (so.CAB, 0.0, 120.0, "chlorophyll a+b, ug/cm2: PROSPECT-D calibration leaves reach ~100"),
    (so.CCA, 0.0, 30.0, "carotenoids, ug/cm2: about a quarter of Cab"),
    (so.CANT, 0.0, 40.0, "anthocyanins, ug/cm2: red / senescent leaves of the PROSPECT-D data"),
    (so.CS, 0.0, 1.5, "senescent material, fraction (brown pigments)"),
    (so.CW, 0.0, 0.1, "equivalent water thickness, cm: succulent leaves"),
    (so.CDM, 0.0, 0.04, "dry matter, g/cm2: thick evergreen leaves"),
    (so.NSTRUCT, 1.0, 4.0, "leaf structure parameter: 1 (monocot) .. 4 (dense dicot)"),
    (so.PROT, 0.0, 0.003, "PROSPECT-PRO proteins, g/cm2 (pro=True rows only)"),
    (so.CBC, 0.0, 0.01, "PROSPECT-PRO carbon-based constituents, g/cm2 (pro=True rows only)"),
    (so.SOIL_B, 0.0, 1.0, "BSM soil brightness"),
    (so.SOIL_LAT, 0.0, 40.0, "BSM spectral coordinate: B = 1 keeps the dry-soil spectrum >= 0 on this box"),
    (so.SOIL_LON, 50.0, 120.0, "BSM spectral coordinate, same box (reference defaults lat 0, lon 100)"),
    (so.SMP, 0.0, 100.0, "soil moisture, %: <= 5 is the dry branch (bsm.py:102-103)"),
    (so.SMC, 5.0, 60.0, "soil moisture capacity, %: Poisson mean (SMp - 5) / SMC up to 19"),
    (so.FILM, 0.0, 0.1, "water film optical thickness, cm"),
    (so.LAI, 0.0, 10.0, "leaf area index: bare soil .. dense forest"),
    (so.LIDFA, -1.0, 1.0, "leaf inclination: (LIDFa, LIDFb) uniform on |a| + |b| <= 1 (sailh.py:351-398)"),
    (so.LIDFB, -1.0, 1.0, "leaf inclination, see LIDFa"),
    (so.HOT_Q, 1e-3, 1.0, "hot-spot parameter, log-uniform"),
    (so.SZA, 0.0, 75.0, "solar zenith, deg: SMAC's validity ends near 75"),
    (so.VZA, 0.0, 70.0, "view zenith, deg"),
    (so.RAA, 0.0, 360.0, "relative azimuth, deg (folded at sailh.py:65)"),
    (so.AOT550, 0.0, 1.0, "aerosol optical thickness at 550 nm (SMAC)"),
    (so.UO3, 0.1, 0.6, "ozone column, atm-cm"),
    (so.UH2O, 0.0, 7.0, "water vapour column, g/cm2: dry polar .. tropical"),
    (so.PA, 500.0, 1050.0, "surface pressure, hPa: 5.5 km altitude .. high pressure"),
    (so.DOY, 1.0, 366.0, "day of year"),
]
LOG_UNIFORM = {so.HOT_Q}

# the reference's end-to-end example (tests/e2e/test_SPART.py): the value of every input not at a bound
DEFAULTS = np.array([40, 0.01, 0.02, 0, 10, 10, 1.5, 0, 0, 0.5, 0, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                     40, 0, 0, 0.325, 0.35, 1.41, 1013.25, 100], dtype=np.float64)


def wide_params(n, seed, pro=False):
    """[n, 27] batch, every input uniform (q log-uniform) over BOUNDS.  (LIDFa, LIDFb) is uniform on the
    diamond |a| + |b| <= 1 with one sample in ten exactly on its edge.  pro=True: PROSPECT-PRO leaves
    (PROT, CBC > 0 with Cdm > 0, so the switch of prospect_5d.py:148-155 zeroes Cdm); otherwise PROT = CBC = 0."""
    rng = np.random.default_rng(seed)
    P = np.zeros((n, so.NPAR))
    for col, lo, hi, _ in BOUNDS:
        if col in LOG_UNIFORM:
            P[:, col] = np.exp(rng.uniform(np.log(lo), np.log(hi), n))
        else:
            P[:, col] = rng.uniform(lo, hi, n)
    P[:, so.DOY] = rng.integers(1, 367, n).astype(np.float64)
    # uniform on the diamond: a square rotated by 45 degrees and scaled
    u, v = rng.uniform(-0.5, 0.5, n), rng.uniform(-0.5, 0.5, n)
    a, b = u + v, u - v
    edge = rng.uniform(0, 1, n) < 0.1
    t = rng.uniform(-1, 1, n)
    sgn = np.where(rng.uniform(0, 1, n) < 0.5, -1.0, 1.0)
    P[:, so.LIDFA] = np.where(edge, t, a)
    P[:, so.LIDFB] = np.where(edge, sgn * (1 - np.abs(t)), b)
    if pro:
        P[:, so.PROT] = rng.uniform(1e-4, 0.003, n)
        P[:, so.CBC] = rng.uniform(1e-4, 0.01, n)
        P[:, so.CDM] = rng.uniform(1e-4, 0.04, n)
    else:
        P[:, so.PROT] = P[:, so.CBC] = 0.0
    return P


def oat_rows():
    """Deterministic rows: every input at its lower and upper bound with the others at DEFAULTS, then corners."""
    rows = []

    def row(**kw):
        r = DEFAULTS.copy()
        for k, v in kw.items():
            r[getattr(so, k)] = v
        rows.append(r)
    for col, lo, hi, _ in BOUNDS:
        if col in (so.LIDFA, so.LIDFB, so.PROT, so.CBC):
            continue
        for v in (lo, hi):
            r = DEFAULTS.copy()
            r[col] = v
            rows.append(r)
    for a, b in ((1, 0), (-1, 0), (0, 1), (0, -1), (0.5, 0.5), (-0.5, -0.5), (0.5, -0.5)):   # LIDF diamond
        row(LIDFA=a, LIDFB=b)
    row(PROT=0.003, CBC=0.01, CDM=0.04)                        # PROSPECT-PRO at its bounds
    row(CW=0.1, CDM=0.04, NSTRUCT=1.0)                         # largest plate absorption, K up to ~17
    row(CW=0.1, CDM=0.04, NSTRUCT=1.0, CAB=120, CANT=40, CS=1.5, CCA=30)
    row(SMC=5.0, SMP=100.0)                                    # Poisson mean 19
    row(SMC=5.0, SMP=100.0, FILM=0.1)
    row(SMP=5.0)                                               # the dry branch boundary
    row(SZA=30.0, VZA=30.0, RAA=0.0)                           # exact hot spot
    row(SZA=75.0, VZA=70.0, RAA=0.0, HOT_Q=1e-3)
    row(SZA=0.0, VZA=0.0, RAA=0.0)                             # nadir
    row(RAA=360.0)
    row(SZA=75.0, VZA=70.0, RAA=180.0, AOT550=1.0, PA=500.0, UH2O=7.0)
    row(LAI=10.0, HOT_Q=1e-3, SZA=75.0, VZA=70.0, RAA=360.0, LIDFA=1.0, LIDFB=0.0)
    return np.array(rows)


def wide_batch(n, seed):
    """Half plain leaves, half PROSPECT-PRO leaves, then the deterministic rows."""
    return np.concatenate([wide_params(n // 2, seed), wide_params(n - n // 2, seed + 1, pro=True), oat_rows()])


# ---------------------------------------------------------------------------------- comparisons
def _max_abs(terms):
    """Largest magnitude over a list of broadcastable arrays."""
    return np.max(np.abs(np.broadcast_arrays(*terms)), axis=0)


def summand_scale(P, sensor, rv, canopy_ok, La):
    """[n, nb, 3] scale s of (R_TOC, R_TOA, L_TOA): the largest magnitude among the summands the output is
    formed of (SPART.py:235-252, smac.py:142-201).  rv: band canopy reflectances [n, nb, 4] (rso, rdo, rsd,
    rdd); a canopy reflectance outside (0, 1) (canopy_ok False) is itself a difference of O(1) terms and
    counts as at least 1.  La: band radiance scale [n, nb] (L_TOA = La R_TOA)."""
    info = so.load_sensor(sensor) if isinstance(sensor, str) else sensor
    atm = so.smac(P[:, so.SZA:so.RAA + 1], P[:, so.AOT550:so.PA + 1], info["SMAC_coef"], terms=True)
    r = np.abs(rv)
    r = np.where(canopy_ok[..., None], r, np.maximum(r, 1.0))
    rso, rdo, rsd, rdd = (r[..., i] for i in range(4))
    ta_ss, ta_oo = np.abs(atm["Ta_ss"]), np.abs(atm["Ta_oo"])
    # Ta_sd = Ta_s - Ta_ss, Ta_do = Ta_o - Ta_oo, Ta_s and Ta_o themselves sums (smac.py:125-126, 205-208)
    t_s, t_o = _max_abs(atm["Ta_s_terms"]), _max_abs(atm["Ta_o_terms"])
    ta_sd, ta_do = np.maximum(t_s, ta_ss), np.maximum(t_o, ta_oo)
    ra_dd, tg = np.abs(atm["Ra_dd"]), np.abs(atm["Tg"])
    with np.errstate(all="ignore"):
        den = np.abs(atm["Ta_ss"] + atm["Ta_sd"])
        toc = ((ta_ss * rso + ta_sd * rdo) + t_s * np.abs(rv[..., 0] * atm["Ta_ss"] + rv[..., 1] * atm["Ta_sd"]) / den) / den
        den = np.abs(1 - rv[..., 3] * atm["Ra_dd"])
        terms = list(atm["Ra_so_terms"])
        terms += [ta_ss * rso * ta_oo, (ta_sd * rdo + ta_ss * rsd * ra_dd * rdo) * ta_oo / den,
                  (ta_ss * rsd + ta_sd * rdd) * ta_do / den]
    toa = tg * _max_abs(terms)
    return np.stack([toc, toa, toa * np.abs(La)], axis=2)


def check_close(got, want, tol, scale=None, what="", max_scaled=MAX_SCALED):
    """Every output within tol relative, or -- only where `scale` is given -- within tol * scale absolute;
    the share that needed the absolute rule must stay below max_scaled.  NaN must meet NaN.  Returns that share."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, what
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN pattern differs"
    with np.errstate(all="ignore"):
        d = np.abs(got - want)
        rel_ok = (d <= tol * np.abs(want)) | nan | (got == want)
        ok = rel_ok if scale is None else rel_ok | (d <= tol * scale)
    if not ok.all():
        i = np.unravel_index(np.argmax(~ok), ok.shape)
        raise AssertionError(f"{what}: {np.count_nonzero(~ok)} of {ok.size} outputs off; first at {i}: "
                             f"got {got[i]!r} want {want[i]!r} rel {d[i] / abs(want[i]):.3e}"
                             + ("" if scale is None else f" scale {scale[i]:.3e}"))
    share = float(np.count_nonzero(~rel_ok)) / max(ok.size, 1)
    assert share <= max_scaled, f"{what}: {share:.2%} of the outputs are only absolutely accurate"
    return share


def oracle_bands(P, sensor, **kw):
    """Oracle outputs [n, nb, 3], band canopy reflectances, the (0, 1) canopy mask and the summand scale."""
    want, rv = so.spart_bands(P, sensor, return_canopy=True, **kw)
    ok = ((rv > 0) & (rv < 1)).all(axis=2)
    with np.errstate(all="ignore"):
        La = want[..., 2] / want[..., 1]
    La = np.where(np.isfinite(La), La, np.nanmax(np.abs(La), axis=0, keepdims=True))
    return want, ok, summand_scale(P, sensor, rv, ok, La)


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    return torch, spart_b200


def to_dev(torch, P):
    return torch.from_numpy(np.ascontiguousarray(P.T)).cuda()


def gpu(env, P, sensor, **kw):
    torch, sb = env
    out = sb.run_batch_params(to_dev(torch, P), sensor, **kw)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def test_generator_covers_the_domain():
    P = wide_batch(20000, 1)
    for col, lo, hi, _ in BOUNDS:
        assert P[:, col].min() >= lo and P[:, col].max() <= hi, col
        assert (P[:, col] == lo).any() and (P[:, col] == hi).any(), col
    ab = np.abs(P[:, so.LIDFA]) + np.abs(P[:, so.LIDFB])
    assert ab.max() <= 1.0 + 1e-15 and np.mean(ab >= 1.0 - 1e-12) > 0.04
    assert (P[:, so.SMP] <= 5).mean() > 0.03
    pro = (P[:, so.PROT] > 0) & (P[:, so.CDM] > 0)
    assert pro.mean() > 0.45
    # the dry-soil spectrum of the GSV box is non-negative at B = 1
    corners = np.array([[1, la, lo, 0, 25, 0] for la in (0, 20, 40) for lo in (50, 85, 120)], dtype=np.float64)
    assert so.bsm(corners, so.load_optical())[1].min() >= 0


@pytest.mark.parametrize("sensor", ["LANDSAT8-OLI", "TerraAqua-MODIS", "Sentinel3A-OLCI", "Sentinel2A-MSI"])
def test_band_kernel_general_geometry(env, sensor):
    """band_kernel<false>: ~20 000 samples per sensor (MODIS and OLCI have two-knot bands)."""
    P = wide_batch(20000, 100 + len(sensor))
    want, ok, s = oracle_bands(P, sensor)
    assert np.isfinite(want).all()
    got = gpu(env, P, sensor)
    check_close(got, want, RTOL64, s, sensor)


GEOMETRIES = [(sza, vza, raa) for sza in (0.0, 75.0) for vza in (0.0, 70.0) for raa in (0.0, 180.0, 360.0)]
GEOMETRIES.append((30.0, 30.0, 0.0))      # exact hot spot off nadir


@pytest.mark.parametrize("sensor", ["TerraAqua-MODIS", "Sentinel2A-MSI"])
def test_band_kernel_uniform_geometry(env, sensor):
    """band_kernel<true> on a grid of fixed geometries at the angle bounds: oracle and general path."""
    base = wide_batch(600, 200)
    for geo in GEOMETRIES:
        P = base.copy()
        P[:, so.SZA:so.RAA + 1] = geo
        want, ok, s = oracle_bands(P, sensor)
        a = gpu(env, P, sensor)
        b = gpu(env, P, sensor, uniform_geometry=True)
        check_close(b, want, RTOL64, s, f"{sensor} {geo} uniform vs oracle")
        check_close(b, a, 1e-12, s, f"{sensor} {geo} uniform vs general")


@pytest.mark.parametrize("sensor", ["LANDSAT8-OLI", "TerraAqua-MODIS", "Sentinel2A-MSI"])
def test_band_kernel_srf(env, sensor):
    """band_kernel_srf against the oracle's full-spectrum SRF convolution (the slow oracle path)."""
    P = wide_batch(300, 300 + len(sensor))
    want, ok, s = oracle_bands(P, sensor, band_mode="srf")
    got = gpu(env, P, sensor, band_mode="srf")
    check_close(got, want, RTOL64, s, sensor)


def test_spectrum_kernel(env):
    """spectrum_kernel: all nine spectra of forward_spectrum, NaN pattern included."""
    torch, sb = env
    P = wide_batch(240, 400)
    want = so.canopy_spectra(P)
    spec = sb.default_engine().forward_spectrum(to_dev(torch, P)).cpu().numpy()
    rv = np.stack([want[k] for k in ("rso", "rdo", "rsd", "rdd")], axis=2)      # [n, 2162, 4]
    canopy_ok = ((rv > 0) & (rv < 1)).all(axis=2)
    names = ["leaf_refl", "leaf_tran", "kChlrel", "soil_refl", "soil_refl_dry", "rso", "rdo", "rsd", "rdd"]
    for i, k in enumerate(names):
        w = want[k]
        got = spec[:, i, :w.shape[1]]
        scale = None
        if k in ("rso", "rdo", "rsd", "rdd"):
            scale = np.where(canopy_ok, np.abs(w), np.maximum(np.abs(w), 1.0))
        check_close(got, w, RTOL64, scale, k)


def plate_k(leaf, idx=slice(None)):
    """PROSPECT plate absorption K [n, nl] of leaf rows [n, 9] (prospect_5d.py:170-179) at wavelength indices idx."""
    opt = so.load_optical()
    leaf = np.array(leaf, dtype=np.float64)
    pro = ((leaf[:, 7] > 0) | (leaf[:, 8] > 0)) & (leaf[:, 1] > 0)
    leaf[pro, 1] = 0.0
    cols = ("Kab", "Kdm", "Kw", "Ks", "Kca", "Kant", None, "prot", "cbc")
    K = sum(leaf[:, i:i + 1] * opt[c][idx, 0][None, :] for i, c in enumerate(cols) if c)
    return K / leaf[:, 6:7]


def tau_piece(K):
    """Index of the plate_tau polynomial piece: K < 1, then [2^(j-1), 2^j) for j = 1..6, then [64, inf)."""
    return np.where(K < 1, 0, np.minimum(np.floor(np.log2(np.maximum(K, 1))) + 1, 7)).astype(int)


def prospect_rows():
    """Leaves whose plate absorption K falls into every piece of the plate_tau table, from K ~ 1e-13 up.
    Inside BOUNDS K stays below 21 (Cw = 0.1 gives 13 at 1926 nm, Cdm = 0.04 gives 4.4 at 400 nm), so the
    pieces [32, 64) and [64, inf) are reached with water columns beyond the leaf range, Cw up to 5 cm (K up to
    ~660) and N = 1.  No row lacks both water and dry matter: such a leaf is all but conservative in the
    near infrared (K < 1e-10), where the N-layer solution is ill-conditioned in 1 - r - t (the kernels and the
    reference then differ by a few 1e-9).  For N > 1 the power b ** (N - 1) of the N-layer solution (prospect_5d.py:219-230) overflows
    in both the reference and the kernels at such K.  Beyond K ~ 700 the plate transmissivity is subnormal and the
    oracle's (1 - K) e^-K + K^2 E1(K) is rounding noise (test_gpu_device_math tests the device value there)."""
    rows = []
    for cw in (0.0, 1e-4, 1e-3, 0.005, 0.02, 0.05, 0.1, 0.2, 0.5, 1.0, 2.0, 5.0):
        for cdm in ((0.004, 0.04) if cw == 0 else (0.0, 0.004, 0.04)):
            for n in ((1.0, 2.5, 4.0) if cw <= 0.1 else (1.0,)):
                rows.append([120.0 if cw > 0.05 else 5.0, cdm, cw, 1.5 if cdm > 0.01 else 0.0, 30.0, 40.0, n, 0, 0])
    rows.append([0.0, 0.04, 0.1, 0.0, 0.0, 0.0, 1.0, 0.003, 0.01])   # PROSPECT-PRO at its bounds
    return np.array(rows)


def test_prospect_all_tau_pieces(env):
    """prospect_batch: K in every piece of the FP64 plate_tau table, K >= 64 included (prospect_rows)."""
    _, sb = env
    leaf = prospect_rows()
    K = plate_k(leaf)
    pieces = np.bincount(tau_piece(K[K > 0]), minlength=8)
    assert (pieces > 50).all(), pieces
    refl, tran, kchl = sb.prospect_batch(leaf)
    w = so.prospect(leaf, so.load_optical())
    for got, want, name in zip((refl, tran, kchl), w, ("refl", "tran", "kChlrel")):
        check_close(got, want, RTOL64, what=name)


def test_fp32_plate_pieces_through_band_path(env):
    """The FP32 plate function through the FP32 band path of the 2001-band synthetic sensor (every wavelength a
    band): the prospect rows whose K stays below 87, where e^-K is still a normal float, against the FP64 oracle at
    the FP32 gate.  That reaches every piece of the table; test_gpu_device_math tests the function on its own."""
    _, sb = env
    leaf = prospect_rows()
    leaf = leaf[plate_k(leaf).max(axis=1) <= 87.0]
    K = plate_k(leaf)
    assert np.bincount(tau_piece(K[K > 0]), minlength=8).min() > 30
    P = np.repeat(DEFAULTS[None, :], leaf.shape[0], axis=0)
    P[:, :9] = leaf
    info = sb.synthetic_fullspectrum_sensorinfo()
    want, ok, s = oracle_bands(P, info)
    got = gpu(env, P, info, precision="fp32")
    assert np.isfinite(got).all()
    valid = np.broadcast_to(ok[..., None], got.shape)
    check_close(got[valid], want[valid], RTOL32, s[valid], "fp32 plate pieces")
    assert valid.mean() > 0.95


def test_bsm_moisture_grid(env):
    """bsm_batch: SMp x SMC x film grid, dry branch (SMp <= 5) and Poisson means up to 19."""
    _, sb = env
    g = np.array([(b, la, lo, smp, smc, film)
                  for b, la, lo in ((0.5, 0.0, 100.0), (1.0, 40.0, 50.0), (0.05, 20.0, 120.0))
                  for smp in (0.0, 4.999, 5.0, 5.001, 20.0, 55.0, 100.0)
                  for smc in (5.0, 12.0, 25.0, 60.0)
                  for film in (0.0, 1e-4, 0.015, 0.05, 0.1)], dtype=np.float64)
    wet, dry = sb.bsm_batch(g)
    w_wet, w_dry = so.bsm(g, so.load_optical())
    check_close(dry, w_dry, RTOL64, what="dry")
    check_close(wet, w_wet, RTOL64, what="wet")
    assert (wet[g[:, 3] <= 5] == dry[g[:, 3] <= 5]).all()


@pytest.mark.parametrize("sensor", ["Sentinel2A-MSI", "TerraAqua-MODIS", "Sentinel3B-OLCI"])
def test_smac_bounds(env, sensor):
    """smac_batch at the angle, AOT, UH2O and PA bounds (and random rows inside them)."""
    _, sb = env
    grid = np.array([(sza, vza, raa, aot, 0.35, uh2o, pa)
                     for sza in (0.0, 40.0, 75.0) for vza in (0.0, 70.0) for raa in (0.0, 90.0, 360.0)
                     for aot in (0.0, 1.0) for uh2o in (0.0, 7.0) for pa in (500.0, 1050.0)], dtype=np.float64)
    P = np.repeat(DEFAULTS[None, :], grid.shape[0], axis=0)
    P[:, so.SZA:so.RAA + 1], P[:, so.AOT550:so.PA + 1] = grid[:, :3], grid[:, 3:]
    P = np.concatenate([P, wide_params(2000, 500)])
    info = so.load_sensor(sensor)
    want = so.smac(P[:, so.SZA:so.RAA + 1], P[:, so.AOT550:so.PA + 1], info["SMAC_coef"], terms=True)
    got = sb.smac_batch(P[:, so.SZA:so.RAA + 1], P[:, so.AOT550:so.PA + 1], sensor)
    terms = _max_abs(want["Ra_so_terms"])
    for i, k in enumerate(sb.stages.ATM_FIELDS):
        w = np.broadcast_to(want[k], got[:, i].shape)
        scale = None
        if k == "Ra_so":
            scale = terms
        elif k in ("Ta_sd", "Ta_do"):      # Ta_s - Ta_ss, Ta_o - Ta_oo
            s, d = ("Ta_s", "Ta_ss") if k == "Ta_sd" else ("Ta_o", "Ta_oo")
            scale = np.maximum(_max_abs(want[s + "_terms"]), np.abs(want[d]))
        check_close(got[:, i], w, RTOL64, scale, k)


def test_sailh_lidf_boundary_and_small_q(env):
    """sailh_batch: (LIDFa, LIDFb) on the edge of |a| + |b| <= 1, q = 1e-3, zenith angles at their bounds."""
    _, sb = env
    t = np.linspace(-1, 1, 21)
    ab = np.concatenate([np.stack([t, 1 - np.abs(t)], 1), np.stack([t, np.abs(t) - 1], 1)])
    canopy = np.array([(lai, a, b, q) for a, b in ab for lai in (0.5, 4.0, 10.0) for q in (1e-3, 0.05)])
    angles = np.array([(75.0, 70.0, 0.0), (40.0, 0.0, 0.0), (75.0, 70.0, 180.0), (30.0, 30.0, 0.0)])
    canopy = np.repeat(canopy, len(angles), axis=0)
    angles = np.tile(angles, (len(canopy) // len(angles), 1))
    P = np.repeat(DEFAULTS[None, :], 1, axis=0)
    cs = so.canopy_spectra(P)
    soil, rho, tau = cs["soil_refl"][0], cs["leaf_refl"][0], cs["leaf_tran"][0]
    got = sb.sailh_batch(soil, rho, tau, canopy, angles)
    rep = lambda x: np.repeat(x[None, :], len(canopy), 0)
    want = np.stack(so.sailh(rep(soil), rep(rho), rep(tau), canopy, angles), axis=1)
    ok = ((want > 0) & (want < 1)).all(axis=1, keepdims=True)
    check_close(got, want, RTOL64, np.where(ok, np.abs(want), np.maximum(np.abs(want), 1.0)), "sailh")


def band_plate_k(P, sensor):
    """Largest plate absorption K [n, nb] over the wavelengths np.interp samples for each band."""
    info = so.load_sensor(sensor) if isinstance(sensor, str) else sensor
    lo, hi, _ = so.band_sample_points(info["wl_smac"].T[0])
    K = plate_k(P[:, :9], np.concatenate([lo, hi]))
    return np.maximum(K[:, :lo.size], K[:, lo.size:])


@pytest.mark.parametrize("sensor", ["LANDSAT8-OLI", "TerraAqua-MODIS", "Sentinel2A-MSI", "Sentinel3A-OLCI"])
def test_fp32_mode(env, sensor):
    """FP32 mode on the wide batches against the FP64 oracle at its gate, on physically valid outputs
    (all four band canopy reflectances in (0, 1))."""
    P = wide_batch(20000, 600 + len(sensor))
    want, ok, s = oracle_bands(P, sensor)
    got = gpu(env, P, sensor, precision="fp32")
    assert np.isfinite(got).all()
    assert ok.mean() > 0.98
    valid = np.broadcast_to(ok[..., None], got.shape)
    check_close(got[valid], want[valid], RTOL32, s[valid], f"{sensor} fp32")


def test_fp32_strong_absorption(env):
    """Leaves at the upper pigment and dry-matter bounds with N slightly above 1: at MODIS band 8 (412 nm) the plate
    absorbs K > 14.5 and tau < 5e-8, below float resolution of 1.  FP32 mode forms tau directly there; the
    difference 1 - (1 - tau) would round to 0 and make b ** (N - 1) infinite (NaN leaf optics)."""
    P = np.repeat(DEFAULTS[None, :], 4, axis=0)
    P[:, so.CAB], P[:, so.CCA], P[:, so.CANT], P[:, so.CS], P[:, so.CDM] = 120.0, 30.0, 40.0, 1.5, 0.04
    P[:, so.NSTRUCT] = [1.005, 1.01, 1.02, 1.03]
    assert band_plate_k(P, "TerraAqua-MODIS")[:, 7].min() > 14.5
    want, ok, s = oracle_bands(P, "TerraAqua-MODIS")
    got = gpu(env, P, "TerraAqua-MODIS", precision="fp32")
    assert np.isfinite(got).all() and ok.all()
    check_close(got, want, RTOL32, s, "fp32 strong absorption")
