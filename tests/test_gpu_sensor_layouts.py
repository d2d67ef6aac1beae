"""Custom sensorinfo dicts (SPART.sensorinfo, build_sensor) at the edges of the sensor layout, against the oracle.

Interp mode: band centres on and next to the grid ends and a hair off an integer, band counts on both sides
of the 16-band chunk of the band kernels (kBandChunk), batches on both sides of the 128-sample tile.
SRF mode: accumulator-slot plans at and beyond the 24-slot limit (kSrfMaxSlots), single-wavelength SRFs,
SRF samples at and beyond 400 / 2400 nm, and a band whose weights are all zero."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import spart_oracle as so  # noqa: E402
from test_gpu_domain import RTOL64, check_close, gpu, oracle_bands, wide_batch  # noqa: E402

SPECIAL_CENTRES = [400.0, 400.5, 2399.5, 2400.0, 401.0 - 1e-9, 401.0 + 1e-9, 1250.0 - 1e-9, 1250.0 + 1e-9,
                   2399.0 + 1e-9, 2400.0 - 1e-9, 865.0, 1610.4]


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    return torch, spart_b200


def smac_coef_at(centres):
    """SMAC coefficients at `centres`, linear in wavelength between the TerraAqua-MODIS bands (the way
    synthetic_fullspectrum_sensorinfo builds its 2001 bands)."""
    modis = so.load_sensor("TerraAqua-MODIS")
    wl = modis["wl_smac"].T[0].astype(np.float64)
    order = np.argsort(wl)
    return {k: np.interp(centres, wl[order], v[0].astype(np.float64)[order])[None, :]
            for k, v in modis["SMAC_coef"].items()}


def sensorinfo(centres, wl_srf=None, p_srf=None):
    """A sensorinfo dict with the reference's keys; default SRF: one sample at the rounded centre."""
    centres = np.asarray(centres, dtype=np.float64)
    if wl_srf is None:
        wl_srf, p_srf = np.round(centres)[None, :], np.ones((1, centres.size))
    return {"SMAC_coef": smac_coef_at(centres), "wl_smac": centres[:, None], "wl_srf_smac": np.asarray(wl_srf, float),
            "p_srf_smac": np.asarray(p_srf, float), "band_id_smac": [f"b{i}" for i in range(centres.size)]}


def layout_centres(nb, seed):
    """nb band centres: the special ones first (rotated so that every count starts elsewhere), then random
    fractional centres; unsorted, as in the MODIS tables."""
    rng = np.random.default_rng(seed)
    sp = np.roll(SPECIAL_CENTRES, seed)
    c = np.concatenate([sp, rng.uniform(400, 2400, max(nb - sp.size, 0))])[:nb]
    return rng.permutation(c)


@pytest.mark.parametrize("nb", [1, 15, 16, 17, 31, 32, 33])
def test_interp_layouts(env, nb):
    """band_kernel<false> and <true> on custom layouts, n = 1, 127, 128, 129, 1000."""
    info = sensorinfo(layout_centres(nb, nb))
    for n in (1, 127, 128, 129, 1000):
        P = wide_batch(n, 10 * nb + n)[:n]
        want, ok, s = oracle_bands(P, info)
        check_close(gpu(env, P, info), want, RTOL64, s, f"nb={nb} n={n} general")
        P[:, so.SZA:so.RAA + 1] = (57.5, 33.0, 123.0)
        want, ok, s = oracle_bands(P, info)
        check_close(gpu(env, P, info, uniform_geometry=True), want, RTOL64, s, f"nb={nb} n={n} uniform")


def test_interp_special_centres_faithful(env):
    """The special centres against the reference's own np.interp over the full spectrum (faithful=True)."""
    info = sensorinfo(np.array(SPECIAL_CENTRES))
    P = wide_batch(200, 7)
    got = gpu(env, P, info)
    want, ok, s = oracle_bands(P, info)
    check_close(got, want, RTOL64, s, "sampled")
    check_close(got, so.spart_bands(P, info, faithful=True), RTOL64, s, "faithful")


def gaussian_srfs(nb, start=1000.0, step=2.0, sigma=10.0, half=30):
    """nb Gaussian SRFs, centres start + step * b, sampled every nm over +-half nm: every band overlaps every
    other one when step * (nb - 1) < 2 half."""
    centres = start + step * np.arange(nb)
    off = np.arange(-half, half + 1, dtype=np.float64)
    wl = centres[None, :] + off[:, None]
    return centres, wl, np.exp(-0.5 * (off[:, None] / sigma) ** 2) * np.ones((1, nb))


def srf_slots(sb, info):
    """Accumulator slots spart_create's interval colouring needs: the largest number of bands whose SRF
    support (first .. last weighted wavelength) contains a wavelength, plus the spare slot."""
    st = sb.tables.build_sensor("custom", info)
    off = np.concatenate([[0], np.cumsum(st.srf_len)])
    open_at = np.zeros(2001, dtype=int)
    for b in range(st.n_bands):
        idx = st.srf_idx[off[b]:off[b + 1]]
        if idx.size:
            open_at[idx.min():idx.max() + 1] += 1
    return int(open_at.max()) + 1


def srf_check(env, info, n=200, seed=11):
    P = wide_batch(n, seed)[:n]
    want, ok, s = oracle_bands(P, info, band_mode="srf")
    got = gpu(env, P, info, band_mode="srf")
    check_close(got, want, RTOL64, s, "srf")
    torch, sb = env
    host = sb.run_batch_params(np.ascontiguousarray(P.T), info, band_mode="srf")
    assert np.array_equal(host, got, equal_nan=True)
    return got, want


@pytest.mark.parametrize("nb,slots", [(22, 23), (23, 24)])
def test_srf_slot_limit(env, nb, slots):
    """Overlapping Gaussian SRFs whose colouring needs 23 and 24 slots (the limit), spare included."""
    _, sb = env
    centres, wl, p = gaussian_srfs(nb)
    info = sensorinfo(centres, wl, p)
    assert srf_slots(sb, info) == slots
    srf_check(env, info)


def test_srf_too_many_slots(env):
    """25 slots: spart_create refuses the sensor, and releases what it had already allocated (the refusal
    comes from the SRF planner, after the wavelength, band and knot tables are on the device)."""
    torch, sb = env
    centres, wl, p = gaussian_srfs(24)
    info = sensorinfo(centres, wl, p)
    assert srf_slots(sb, info) == 25
    eng = sb.default_engine()
    with pytest.raises(sb.SpartError, match="too many overlapping bands"):
        eng.sensor(info)
    free0 = torch.cuda.mem_get_info(eng.device)[0]
    for _ in range(200):
        with pytest.raises(sb.SpartError, match="too many overlapping bands"):
            eng.sensor(info)
    # a leak would keep at least the 272 KB wavelength table per refusal, about 54 MB in all
    assert abs(torch.cuda.mem_get_info(eng.device)[0] - free0) <= 2 << 20


def test_srf_single_wavelength_ends_and_zero_weight(env):
    """A single-wavelength SRF, SRF samples at and beyond the 400 / 2400 nm ends (the nearest grid point is
    the end), Gaussian bands, and bands whose weights are all zero: the reference's 0 / 0 makes all three
    outputs of those NaN (calculate_spectral_convolution, SPART.py:389-396)."""
    nsrf = 9
    cols = []

    def band(wls, ps):
        w, q = np.full(nsrf, 1000.0), np.zeros(nsrf)
        w[:len(wls)], q[:len(ps)] = wls, ps
        cols.append((w, q))
    band([865.0], [1.0])                                               # single wavelength
    band([390.0, 395.0, 399.6, 400.0, 400.4, 401.0], [1, 2, 3, 4, 5, 6])   # at and below 400 nm
    band([2398.0, 2399.6, 2400.0, 2400.4, 2405.0, 2500.0], [1, 1, 2, 2, 3, 3])   # at and beyond 2400 nm
    band([650.0, 660.0, 670.0], [0.0, 0.0, 0.0])                       # all weights zero
    band(np.linspace(1500, 1580, nsrf), np.exp(-0.5 * np.linspace(-2, 2, nsrf) ** 2))
    band([900.0, 901.0], [0.0, 0.0])                                   # a second empty band
    band([2000.0, 2000.2, 2000.4], [1.0, 0.5, 0.25])                   # samples sharing one grid point
    wl = np.stack([c[0] for c in cols], axis=1)
    p = np.stack([c[1] for c in cols], axis=1)
    info = sensorinfo(np.array([865.0, 400.0, 2400.0, 660.0, 1540.0, 900.5, 2000.0]), wl, p)
    got, want = srf_check(env, info, n=300, seed=12)
    empty = np.array([3, 5])
    assert np.isnan(want[:, empty]).all() and np.isnan(got[:, empty]).all()
    full = np.setdiff1d(np.arange(7), empty)
    assert np.isfinite(got[:, full]).all()
    # the empty bands do not disturb the others: the same bands without them
    keep = full
    info2 = sensorinfo(info["wl_smac"][keep, 0], wl[:, keep], p[:, keep])
    _, sb = env
    P = wide_batch(300, 12)[:300]
    assert np.array_equal(gpu(env, P, info2, band_mode="srf"), got[:, keep])
    # the soil-library twin of the SRF kernel walks the same plan: per library row, the bits of the
    # soil_spectrum= run, NaN bands included, and the oracle for that row
    soils = np.array([[1.0, 20.0, 85.0, 0.0, 25.0, 0.0], [0.4, 5.0, 110.0, 0.0, 25.0, 0.0]])
    lib = sb.SoilLibrary(so.bsm(soils, so.load_optical())[1])
    idx = np.arange(300) % 2
    Pl = P.copy()
    Pl[:, so.SOIL_B] = idx
    lgot = gpu(env, Pl, info, band_mode="srf", soil_library=lib)
    for i in range(2):
        one = gpu(env, Pl, info, band_mode="srf", soil_spectrum=lib.spectra[i])
        assert np.array_equal(lgot[idx == i], one[idx == i], equal_nan=True)
    assert np.isnan(lgot[:, empty]).all() and np.isfinite(lgot[:, full]).all()
    rows = idx == 1
    want, ok, s = oracle_bands(Pl[rows], info, band_mode="srf", soil_rdry=lib.spectra[1])
    check_close(lgot[rows], want, RTOL64, s, "srf soil library")
