"""Pin the NumPy oracle (oracle/spart_oracle.py) against outputs of the unmodified
reference recorded by tools/make_golden.py (O1 = raw, O2 = exact-E1 variant)."""
import numpy as np
import pytest

import spart_oracle as so
from conftest import golden_columns, load_golden, relerr

BATCHES = ["cfg2_S2A", "cfg3_L8", "cfg5_S2B", "rand_MODIS", "rand_OLCI", "rand_L7"]


@pytest.mark.parametrize("name", BATCHES)
def test_oracle_matches_reference_batches(name, optical):
    g = load_golden(f"batch_{name}.npz")
    sensor = str(g["sensor"])
    out = so.spart_bands(g["params"], sensor, optical)
    assert out.shape == g["O2"].shape
    # O2 (reference with exact E1): the oracle is the same arithmetic -> rounding level
    assert relerr(out, g["O2"]) < 1e-12
    # O1 (raw reference): bounded by its own QUADPACK tolerance (SURVEY.md 8(c): <= 8.1e-9)
    assert relerr(out, g["O1"]) < 5e-8
    # and well inside the tolerance the reference's own golden tests accept (1.5e-7 abs)
    assert np.max(np.abs(out[..., :2] - g["O1"][..., :2])) < 1.5e-7


def test_oracle_faithful_equals_fast(optical):
    g = load_golden("batch_rand_MODIS.npz")
    P = g["params"][:6]
    a = so.spart_bands(P, "TerraAqua-MODIS", optical, faithful=True)
    b = so.spart_bands(P, "TerraAqua-MODIS", optical, faithful=False)
    assert relerr(b, a) < 1e-13
    assert relerr(a, g["O2"][:6]) < 1e-12


@pytest.mark.parametrize("sensor", so.SENSORS)
def test_oracle_e2e_defaults(sensor, optical):
    """tests/e2e/test_SPART.py of the reference: conftest defaults on all nine sensors."""
    g = load_golden("e2e.npz")
    out = so.spart_bands(g["params_defaults"][None, :], sensor, optical)[0]
    assert (out > 0).all()                      # the reference's own assertion
    assert relerr(out, g[f"{sensor}.O2"]) < 1e-12
    assert relerr(out, g[f"{sensor}.O1"]) < 5e-8


def test_oracle_readme_quickstart(optical):
    g = load_golden("e2e.npz")
    out = so.spart_bands(g["params_readme"][None, :], "TerraAqua-MODIS", optical)[0]
    assert np.isfinite(out).all()
    assert relerr(out, g["README.O2"]) < 1e-12
    assert relerr(out, g["README.O1"]) < 5e-8


def test_oracle_spectra(optical):
    g = load_golden("spectra.npz")
    cs = so.canopy_spectra(g["params"], optical)
    for k in ("leaf_refl", "leaf_tran", "kChlrel", "soil_refl", "soil_refl_dry", "rso", "rdo", "rsd", "rdd"):
        ref = g[f"O2.{k}"]
        got = golden_columns(cs[k], g)
        assert got.shape == ref.shape
        assert (np.isnan(got) == np.isnan(ref)).all(), k
        assert relerr(got, ref) < 1e-11, k
        # raw reference: the reference's accepted tolerances (test_PROSPECT decimal=7, test_SAILH decimal=6)
        o1 = g[f"O1.{k}"]
        ok = ~np.isnan(o1)
        assert np.max(np.abs(got[ok] - o1[ok])) < 1.5e-7, k
    lidf = so.leafangles(g["params"][:, so.LIDFA], g["params"][:, so.LIDFB])
    assert relerr(lidf, g["O1.lidf"]) < 1e-12


def test_oracle_prospect_grid(optical):
    """Subset of the reference's PROSPECT unit-test grid (build_PROSPECT_tests.py:38-50)."""
    g = load_golden("prospect_grid.npz")
    leaf = np.zeros((g["leaf7"].shape[0], 9))
    leaf[:, :7] = g["leaf7"]
    refl, tran, kchl = so.prospect(leaf, optical)
    got = golden_columns(np.stack([refl, tran, kchl], axis=1), g)
    assert relerr(got, g["O2"]) < 1e-11
    np.testing.assert_almost_equal(got, g["O1"], decimal=7)   # the reference's own criterion


def test_oracle_sailh_grid(optical):
    """Subset of the reference's SAILH unit-test grid (build_SAILH_tests.py:87-101)."""
    g = load_golden("sailh_grid.npz")
    c7 = g["canopy_angles7"]
    n = c7.shape[0]
    rs, rho, tau = (np.repeat(g[k][None, :], n, 0) for k in ("soil_refl", "leaf_refl", "leaf_tran"))
    lidf = so.leafangles(c7[:, 1], c7[:, 2])
    assert relerr(lidf, g["lidf"]) < 1e-12
    got = golden_columns(np.stack(so.sailh(rs, rho, tau, c7[:, :4], c7[:, 4:7]), axis=1), g)
    ok = np.isfinite(g["O1"])
    assert (np.isfinite(got) == ok).all()
    assert relerr(got[ok], g["O1"][ok]) < 1e-9
    np.testing.assert_array_almost_equal(got[ok], g["O1"][ok], decimal=6)  # reference's criterion


def test_oracle_cfg4_synthetic_sensor(optical):
    g = load_golden("batch_cfg4_SYNTH2001.npz")
    sensor = so.synthetic_fullspectrum_sensor()
    out = so.spart_bands(g["params"], sensor, optical)
    assert out.shape == (g["params"].shape[0], 2001, 3)
    assert relerr(out, g["O2"]) < 1e-11
    assert relerr(out, g["O1"]) < 1e-6


@pytest.mark.parametrize("name", ["soilfile_Sentinel2A", "soilfile_TerraAqua"])
def test_oracle_user_soil_spectrum(name, optical):
    """SoilParametersFromFile path of the reference (bsm.py:42-43, 155-226)."""
    g = load_golden(f"{name}.npz")
    out = so.spart_bands(g["params"], str(g["sensor"]), optical, soil_rdry=g["rdry"])
    assert relerr(out, g["O2"]) < 1e-12
    assert relerr(out, g["O1"]) < 5e-8


def test_closest_index_semantics():
    """get_closest_index (SPART.py:381-387): ties -> lower index, NaN -> 0."""
    wl_hi = np.arange(400, 2401)
    wl = np.array([[350.0, 400.5], [np.nan, 2400.49], [2500.0, 1000.0]])
    idx = so.closest_index(wl, wl_hi)
    assert idx.tolist() == [[0, 0], [0, 2000], [2000, 600]]


def test_oracle_bare_soil_rows(optical):
    """LAI = 0 and LAI -> 0 rows recorded from the unmodified reference (sailh.py:112-114)."""
    g = load_golden("edge_lai0.npz")
    got = so.spart_bands(g["params"], str(g["sensor"]), optical)
    assert np.isfinite(g["O1"]).all()
    assert relerr(got, g["O2"]) < 1e-12
    assert relerr(got, g["O1"]) < 5e-8


@pytest.mark.parametrize("name", ["srf_Sentinel2A", "srf_LANDSAT8", "srf_TerraAqua"])
def test_oracle_srf_band_mode_is_the_references_convolution(name, optical):
    """band_mode="srf" against the reference's own calculate_spectral_convolution (SPART.py:358-396)
    applied to the canopyopt of a reference run, followed by the reference's atmopt and TOC->TOA algebra
    (recorded by tools/make_golden.py::run_srf)."""
    g = load_golden(f"{name}.npz")
    got = so.spart_bands(g["params"], str(g["sensor"]), optical, band_mode="srf")
    assert relerr(got, g["O2"]) < 1e-12
    assert relerr(got, g["O1"]) < 5e-8


def test_oracle_user_assigned_lidf(optical):
    """A leaf inclination distribution assigned after construction (canopy.lidf = ...) is used by SAILH as is
    (sailh.py:81-97): rows recorded from the unmodified reference (tools/make_golden.py::run_userlidf)."""
    g = load_golden("user_lidf.npz")
    got = so.spart_bands(g["params"], str(g["sensor"]), optical, lidf=g["lidf"])
    assert relerr(got, g["O2"]) < 1e-12
    assert relerr(got, g["O1"]) < 5e-8
    assert relerr(so.spart_bands(g["params"], str(g["sensor"]), optical), g["O2"]) > 1e-3      # the override matters
