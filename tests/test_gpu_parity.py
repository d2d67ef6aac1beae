"""Parity of the CUDA path (called through the C ABI) against the oracle and the golden
fixtures recorded from the unmodified reference.

FP64 gate (BASELINE.json north_star): relative error <= 1e-9 against the reference's
documented arithmetic (O2 / oracle).  Against the raw reference (O1) the bound is the
reference's own QUADPACK noise, <= 5e-8 relative and inside the 1.5e-7 absolute tolerance
of the reference's unit tests (SURVEY.md section 8(c))."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from conftest import golden_columns, load_golden, relerr  # noqa: E402

RTOL64 = 1e-9
RTOL32 = 1e-4      # FP32 mode (BASELINE.json north_star)


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    import spart_oracle as so
    assert torch.cuda.is_available()
    return torch, spart_b200, so


def gpu_bands(env, P, sensor, precision="fp64"):
    torch, sb, _ = env
    dev = torch.from_numpy(np.ascontiguousarray(np.asarray(P, dtype=np.float64).T)).cuda()
    out = sb.run_batch_params(dev, sensor, precision=precision)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("name", ["cfg2_S2A", "cfg3_L8", "cfg5_S2B", "rand_MODIS", "rand_OLCI", "rand_L7"])
def test_bands_vs_reference_golden(env, name):
    g = load_golden(f"batch_{name}.npz")
    got = gpu_bands(env, g["params"], str(g["sensor"]))
    assert got.shape == g["O2"].shape
    assert relerr(got, g["O2"]) < RTOL64
    assert relerr(got, g["O1"]) < 5e-8
    assert np.max(np.abs(got[..., :2] - g["O1"][..., :2])) < 1.5e-7


@pytest.mark.parametrize("sensor,cfg", [("Sentinel2A-MSI", 2), ("LANDSAT8-OLI", 3), ("TerraAqua-MODIS", 3),
                                        ("Sentinel3B-OLCI", 3), ("LANDSAT5-TM", 2), ("Sentinel2B-MSI", 5)])
def test_bands_vs_oracle_random(env, sensor, cfg):
    _, _, so = env
    P = so.synthetic_params(2000, cfg, seed=1000 + cfg)
    want = so.spart_bands(P, sensor)
    got = gpu_bands(env, P, sensor)
    assert relerr(got, want) < RTOL64


def _fp32_report(env, P, sensor):
    _, _, so = env
    want, canopy = so.spart_bands(P, sensor, return_canopy=True)
    got = gpu_bands(env, P, sensor, precision="fp32")
    with np.errstate(all="ignore"):
        e = np.abs(got - want) / np.abs(want)
    # physically valid SAILH output: all four canopy reflectances inside (0, 1).  Outside that
    # range (the reference returns rso < 0 or rdd > 1 for near-conservative leaves under dense
    # canopies) R_TOC is a difference of O(1) terms and no single-precision evaluation can be
    # relatively accurate.
    valid = ((canopy > 0) & (canopy < 1)).all(axis=2)
    return got, want, e, valid


@pytest.mark.parametrize("sensor,cfg", [("Sentinel2A-MSI", 2), ("Sentinel2B-MSI", 5), ("LANDSAT7-ETM", 2),
                                        ("Sentinel2A-MSI", 4)])
def test_fp32_mode_lut_configs(env, sensor, cfg):
    """FP32 mode on the fixed-geometry LUT distributions of BASELINE.json (configs 2, 4, 5):
    relative error <= 1e-4 on EVERY output against the FP64 oracle."""
    _, _, so = env
    P = so.synthetic_params(50000, cfg, seed=2000 + cfg)
    got, want, e, valid = _fp32_report(env, P, sensor)
    assert np.isfinite(got).all()
    assert e.max() < RTOL32


@pytest.mark.parametrize("sensor", ["LANDSAT8-OLI", "TerraAqua-MODIS", "Sentinel3A-OLCI"])
def test_fp32_mode_random_geometry(env, sensor):
    """FP32 mode with random sun/view angles and PROSPECT-PRO leaves (config 3): relative error
    <= 1e-4 on every physically valid output.  Near-conservative leaves (rho + tau > 0.98) under dense
    canopies make the canopy solution ill-conditioned in the leaf absorptance; the FP32 mode carries
    1 - rho - tau from a FP64 Stokes solve and uses cancellation-free SAIL forms (tools/fp32_study.py)."""
    _, _, so = env
    P = so.synthetic_params(50000, 3, seed=2003)
    got, want, e, valid = _fp32_report(env, P, sensor)
    assert valid.mean() > 0.99
    assert e[valid].max() < RTOL32


def test_fp32_mode_goldens_and_edges(env):
    _, sb, so = env
    for name in ("cfg2_S2A", "cfg5_S2B"):
        g = load_golden(f"batch_{name}.npz")
        got = gpu_bands(env, g["params"], str(g["sensor"]), precision="fp32")
        assert relerr(got, g["O1"]) < RTOL32
    P = so.synthetic_params(64, 2, seed=77)
    P[0:8, so.SMP] = [0.0, 4.99, 5.0, 5.01, 3.0, 1.0, 5.0, 2.0]                 # dry-soil branch
    P[8:16, so.PROT], P[8:16, so.CBC] = 0.001, 0.004                           # PROSPECT-PRO switch (Cdm > 0)
    P[16:24, so.SZA], P[16:24, so.VZA] = 30.0, 30.0                            # exact hot spot
    P[24:28, so.RAA] = [180.0, 360.0, 540.0, 270.0]
    P[28:32, so.SZA] = 0.0
    P[32:36, so.LAI] = [1e-2, 0.05, 10.0, 15.0]
    P[36:40, so.SZA] = 30.0
    P[36:40, so.VZA] = 30.0 + np.array([1e-4, 1e-3, 1e-2, 0.1])                # almost in the hot spot
    got, want, e, valid = _fp32_report(env, P, "LANDSAT8-OLI")
    assert np.isfinite(got).all()
    ev = np.where(valid[..., None], e, 0.0)
    worst = np.unravel_index(np.argmax(ev), ev.shape)
    # branch / geometry edge cases, LAI 0.01 ... 15, near-hot-spot rows
    assert ev.max() < RTOL32, f"row {worst[0]} band {worst[1]} output {worst[2]}: {ev.max():.3e}"
    # uniform-geometry flag and host path in FP32 mode
    P = so.synthetic_params(3000, 2, seed=5)
    pt = np.ascontiguousarray(P.T)
    a = sb.run_batch_params(pt, "Sentinel2A-MSI", precision="fp32")
    b = sb.run_batch_params(pt, "Sentinel2A-MSI", precision="fp32", uniform_geometry=True)
    assert relerr(b, a) < 1e-5
    assert relerr(b, so.spart_bands(P, "Sentinel2A-MSI")) < RTOL32


def test_e2e_defaults_all_sensors(env):
    """The reference's e2e test (tests/e2e/test_SPART.py) through the reference-shaped API."""
    _, sb, so = env
    g = load_golden("e2e.npz")
    for sensor in so.SENSORS:
        spart = sb.SPART(sb.SoilParameters(0.5, 0, 100, 20, 25, 0.015), sb.LeafBiology(40, 0.01, 0.02, 0, 10, 10, 1.5),
                         sb.CanopyStructure(3, -0.35, -0.15, 0.05), sb.AtmosphericProperties(0.325, 0.35, 1.41),
                         sb.Angles(40, 0, 0), sensor, 100)
        res = spart.run()
        assert list(res.columns) == ["Band", "L_TOA", "R_TOA", "R_TOC"]
        assert (res["L_TOA"] > 0).all() and (res["R_TOA"] > 0).all() and (res["R_TOC"] > 0).all()
        got = np.stack([res["R_TOC"].to_numpy(), res["R_TOA"].to_numpy(), res["L_TOA"].to_numpy()], axis=1)
        assert relerr(got, g[f"{sensor}.O2"]) < RTOL64
        assert relerr(got, g[f"{sensor}.O1"]) < 5e-8


def test_readme_quickstart(env):
    _, sb, _ = env
    g = load_golden("e2e.npz")
    spart = sb.SPART(sb.SoilParameters(0.5, 0, 100, 15, 25, 0.015), sb.LeafBiology(40, 10, 0.02, 0.01, 0, 10, 1.5),
                     sb.CanopyStructure(3, -0.35, -0.15, 0.05), sb.AtmosphericProperties(0.3246, 0.3480, 1.4116, 1013.25),
                     sb.Angles(40, 0, 0), "TerraAqua-MODIS", 100)
    res = spart.run()
    got = np.stack([res["R_TOC"].to_numpy(), res["R_TOA"].to_numpy(), res["L_TOA"].to_numpy()], axis=1)
    assert np.isfinite(got).all()
    assert relerr(got, g["README.O2"]) < RTOL64
    assert res.index.to_numpy().tolist() == pytest.approx(sb.load_sensor_info("TerraAqua-MODIS")["wl_smac"].T[0].tolist())


def test_spectra_vs_reference_golden(env):
    torch, sb, so = env
    g = load_golden("spectra.npz")
    P = g["params"]
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    spec = sb.default_engine().forward_spectrum(dev).cpu().numpy()
    names = ["leaf_refl", "leaf_tran", "kChlrel", "soil_refl", "soil_refl_dry", "rso", "rdo", "rsd", "rdd"]
    for i, k in enumerate(names):
        ref = g[f"O2.{k}"]
        got = golden_columns(spec[:, i, :2001 if k in ("kChlrel", "soil_refl_dry") else spec.shape[2]], g)
        assert got.shape == ref.shape, k
        assert (np.isnan(got) == np.isnan(ref)).all(), k
        assert relerr(got, ref) < RTOL64, k
        o1 = g[f"O1.{k}"]
        ok = ~np.isnan(o1)
        assert np.max(np.abs(got[ok] - o1[ok])) < 1.5e-7, k


def test_leafangles(env):
    _, sb, so = env
    rng = np.random.default_rng(5)
    ab = np.stack([rng.uniform(-1, 1, 4000), rng.uniform(-1, 1, 4000)], axis=1)
    ab = ab[np.abs(ab).sum(1) <= 1.0]
    ab = np.concatenate([ab, [[-0.35, -0.15], [0.0, 0.0], [1.0, 0.0], [-1.0, 0.0], [0.0, 1.0], [0.0, -1.0]]])
    want = so.leafangles(ab[:, 0], ab[:, 1])
    got = sb.default_engine().leafangles(ab)
    assert np.max(np.abs(got - want)) < 1e-12
    g = load_golden("sailh_grid.npz")
    got = sb.default_engine().leafangles(g["canopy_angles7"][:, 1:3])
    assert np.max(np.abs(got - g["lidf"])) < 1e-12


def test_host_path_equals_device_path(env):
    _, sb, so = env
    P = so.synthetic_params(5000, 3, seed=9)
    dev = gpu_bands(env, P, "LANDSAT8-OLI")
    pt = np.ascontiguousarray(P.T)
    host = sb.run_batch_params(pt, "LANDSAT8-OLI")
    assert np.array_equal(host, dev)
    # strided rows (ld > n): a column window of a larger block
    big = np.zeros((27, 7000))
    big[:, 1000:6000] = pt
    host2 = sb.run_batch_params(big[:, 1000:6000], "LANDSAT8-OLI")
    assert np.array_equal(host2, dev)


def test_edge_cases(env):
    """Empty and single-sample batches, dry soil branch (bsm.py:102-103), PROSPECT-PRO switch
    (prospect_5d.py:148-155), exact hot spot dso == 0 (sailh.py:126-127), relative azimuth
    folding (sailh.py:65) and the SMAC cksi clamp (smac.py:134-135)."""
    torch, sb, so = env
    assert gpu_bands(env, np.zeros((0, 27)), "Sentinel2A-MSI").shape == (0, 13, 3)
    P = so.synthetic_params(64, 3, seed=77)
    P[0:8, so.SMP] = [0.0, 4.99, 5.0, 5.01, 3.0, 1.0, 5.0, 2.0]          # mu <= 0 -> wet = dry
    P[8:16, so.CDM] = 0.01                                              # PRO inputs with Cdm > 0
    P[16:24, so.VZA] = P[16:24, so.SZA]
    P[16:24, so.RAA] = 0.0                                              # dso == 0
    P[24:28, so.RAA] = [180.0, 360.0, 540.0, 270.0]
    P[28:32, so.SZA] = 0.0
    P[28:32, so.VZA] = 0.0                                              # cksi = -1 (clamp boundary)
    P[32:36, so.LAI] = [1e-3, 0.01, 10.0, 15.0]
    for sensor in ("LANDSAT8-OLI", "TerraAqua-MODIS"):
        want = so.spart_bands(P, sensor)
        got = gpu_bands(env, P, sensor)
        assert relerr(got, want) < RTOL64
    one = gpu_bands(env, P[:1], "LANDSAT8-OLI")
    assert np.array_equal(one[0], gpu_bands(env, P, "LANDSAT8-OLI")[0])


@pytest.mark.parametrize("name", ["soilfile_Sentinel2A", "soilfile_TerraAqua"])
def test_user_soil_spectrum(env, name):
    """SoilParametersFromFile: batched entry point and the SPART class against the reference."""
    torch, sb, so = env
    g = load_golden(f"{name}.npz")
    P, sensor, rdry = g["params"], str(g["sensor"]), g["rdry"]
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    got = sb.run_batch_params(dev, sensor, soil_spectrum=rdry).cpu().numpy()
    assert relerr(got, g["O2"]) < RTOL64
    assert relerr(got, g["O1"]) < 5e-8
    host = sb.run_batch_params(np.ascontiguousarray(P.T), sensor, soil_spectrum=rdry)
    assert np.array_equal(host, got)
    got32 = sb.run_batch_params(dev, sensor, soil_spectrum=rdry, precision="fp32").cpu().numpy()
    assert np.percentile(np.abs(got32 - got) / np.abs(got), 99) < RTOL32
    p = P[0]
    spart = sb.SPART(sb.SoilParametersFromFile(rdry[:, None].copy(), p[12], p[13], p[14]),
                     sb.LeafBiology(*p[0:9]), sb.CanopyStructure(*p[15:19]), sb.AtmosphericProperties(*p[22:26]),
                     sb.Angles(*p[19:22]), sensor, int(p[26]))
    res = spart.run(debug=True)
    one = np.stack([res["R_TOC"].to_numpy(), res["R_TOA"].to_numpy(), res["L_TOA"].to_numpy()], axis=1)
    assert relerr(one, g["O2"][0]) < RTOL64
    assert np.allclose(spart.soilopt.refl_dry[:, 0], rdry, rtol=0, atol=0)
    assert "rsoil" in res.columns


def test_prospect_stage_reference_grid(env):
    """The reference's PROSPECT unit test (tests/unit/test_PROSPECT.py:17-28) on a subset of its grid
    (build_PROSPECT_tests.py:38-50), through the reference-shaped PROSPECT_5D and the batched form."""
    _, sb, _ = env
    g = load_golden("prospect_grid.npz")
    refl, tran, kchl = sb.prospect_batch(g["leaf7"])
    got = golden_columns(np.stack([refl, tran, kchl], axis=1), g)
    assert relerr(got, g["O2"]) < RTOL64
    np.testing.assert_almost_equal(got, g["O1"], decimal=7)          # the reference's own criterion
    r = sb.PROSPECT_5D(sb.LeafBiology(*g["leaf7"][0]), sb.load_optical_parameters())
    assert r.refl.shape == (2001, 1) and np.array_equal(r.refl[:, 0], refl[0]) and np.array_equal(r.kChlrel[:, 0], kchl[0])


def test_sailh_stage_reference_grid(env):
    """The reference's SAILH unit test (tests/unit/test_SAILH.py:19-38) on a subset of its grid
    (build_SAILH_tests.py:87-101) with the recorded default leaf / soil optics as inputs."""
    _, sb, so = env
    g = load_golden("sailh_grid.npz")
    c7 = g["canopy_angles7"]
    got = sb.sailh_batch(g["soil_refl"], g["leaf_refl"], g["leaf_tran"], c7[:, :4], c7[:, 4:7])
    ok = np.isfinite(g["O1"])
    cols = golden_columns(got, g)
    assert (np.isfinite(cols) == ok).all()
    assert relerr(cols[ok], g["O1"][ok]) < RTOL64
    np.testing.assert_array_almost_equal(cols[ok], g["O1"][ok], decimal=6)   # the reference's own criterion
    # reference-shaped single call, per-sample spectra, and the length check of sailh.py:37-44
    soil = sb.stages.SoilOptics(g["soil_refl"][:, None], None)
    leaf = sb.stages.LeafOptics(g["leaf_refl"][:, None], g["leaf_tran"][:, None], None)
    r = sb.SAILH(soil, leaf, sb.CanopyStructure(*c7[3, :4]), sb.Angles(*c7[3, 4:7]))
    assert np.array_equal(r.rso[:, 0], got[3, 0]) and np.array_equal(r.rdd[:, 0], got[3, 3])
    n = c7.shape[0]
    per = sb.sailh_batch(np.repeat(g["soil_refl"][None], n, 0), np.repeat(g["leaf_refl"][None], n, 0),
                         np.repeat(g["leaf_tran"][None], n, 0), c7[:, :4], c7[:, 4:7])
    assert np.array_equal(per, got, equal_nan=True)
    with pytest.raises(RuntimeError):
        sb.SAILH(soil, sb.stages.LeafOptics(g["leaf_refl"][:2001, None], g["leaf_tran"][:2001, None], None),
                 sb.CanopyStructure(3, -0.35, -0.15, 0.05), sb.Angles(40, 0, 0))


def test_bsm_stage_and_padding(env):
    _, sb, so = env
    g = load_golden("spectra.npz")
    P = g["params"]
    wet, dry = sb.bsm_batch(P[:, 9:15])
    wet, dry = golden_columns(wet, g), golden_columns(dry, g)
    assert relerr(wet, g["O2.soil_refl"][:, :wet.shape[1]]) < RTOL64 and relerr(dry, g["O2.soil_refl_dry"]) < RTOL64
    soilopt = sb.BSM(sb.SoilParameters(*P[0, 9:15]))
    leafbio = sb.LeafBiology(*P[0, 0:9])
    leafopt = sb.PROSPECT_5D(leafbio)
    soilopt = sb.set_soil_refl_trans_assumptions(soilopt)
    leafopt = sb.set_leaf_refl_trans_assumptions(leafopt, leafbio)
    assert soilopt.refl.shape == (2162, 1) and leafopt.tran.shape == (2162, 1) and leafopt.refl[-1, 0] == 0.01
    r = sb.SAILH(soilopt, leafopt, sb.CanopyStructure(*P[0, 15:19]), sb.Angles(*P[0, 19:22]))
    assert relerr(golden_columns(r.rso[:, 0], g), g["O2.rso"][0]) < RTOL64


def test_uniform_geometry_flag_is_only_an_optimisation(env):
    """SPART_FLAG_UNIFORM_GEOMETRY (shared sun/observer angles) must not change a single bit
    pattern beyond rounding: compare with the general path and with the oracle."""
    torch, sb, so = env
    P = so.synthetic_params(3000, 2, seed=21)
    P[:, so.SZA], P[:, so.VZA], P[:, so.RAA] = 33.0, 12.5, 140.0
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    a = sb.run_batch_params(dev, "Sentinel2A-MSI").cpu().numpy()
    b = sb.run_batch_params(dev, "Sentinel2A-MSI", uniform_geometry=True).cpu().numpy()
    assert relerr(b, a) < 1e-13
    assert relerr(b, so.spart_bands(P, "Sentinel2A-MSI")) < RTOL64
    c = sb.run_batch(P[:, 0:9], P[:, 9:15], P[:, 15:19], [33.0, 12.5, 140.0], P[:, 22:26], P[:, 26], "Sentinel2A-MSI")
    assert np.array_equal(c, b)


@pytest.mark.parametrize("sensor,n", [("TerraAqua-MODIS", 1000), ("Sentinel3A-OLCI", 777), ("LANDSAT8-OLI", 129),
                                      ("Sentinel2B-MSI", 1)])
def test_uniform_geometry_all_band_layouts(env, sensor, n):
    """The uniform-geometry band kernel (geometry folded into per-band constants once per block)
    against the general kernel and the oracle: two-knot bands (MODIS, OLCI), more than one band
    chunk (20 / 21 bands), ragged last tile, single sample; off-nadir, off-principal-plane angles."""
    torch, sb, so = env
    P = so.synthetic_params(n, 3, seed=77)
    P[:, so.SZA], P[:, so.VZA], P[:, so.RAA] = 51.25, 27.5, 97.0
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    a = sb.run_batch_params(dev, sensor).cpu().numpy()
    b = sb.run_batch_params(dev, sensor, uniform_geometry=True).cpu().numpy()
    assert relerr(b, a) < 1e-13
    assert relerr(b, so.spart_bands(P, sensor)) < RTOL64


@pytest.mark.parametrize("name", ["cfg2_S2A", "cfg5_S2B"])
def test_uniform_geometry_vs_reference_golden(env, name):
    """The fixed-geometry goldens of the unmodified reference through the uniform-geometry path."""
    torch, sb, _ = env
    g = load_golden(f"batch_{name}.npz")
    P = np.asarray(g["params"], dtype=np.float64)
    assert np.ptp(P[:, 19:22], axis=0).max() == 0.0        # these batches share one geometry
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    got = sb.run_batch_params(dev, str(g["sensor"]), uniform_geometry=True).cpu().numpy()
    assert relerr(got, g["O2"]) < RTOL64
    assert relerr(got, g["O1"]) < 5e-8


def test_cfg4_synthetic_fullspectrum_sensor(env):
    _, sb, so = env
    g = load_golden("batch_cfg4_SYNTH2001.npz")
    info = sb.synthetic_fullspectrum_sensorinfo()
    got = gpu_bands(env, g["params"], info)
    assert got.shape == (g["params"].shape[0], 2001, 3)
    assert relerr(got, g["O2"]) < RTOL64
    assert relerr(got, g["O1"]) < 1e-6


def test_large_batch_properties(env):
    """1M-sample configuration of BASELINE.json (config 2): size-independent properties --
    determinism, independence from batch position, finiteness and physical range."""
    torch, sb, so = env
    n = 1_000_000
    P = so.synthetic_params(n, 2)
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    a = sb.run_batch_params(dev, "Sentinel2A-MSI")
    b = sb.run_batch_params(dev, "Sentinel2A-MSI")
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert torch.isfinite(a).all()
    assert (a[..., 0] > 0).all() and (a[..., 0] < 1).all() and (a[..., 1] > 0).all() and (a[..., 1] < 1.5).all()
    # a permuted batch gives the permuted result (no cross-sample state)
    perm = torch.randperm(n, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    c = sb.run_batch_params(dev[:, perm].contiguous(), "Sentinel2A-MSI")
    assert torch.equal(c, a[perm])
    # 100 000 random rows of the batch against the oracle at the FP64 gate (VERDICT r1: 256 rows were thin)
    idx = np.random.default_rng(0).choice(n, 100_000, replace=False)
    want = np.concatenate([so.spart_bands(P[i], "Sentinel2A-MSI") for i in np.array_split(idx, 20)])
    assert relerr(a[torch.from_numpy(idx).cuda()].cpu().numpy(), want) < RTOL64
    # the folded-geometry kernels on the whole batch: a few ulp from the general path
    u = sb.run_batch_params(dev, "Sentinel2A-MSI", broadcast_rows=[7, 8, 13, 14, 19, 20, 21])
    assert float(((u - a).abs() / a.abs()).max()) < 1e-12


def test_large_batch_random_geometry_vs_oracle(env):
    """BASELINE config 3 (PROSPECT-PRO, random sun / view angles, LANDSAT8-OLI) at 1M samples: 100 000 rows
    against the oracle at the FP64 gate; FP32 mode on the same rows at its gate."""
    torch, sb, so = env
    n = 1_000_000
    P = so.synthetic_params(n, 3)
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    a = sb.run_batch_params(dev, "LANDSAT8-OLI", broadcast_rows=[1, 13, 14])
    idx = np.random.default_rng(1).choice(n, 100_000, replace=False)
    res = [so.spart_bands(P[i], "LANDSAT8-OLI", return_canopy=True) for i in np.array_split(idx, 20)]
    want = np.concatenate([r[0] for r in res])
    canopy = np.concatenate([r[1] for r in res])
    tidx = torch.from_numpy(idx).cuda()
    assert relerr(a[tidx].cpu().numpy(), want) < RTOL64
    f = sb.run_batch_params(dev, "LANDSAT8-OLI", broadcast_rows=[1, 13, 14], precision="fp32")[tidx].cpu().numpy()
    valid = ((canopy > 0) & (canopy < 1)).all(axis=2)
    with np.errstate(all="ignore"):
        e = np.abs(f - want) / np.abs(want)
    assert valid.mean() > 0.99 and e[valid].max() < RTOL32


def test_full_reference_unit_test_grids(env):
    """The reference's complete unit-test grids -- 6480 PROSPECT cases (build_PROSPECT_tests.py:38-50) and
    8100 SAILH cases (build_SAILH_tests.py:87-101) -- GPU against the oracle (the 24-row subsets recorded
    from the reference itself pin the oracle, tests/test_oracle_golden.py)."""
    import itertools
    torch, sb, so = env
    opt = so.load_optical()
    grid = np.array(list(itertools.product(np.arange(10, 85, 10), np.arange(0.005, 0.025, 0.01),
                                           np.arange(0.02, 0.12, 0.04), np.arange(0, 1.5, 0.5), np.arange(10, 35, 10),
                                           np.arange(10, 35, 10), np.arange(1.0, 3.5, 0.5))), dtype=np.float64)
    assert grid.shape == (6480, 7)
    refl, tran, kchl = sb.prospect_batch(grid)
    leaf9 = np.concatenate([grid, np.zeros((6480, 2))], axis=1)
    w = so.prospect(leaf9, opt)
    for got, want, name in zip((refl, tran, kchl), w, ("refl", "tran", "kChlrel")):
        assert relerr(got, want) < RTOL64, name
    grid = np.array(list(itertools.product(np.arange(1, 8, 3), np.arange(-1, 1, 0.4), np.arange(-1, 1, 0.4),
                                           np.arange(0.01, 0.2, 0.05), np.arange(0, 75, 30), np.arange(0, 75, 30),
                                           np.arange(0, 180, 80))), dtype=np.float64)
    assert grid.shape == (8100, 7)
    g = load_golden("sailh_grid.npz")        # the grid's fixed leaf / soil optics (build_SAILH_tests.py:11-28)
    got = sb.sailh_batch(g["soil_refl"], g["leaf_refl"], g["leaf_tran"], grid[:, :4], grid[:, 4:7])
    rep = lambda x: np.repeat(x[None, :], 8100, 0)
    with np.errstate(all="ignore"):
        want = np.stack(so.sailh(rep(g["soil_refl"]), rep(g["leaf_refl"]), rep(g["leaf_tran"]), grid[:, :4],
                                 grid[:, 4:7]), axis=1)
    assert (np.isfinite(got) == np.isfinite(want)).all()
    assert relerr(got, want) < RTOL64


@pytest.mark.parametrize("sensor,cfg", [("Sentinel2A-MSI", 2), ("LANDSAT8-OLI", 3), ("TerraAqua-MODIS", 3)])
def test_srf_band_mode(env, sensor, cfg):
    """band_mode="srf": SRF-weighted band means of the canopy reflectances
    (calculate_spectral_convolution, SPART.py:358-396, applied to canopyopt), then the same
    SMAC / TOC->TOA algebra.  Oracle = that function on the oracle's full spectra."""
    torch, sb, so = env
    P = so.synthetic_params(300, cfg, seed=3000 + cfg)
    want = so.spart_bands(P, sensor, band_mode="srf")
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    got = sb.run_batch_params(dev, sensor, band_mode="srf").cpu().numpy()
    assert relerr(got, want) < RTOL64
    interp = sb.run_batch_params(dev, sensor).cpu().numpy()
    assert relerr(got, interp) > 1e-4        # it really is a different band definition
    host = sb.run_batch_params(np.ascontiguousarray(P.T), sensor, band_mode="srf")
    assert np.array_equal(host, got)
    with pytest.raises(sb.SpartError):
        sb.run_batch_params(dev, sensor, band_mode="srf", precision="fp32")


@pytest.mark.parametrize("name", ["srf_Sentinel2A", "srf_LANDSAT8", "srf_TerraAqua"])
def test_srf_band_mode_vs_reference_golden(env, name):
    """SRF band mode against goldens recorded from the reference itself: its
    calculate_spectral_convolution (SPART.py:358-396) applied to its canopyopt, then its own atmopt
    and TOC->TOA algebra (tools/make_golden.py::run_srf)."""
    torch, sb, _ = env
    g = load_golden(f"{name}.npz")
    dev = torch.from_numpy(np.ascontiguousarray(g["params"].T)).cuda()
    got = sb.run_batch_params(dev, str(g["sensor"]), band_mode="srf").cpu().numpy()
    assert relerr(got, g["O2"]) < RTOL64
    assert relerr(got, g["O1"]) < 5e-8


def test_multi_sensor_shares_the_per_sample_work(env):
    """Config 5 of BASELINE.json (Sentinel-2A + -2B on one batch): the second sensor reuses the
    per-sample record (SPART_FLAG_REUSE_RECORD) and must give exactly the single-sensor result."""
    torch, sb, so = env
    P = so.synthetic_params(5000, 5, seed=50)
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    for prec in ("fp64", "fp32"):
        a, b = sb.run_batch_params(dev, ["Sentinel2A-MSI", "Sentinel2B-MSI"], precision=prec, uniform_geometry=True)
        assert torch.equal(a, sb.run_batch_params(dev, "Sentinel2A-MSI", precision=prec, uniform_geometry=True))
        assert torch.equal(b, sb.run_batch_params(dev, "Sentinel2B-MSI", precision=prec, uniform_geometry=True))
    ha, hb = sb.run_batch_params(np.ascontiguousarray(P.T), ["Sentinel2A-MSI", "Sentinel2B-MSI"])
    assert relerr(hb, so.spart_bands(P, "Sentinel2B-MSI")) < RTOL64 and ha.shape == (5000, 13, 3)


@pytest.mark.parametrize("sensor", ["Sentinel2A-MSI", "TerraAqua-MODIS", "LANDSAT8-OLI", "Sentinel3B-OLCI"])
def test_smac_stage(env, sensor):
    """SMAC alone against the oracle's restatement of smac.py:14-213 (nine AtmosphericOptics arrays;
    float32 Sentinel-2 coefficients keep their NumPy dtype semantics)."""
    _, sb, so = env
    P = so.synthetic_params(3000, 3, seed=71)
    P[:4, so.SZA], P[:4, so.VZA] = 0.0, 0.0                       # cksi clamp boundary (smac.py:134-135)
    want = so.smac(P[:, so.SZA:so.RAA + 1], P[:, so.AOT550:so.PA + 1], so.load_sensor(sensor)["SMAC_coef"])
    got = sb.smac_batch(P[:, so.SZA:so.RAA + 1], P[:, so.AOT550:so.PA + 1], sensor)
    for i, k in enumerate(sb.stages.ATM_FIELDS):
        assert relerr(got[:, i], np.broadcast_to(want[k], got[:, i].shape)) < RTOL64, k
    one = sb.SMAC(sb.Angles(*P[7, so.SZA:so.RAA + 1]), sb.AtmosphericProperties(*P[7, so.AOT550:so.PA + 1]), sensor)
    assert one.Tg.shape == (1, got.shape[2]) and np.array_equal(one.Ra_so[0], got[7, 4])


def test_lut_generate_and_nearest(env, tmp_path):
    """LUT consumer: chunked generation and nearest-entry retrieval against a brute-force search."""
    torch, sb, so = env
    P = so.synthetic_params(6000, 2, seed=91)
    lut = sb.lut.generate(P.T, "Sentinel2A-MSI", column=0, chunk=2500, path=str(tmp_path / "lut.npz"),
                          uniform_geometry=True)
    assert lut.shape == (6000, 13) and lut.dtype == torch.float32
    want = so.spart_bands(P[:200], "Sentinel2A-MSI")[:, :, 0]
    assert relerr(lut[:200].cpu().numpy(), want) < 1e-6                       # float32 storage
    z = np.load(tmp_path / "lut.npz")
    assert z["lut"].shape == (6000, 13) and z["params"].shape == (6000, 27)
    g = torch.Generator(device="cuda").manual_seed(1)
    for nb, n, m in ((13, 6000, 777), (26, 5000, 300), (6, 333, 1000), (1, 100, 5)):
        L = torch.rand((n, nb), generator=g, device="cuda", dtype=torch.float32)
        O = torch.rand((m, nb), generator=g, device="cuda", dtype=torch.float32)
        w = torch.rand(nb, generator=g, device="cuda", dtype=torch.float32) + 0.1
        for weights in (None, w):
            idx, cost = sb.lut.nearest(L, O, weights)
            ww = torch.ones(nb, device="cuda") if weights is None else weights
            d = ((O[:, None, :].double() - L[None, :, :].double()) ** 2 * ww.double()).sum(-1)
            best = d.min(dim=1)
            # the chosen entry is optimal up to float rounding of the cost
            assert torch.all(d.gather(1, idx[:, None])[:, 0] <= best.values * (1 + 1e-5) + 1e-12)
            assert torch.allclose(cost.double(), best.values, rtol=1e-4, atol=1e-9)
    # an observation that is a LUT row finds itself; retrieval of noisy simulations finds a near neighbour
    idx, cost = sb.lut.nearest(lut, lut[100:164].clone())
    assert torch.equal(idx.cpu(), torch.arange(100, 164)) and float(cost.max()) == 0.0


def test_spart_class_api_details(env):
    """Drop-in details of SPART(...).run() (SPART.py:254-269): column order, Band labels, index
    dtype per sensor, debug column, mutable parameter attributes, custom sensorinfo dicts."""
    torch, sb, so = env
    args = lambda: (sb.SoilParameters(0.5, 0, 100, 20, 25, 0.015), sb.LeafBiology(40, 0.01, 0.02, 0, 10, 10, 1.5),
                    sb.CanopyStructure(3, -0.35, -0.15, 0.05), sb.AtmosphericProperties(0.325, 0.35, 1.41),
                    sb.Angles(40, 0, 0))
    s2 = sb.SPART(*args(), "Sentinel2A-MSI", 100)
    df = s2.run(debug=True)
    assert list(df.columns) == ["Band", "L_TOA", "R_TOA", "R_TOC", "rsoil"]
    assert df.index.dtype == np.uint16 and list(df["Band"]) == [""] * 13          # as in the reference's pickle
    assert s2.R_TOC.shape == (1, 13) and s2.L_TOA.shape == (1, 13)
    assert s2.canopyopt.rso.shape == (2162, 1) and s2.leafopt.kChlrel.shape == (2001, 1)
    assert np.allclose(df["rsoil"].to_numpy(), np.interp(df.index.to_numpy(), s2.spectral.wlS, s2.soilopt.refl[:, 0]))
    modis = sb.SPART(*args(), "TerraAqua-MODIS", 100).run()
    assert modis.index.dtype == np.float64 and modis["Band"].iloc[0].startswith("Band")
    # parameters are plain mutable attributes; every run() is a fresh evaluation (no stale-SMAC bug)
    before = s2.run()["R_TOA"].to_numpy().copy()
    s2.angles = sb.Angles(30, 10, 90)
    after = s2.run()["R_TOA"].to_numpy()
    fresh = sb.SPART(*args()[:4], sb.Angles(30, 10, 90), "Sentinel2A-MSI", 100).run()["R_TOA"].to_numpy()
    assert not np.allclose(before, after) and np.array_equal(after, fresh)
    # a user-assigned sensorinfo dict (the reference's attribute is plain, SPART.py:95)
    custom = sb.SPART(*args(), "TerraAqua-MODIS", 100)
    custom.sensorinfo = sb.synthetic_fullspectrum_sensorinfo()
    out = custom.run()
    assert len(out) == 2001 and np.isfinite(out["R_TOC"].to_numpy()).all()
    with pytest.raises(FileNotFoundError):
        sb.SPART(*args(), "NoSuchSensor", 100)
    row = sb.row_as_dataframe(torch.from_numpy(np.stack([df["R_TOC"], df["R_TOA"], df["L_TOA"]], axis=1)),
                              "Sentinel2A-MSI")
    assert np.array_equal(row["L_TOA"].to_numpy(), df["L_TOA"].to_numpy())
