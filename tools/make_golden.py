#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference.

Runs only in the build container (needs /root/reference, scipy's QUADPACK and a stub for
the missing `nvtx` package).  The GPU box never runs this; it only sees the committed
.npz files.  Two reference variants are recorded for every case (SURVEY.md section 8(c)):

  O1  the raw reference, one fresh SPART object per sample, np.float64 scalar inputs;
  O2  the same code with only `integrate.quad` *inside prospect_5d* replaced by
      scipy.special.exp1 (the function prospect_5d.py:186-188 says it implements).

Usage:  python tools/make_golden.py [--jobs 8]
"""
import argparse
import itertools
import multiprocessing as mp
import sys
import warnings
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tools" / "_nvtx_stub"))
sys.path.insert(1, "/root/reference/src")
sys.path.insert(2, str(ROOT / "oracle"))
GOLD = ROOT / "tests" / "golden"

warnings.simplefilter("ignore")


class _ExactE1Shim:
    """Stands in for the name `integrate` inside prospect_5d only (O2)."""

    @staticmethod
    def quad(func, a, b, *args, **kw):
        from scipy.special import exp1
        assert np.isinf(b)
        return (float(exp1(a)), 0.0)


def _ref_modules(o2):
    import scipy.integrate
    import SPART
    import SPART.prospect_5d as p5
    p5.integrate = _ExactE1Shim if o2 else scipy.integrate
    return SPART


def _objects(SPART, p):
    f = np.float64
    leaf = SPART.LeafBiology(f(p[0]), f(p[1]), f(p[2]), f(p[3]), f(p[4]), f(p[5]), f(p[6]), f(p[7]), f(p[8]))
    soil = SPART.SoilParameters(f(p[9]), f(p[10]), f(p[11]), f(p[12]), f(p[13]), f(p[14]))
    canopy = SPART.CanopyStructure(f(p[15]), f(p[16]), f(p[17]), f(p[18]))
    angles = SPART.Angles(f(p[19]), f(p[20]), f(p[21]))
    atm = SPART.AtmosphericProperties(f(p[22]), f(p[23]), f(p[24]), f(p[25]))
    return soil, leaf, canopy, atm, angles


def run_one(task):
    """task = (params[27], sensor name or 'SYNTH2001', o2 flag, want_spectra)."""
    import contextlib
    import io
    p, sensor, o2, want_spectra = task
    SPART = _ref_modules(o2)
    soil, leaf, canopy, atm, angles = _objects(SPART, p)
    doy = int(p[26])
    with contextlib.redirect_stdout(io.StringIO()):
        if sensor == "SYNTH2001":
            import spart_oracle
            sp = SPART.SPART(soil, leaf, canopy, atm, angles, "TerraAqua-MODIS", doy)
            sp.sensorinfo = spart_oracle.synthetic_fullspectrum_sensor()
        else:
            sp = SPART.SPART(soil, leaf, canopy, atm, angles, sensor, doy)
        df = sp.run()
    out = np.stack([df["R_TOC"].to_numpy(), df["R_TOA"].to_numpy(), df["L_TOA"].to_numpy()], axis=1)
    spec = None
    if want_spectra:
        spec = dict(
            leaf_refl=sp.leafopt.refl[:, 0], leaf_tran=sp.leafopt.tran[:, 0], kChlrel=sp.leafopt.kChlrel[:, 0],
            soil_refl=sp.soilopt.refl[:, 0], soil_refl_dry=sp.soilopt.refl_dry[:, 0],
            rso=sp.canopyopt.rso[:, 0], rdo=sp.canopyopt.rdo[:, 0],
            rsd=sp.canopyopt.rsd[:, 0], rdd=sp.canopyopt.rdd[:, 0], lidf=canopy.lidf[:, 0],
        )
    return out, spec


def run_userlidf(task):
    """Reference run with a leaf inclination distribution assigned after construction
    (canopy.lidf = ..., which SAILH uses as is, sailh.py:81-97).  task = (params[27], lidf[13], sensor, o2)."""
    import contextlib
    import io
    p, lidf, sensor, o2 = task
    SPART = _ref_modules(o2)
    soil, leaf, canopy, atm, angles = _objects(SPART, p)
    canopy.lidf = np.asarray(lidf, dtype=np.float64).reshape(13, 1)
    with contextlib.redirect_stdout(io.StringIO()):
        df = SPART.SPART(soil, leaf, canopy, atm, angles, sensor, int(p[26])).run()
    return np.stack([df["R_TOC"].to_numpy(), df["R_TOA"].to_numpy(), df["L_TOA"].to_numpy()], axis=1)


def run_soilfile(task):
    """Reference run with SoilParametersFromFile(ndarray) (bsm.py:155-226)."""
    import contextlib
    import io
    p, rdry, sensor, o2 = task
    SPART = _ref_modules(o2)
    from SPART.bsm import SoilParametersFromFile
    _, leaf, canopy, atm, angles = _objects(SPART, p)
    f = np.float64
    soil = SoilParametersFromFile(rdry[:, None].copy(), f(p[12]), f(p[13]), f(p[14]))
    with contextlib.redirect_stdout(io.StringIO()):
        df = SPART.SPART(soil, leaf, canopy, atm, angles, sensor, int(p[26])).run()
    return np.stack([df["R_TOC"].to_numpy(), df["R_TOA"].to_numpy(), df["L_TOA"].to_numpy()], axis=1)


def run_prospect(task):
    import contextlib
    import io
    leaf7, o2 = task
    SPART = _ref_modules(o2)
    from SPART.prospect_5d import PROSPECT_5D, LeafBiology
    with contextlib.redirect_stdout(io.StringIO()):
        r = PROSPECT_5D(LeafBiology(*[np.float64(v) for v in leaf7]), SPART.load_optical_parameters())
    return np.stack([r.refl[:, 0], r.tran[:, 0], r.kChlrel[:, 0]])


def run_sailh(task):
    c7, rho, tau, rs = task
    _ref_modules(False)
    from SPART.sailh import SAILH, Angles, CanopyStructure
    from SPART.bsm import SoilOptics
    from SPART.prospect_5d import LeafOptics
    f = np.float64
    canopy = CanopyStructure(f(c7[0]), f(c7[1]), f(c7[2]), f(c7[3]))
    r = SAILH(SoilOptics(rs[:, None], None), LeafOptics(rho[:, None], tau[:, None], None),
              canopy, Angles(f(c7[4]), f(c7[5]), f(c7[6])))
    return np.stack([r.rso[:, 0], r.rdo[:, 0], r.rsd[:, 0], r.rdd[:, 0]]), canopy.lidf[:, 0]


def run_srf(task):
    """SRF band mode golden from the reference's own functions: calculate_spectral_convolution
    (SPART.py:358-396) applied to the four canopyopt spectra of a reference run, then the reference's SMAC
    output and TOC->TOA algebra (SPART.py:235-252) as they stand after run()."""
    import contextlib
    import io
    p, sensor, o2 = task
    SPART = _ref_modules(o2)
    from SPART.SPART import calculate_spectral_convolution
    soil, leaf, canopy, atm, angles = _objects(SPART, p)
    with contextlib.redirect_stdout(io.StringIO()):
        sp = SPART.SPART(soil, leaf, canopy, atm, angles, sensor, int(p[26]))
        df = sp.run()
    wl = sp.ETpar["wl_Ea"] if hasattr(sp, "ETpar") else np.arange(400, 2401)[:, None]
    rv = {k: calculate_spectral_convolution(wl, getattr(sp.canopyopt, k)[:2001], sp.sensorinfo)
          for k in ("rso", "rdo", "rdd", "rsd")}
    a = sp.atmopt
    La = sp._La                        # SRF-convolved ET radiance of this sample, SPART.py:183-185
    rtoa0 = a.Ra_so + a.Ta_ss * rv["rso"] * a.Ta_oo
    rtoa1 = ((a.Ta_sd * rv["rdo"] + a.Ta_ss * rv["rsd"] * a.Ra_dd * rv["rdo"]) * a.Ta_oo) / (1 - rv["rdd"] * a.Ra_dd)
    rtoa2 = (a.Ta_ss * rv["rsd"] + a.Ta_sd * rv["rdd"]) * a.Ta_do / (1 - rv["rdd"] * a.Ra_dd)
    R_TOC = (a.Ta_ss * rv["rso"] + a.Ta_sd * rv["rdo"]) / (a.Ta_ss + a.Ta_sd)
    R_TOA = a.Tg * (rtoa0 + rtoa1 + rtoa2)
    band = np.stack([rv["rso"], rv["rdo"], rv["rsd"], rv["rdd"]], axis=1)
    L_TOA = La * R_TOA
    return np.stack([R_TOC[0], R_TOA[0], L_TOA[0]], axis=1), band


def conftest_defaults():
    """tests/conftest.py:90-112 defaults, DOY 100 (tests/e2e/test_SPART.py:30-39)."""
    p = np.zeros(27)
    p[0:9] = [40, 0.01, 0.02, 0, 10, 10, 1.5, 0, 0]
    p[9:15] = [0.5, 0, 100, 20, 25, 0.015]
    p[15:19] = [3, -0.35, -0.15, 0.05]
    p[19:22] = [40, 0, 0]
    p[22:26] = [0.325, 0.35, 1.41, 1013.25]
    p[26] = 100
    return p


def thin_spectra(arrays, step):
    """Keeps a fixture file under 1 MB: every array of `arrays` whose last axis holds a spectrum (2001 or 2162
    wavelengths) is cut to every `step`-th wavelength plus 400-415 nm (where the README case is NaN) and the
    edges of the 2001-sample range; all rows are kept.  The kept indices are stored as `wl_idx` (the tests
    select the same columns with conftest.golden_columns)."""
    idx = np.unique(np.r_[np.arange(0, 2162, step), np.arange(16), 1999, 2000, 2001, 2161])
    out = {k: a[..., idx[idx < a.shape[-1]]] if a.ndim and a.shape[-1] in (2001, 2162) else a for k, a in arrays.items()}
    out["wl_idx"] = idx
    return out


def readme_quickstart():
    """README.md:23-31 (note the positional slip: Cdm=10, Cs=0.01, Cca=0)."""
    p = conftest_defaults()
    p[0:9] = [40, 10, 0.02, 0.01, 0, 10, 1.5, 0, 0]
    p[12] = 15
    p[22:26] = [0.3246, 0.3480, 1.4116, 1013.25]
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--jobs", type=int, default=8)
    ap.add_argument("--n", type=int, default=48, help="random samples per batch fixture")
    ap.add_argument("--only", default=None, help="regenerate only this fixture group (e.g. soilfile)")
    args = ap.parse_args()
    import spart_oracle as so
    GOLD.mkdir(parents=True, exist_ok=True)
    pool = mp.Pool(args.jobs)

    def run_batch(P, sensor, spectra=False):
        res = {}
        for tag, o2 in (("O1", False), ("O2", True)):
            r = pool.map(run_one, [(p, sensor, o2, spectra) for p in P], chunksize=1)
            res[tag] = np.stack([x[0] for x in r])
            if spectra:
                for k in r[0][1]:
                    res[f"{tag}.{k}"] = np.stack([x[1][k] for x in r])
        return res

    # 6. user-supplied dry-soil spectrum (SoilParametersFromFile)
    if args.only in (None, "soilfile"):
        wl = np.arange(400, 2401, dtype=np.float64)
        rdry = 0.08 + 0.32 * (1 - np.exp(-(wl - 400) / 650)) - 0.05 * np.exp(-((wl - 1930) / 60) ** 2) \
            - 0.03 * np.exp(-((wl - 1440) / 50) ** 2)
        P = so.synthetic_params(16, 3, seed=61)
        for sensor in ("Sentinel2A-MSI", "TerraAqua-MODIS"):
            o1 = np.stack(pool.map(run_soilfile, [(p, rdry, sensor, False) for p in P]))
            o2 = np.stack(pool.map(run_soilfile, [(p, rdry, sensor, True) for p in P]))
            np.savez_compressed(GOLD / f"soilfile_{sensor.split('-')[0]}.npz", params=P, rdry=rdry,
                                sensor=np.array(sensor), O1=o1, O2=o2)
        print("soilfile done", flush=True)
        if args.only:
            pool.close()
            return

    # 7b. a user-assigned leaf inclination distribution (canopy.lidf = ...)
    if args.only in (None, "userlidf"):
        P = so.synthetic_params(8, 3, seed=63)
        rng = np.random.default_rng(64)
        L = rng.dirichlet(np.ones(13), size=8)
        L[0] = 1.0 / 13                                        # uniform over the classes
        L[1] = so.leafangles(np.array([-0.35]), np.array([-0.15]))[0]       # spherical, whatever LIDFa / LIDFb say
        res = {}
        for o2 in (False, True):
            outs = pool.map(run_userlidf, [(P[i], L[i], "LANDSAT8-OLI", o2) for i in range(8)])
            res["O2" if o2 else "O1"] = np.stack(outs)
        np.savez_compressed(GOLD / "user_lidf.npz", params=P, lidf=L, sensor=np.array("LANDSAT8-OLI"), **res)
        print("userlidf done", flush=True)
        if args.only:
            pool.close()
            return

    # 7. bare soil (LAI = 0 and LAI -> 0) with narrow and wide hot spots: sailh.py:112-114 guards LAI > 0
    if args.only in (None, "edge"):
        P = so.synthetic_params(12, 3, seed=62)
        P[:, so.LAI] = [0, 0, 0, 0, 0, 0, 1e-9, 1e-6, 1e-4, 1e-3, 0, 0]
        P[:, so.HOT_Q] = [0.01, 0.05, 0.001, 0.2, 0.01, 0.05, 0.01, 0.05, 0.01, 0.05, 0.01, 0.05]
        P[4:6, so.SZA], P[4:6, so.VZA], P[4:6, so.RAA] = 40.0, 0.0, 0.0
        P[10:12, so.VZA], P[10:12, so.RAA] = P[10:12, so.SZA], 0.0        # bare soil in the exact hot spot
        r = run_batch(P, "LANDSAT8-OLI")
        np.savez_compressed(GOLD / "edge_lai0.npz", params=P, sensor=np.array("LANDSAT8-OLI"), O1=r["O1"], O2=r["O2"])
        print("edge done", flush=True)
        if args.only:
            pool.close()
            return

    # 8. SRF band mode from the reference's own calculate_spectral_convolution on its canopyopt
    if args.only in (None, "srf"):
        for sensor, cfg in (("Sentinel2A-MSI", 2), ("LANDSAT8-OLI", 3), ("TerraAqua-MODIS", 3)):
            P = so.synthetic_params(12, cfg, seed=63)
            res = {}
            for tag, o2 in (("O1", False), ("O2", True)):
                r = pool.map(run_srf, [(p, sensor, o2) for p in P], chunksize=1)
                res[tag] = np.stack([x[0] for x in r])
                res[tag + ".canopy_bands"] = np.stack([x[1] for x in r])
            np.savez_compressed(GOLD / f"srf_{sensor.split('-')[0]}.npz", params=P, sensor=np.array(sensor), **res)
        print("srf done", flush=True)
        if args.only:
            pool.close()
            return

    # 1. e2e: conftest defaults on all nine sensors + README quickstart + example script
    e2e = {}
    d = conftest_defaults()
    for s in so.SENSORS:
        r = run_batch(d[None, :], s)
        e2e[f"{s}.O1"], e2e[f"{s}.O2"] = r["O1"][0], r["O2"][0]
    r = run_batch(readme_quickstart()[None, :], "TerraAqua-MODIS")
    e2e["README.O1"], e2e["README.O2"] = r["O1"][0], r["O2"][0]
    e2e["params_defaults"], e2e["params_readme"] = d, readme_quickstart()
    np.savez_compressed(GOLD / "e2e.npz", **e2e)
    print("e2e done", flush=True)

    # 2. random batches per BASELINE.json config
    n = args.n
    batches = {
        "cfg2_S2A": (so.synthetic_params(n, 2), "Sentinel2A-MSI"),
        "cfg3_L8": (so.synthetic_params(n, 3), "LANDSAT8-OLI"),
        "cfg5_S2B": (so.synthetic_params(n, 5), "Sentinel2B-MSI"),
        "rand_MODIS": (so.synthetic_params(n, 3, seed=777), "TerraAqua-MODIS"),
        "rand_OLCI": (so.synthetic_params(n // 2, 3, seed=778), "Sentinel3A-OLCI"),
        "rand_L7": (so.synthetic_params(n // 2, 2, seed=779), "LANDSAT7-ETM"),
    }
    for name, (P, sensor) in batches.items():
        r = run_batch(P, sensor)
        np.savez_compressed(GOLD / f"batch_{name}.npz", params=P, sensor=np.array(sensor), O1=r["O1"], O2=r["O2"])
        print(name, "done", flush=True)

    # 3. intermediate spectra (leafopt, soilopt, canopyopt) for a few samples incl. README NaN case
    P = np.concatenate([so.synthetic_params(3, 2, seed=31), so.synthetic_params(3, 3, seed=32),
                        conftest_defaults()[None, :], readme_quickstart()[None, :]])
    r = run_batch(P, "Sentinel2A-MSI", spectra=True)
    np.savez_compressed(GOLD / "spectra.npz", params=P, **thin_spectra(r, 3))
    print("spectra done", flush=True)

    # 4. config 4: synthetic 2001-band sensor
    P = so.synthetic_params(4, 4)
    r = run_batch(P, "SYNTH2001")
    np.savez_compressed(GOLD / "batch_cfg4_SYNTH2001.npz", params=P, sensor=np.array("SYNTH2001"),
                        O1=r["O1"], O2=r["O2"])
    print("cfg4 done", flush=True)

    # 5. subsets of the reference's own unit-test grids
    #    (tests/unit/test_PROSPECT/build_PROSPECT_tests.py:38-50, test_SAILH/build_SAILH_tests.py:87-101)
    rng = np.random.default_rng(42)
    grid = list(itertools.product(np.arange(10, 85, 10), np.arange(0.005, 0.025, 0.01), np.arange(0.02, 0.12, 0.04),
                                  np.arange(0, 1.5, 0.5), np.arange(10, 35, 10), np.arange(10, 35, 10),
                                  np.arange(1.0, 3.5, 0.5)))
    assert len(grid) == 6480
    pick = rng.choice(len(grid), 24, replace=False)
    leaf7 = np.array([grid[i] for i in pick], dtype=np.float64)
    o1 = np.stack(pool.map(run_prospect, [(l, False) for l in leaf7]))
    o2 = np.stack(pool.map(run_prospect, [(l, True) for l in leaf7]))
    np.savez_compressed(GOLD / "prospect_grid.npz", leaf7=leaf7, **thin_spectra(dict(O1=o1, O2=o2), 2))
    print("prospect grid done", flush=True)

    grid = list(itertools.product(np.arange(1, 8, 3), np.arange(-1, 1, 0.4), np.arange(-1, 1, 0.4),
                                  np.arange(0.01, 0.2, 0.05), np.arange(0, 75, 30), np.arange(0, 75, 30),
                                  np.arange(0, 180, 80)))
    assert len(grid) == 8100
    pick = rng.choice(len(grid), 24, replace=False)
    c7 = np.array([grid[i] for i in pick], dtype=np.float64)
    # default leaf / soil optics of the SAILH grid (build_SAILH_tests.py:11-28), from the raw reference
    _, spec = run_one((conftest_defaults(), "Sentinel2A-MSI", False, True))
    rho, tau, rs = spec["leaf_refl"], spec["leaf_tran"], spec["soil_refl"]
    res = pool.map(run_sailh, [(c, rho, tau, rs) for c in c7])
    np.savez_compressed(GOLD / "sailh_grid.npz", canopy_angles7=c7, leaf_refl=rho, leaf_tran=tau, soil_refl=rs,
                        lidf=np.stack([x[1] for x in res]), **thin_spectra(dict(O1=np.stack([x[0] for x in res])), 2))
    print("sailh grid done", flush=True)
    pool.close()


if __name__ == "__main__":
    main()
