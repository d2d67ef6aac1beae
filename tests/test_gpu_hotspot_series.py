"""geometry_kernel's hot-spot integral on rows that take each of its two paths (the series and the Gauss-Legendre
panels, see spart_device.cuh::hotspot_integrals): band results and forward_spectrum's rso against the oracle at
1e-12 relative, with the leaf inclination distribution given to both so that only the canopy path differs."""
import sys

import numpy as np
import pytest

from conftest import ROOT, relerr

sys.path.insert(0, str(ROOT / "tools"))
import check_hotspot_series as hs  # noqa: E402
import spart_oracle as so  # noqa: E402

SENSOR = "Sentinel2A-MSI"
# LAI, q, sza, vza, raa, path
ROWS = [
    (8.0, 1e-3, 40.0, 0.0, 0.0, "series"),        # dense canopy, small q (alpha ~ 800)
    (5.0, 0.05, 40.0, 0.0, 0.0, "series"),
    (3.0, 0.1, 60.0, 30.0, 120.0, "series"),
    (20.0, 0.01, 80.0, 60.0, 180.0, "series"),
    (1e-3, 0.05, 40.0, 0.0, 0.0, "series"),       # sparse: e^E within 0.2 % of 1
    (1e-3, 1.0, 30.0, 20.0, 90.0, "series"),
    (3.0, 1.0, 45.0, 10.0, 30.0, "series"),       # large q
    (6.0, 0.5, 70.0, 50.0, 10.0, "series"),
    (3.0, 0.1, 30.0, 30.5, 0.0, "series"),        # near the hot spot, Cq ~ 30
    (3.0, 0.1, 0.0, 9.2e-3, 0.0, "series"),       # nearer, s ~ 900 <= SMAX
    (3.0, 0.1, 0.0, 8e-4, 0.0, "panels"),         # nearer still: s ~ 1.04e4 > SMAX
    (3.5e-7, 1.0, 0.0, 1e-8, 0.0, "series"),      # LAI -> 0 next to the hot spot: 74 terms
    (1e-15, 1.0, 0.0, 2.91e-17, 0.0, "series"),   # runs to the NMAX cap, s ~ 950
    (3.5e-7, 1.0, 0.0, 1e-9, 0.0, "panels"),      # s ~ 9.7e3 > SMAX
    (3.0, 0.1, 0.0, 0.0, 0.0, "panels"),          # exact hot spot, dso = 0
    (0.0, 0.05, 40.0, 0.0, 0.0, "panels"),        # bare soil
]
# Next to the hot spot the rows keep the sun at nadir: dso = tan(vza) is then well conditioned.  Elsewhere it is a
# difference of O(1) terms (sailh.py:78), whose rounding makes the oracle and the GPU see different geometries.


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    return torch, spart_b200


def rows():
    P = np.repeat(so.synthetic_params(1, 2, seed=4), len(ROWS), axis=0)
    for i, (lai, q, sza, vza, raa, _) in enumerate(ROWS):
        P[i, [so.LAI, so.HOT_Q, so.SZA, so.VZA, so.RAA]] = lai, q, sza, vza, raa
    P[:, so.LIDFA], P[:, so.LIDFB] = -0.35, -0.15
    return P, so.leafangles(P[:, so.LIDFA], P[:, so.LIDFB])


def test_rows_take_the_intended_path():
    P, lidf = rows()
    K, k, dso = hs.geometry(P[:, so.SZA], P[:, so.VZA], P[:, so.RAA], P[:, so.LAI], P[:, so.LIDFA], P[:, so.LIDFB])
    A, Cq, alpha, _ = hs.setup(K, k, P[:, so.LAI], P[:, so.HOT_Q], dso)
    assert hs.use_series(A, Cq, alpha).tolist() == [r[-1] == "series" for r in ROWS]


@pytest.mark.gpu
def test_bands_and_rso_against_the_oracle(env):
    torch, sb = env
    P, lidf = rows()
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    eng = sb.default_engine()
    got = eng.forward_bands(dev, SENSOR, lidf=lidf).cpu().numpy()
    want = so.spart_bands(P, SENSOR, lidf=lidf)
    errs = [relerr(got[i], want[i]) for i in range(len(ROWS))]
    print("band results, max relative error per row:", " ".join(f"{e:.1e}" for e in errs))
    spec = eng.forward_spectrum(dev, lidf=lidf).cpu().numpy()
    rso = so.sailh(spec[:, 3], spec[:, 0], spec[:, 1], P[:, so.LAI:so.HOT_Q + 1], P[:, so.SZA:so.RAA + 1],
                   lidf=lidf)[0]
    errs_rso = [relerr(spec[i, 5], rso[i]) for i in range(len(ROWS))]
    print("rso, max relative error per row:", " ".join(f"{e:.1e}" for e in errs_rso))
    assert max(errs_rso) < 1e-12
    assert max(errs) < 1e-12


@pytest.mark.gpu
def test_rows_do_not_depend_on_their_warp(env):
    """Each lane stops the series at its own term count.  A row evaluated alone equals, bit for bit, the same row
    in the mixed batch; and 65 536 config-3 rows (random angles, so warps whose lanes need from a few to about 50 terms) plus these
    rows give the same bits in a shuffled order, where every row meets other warp mates.  A warp-wide term count
    would add terms below 1e-17 of the sum, which change the last bit of some of these rows."""
    torch, sb = env
    P, _ = rows()
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    batch = sb.run_batch_params(dev, SENSOR)
    for i in range(len(ROWS)):
        alone = sb.run_batch_params(dev[:, i:i + 1].contiguous(), SENSOR)
        assert torch.equal(alone[0], batch[i]), ROWS[i]
    big = np.concatenate([so.synthetic_params(65536, 3, seed=12), P])
    dev = torch.from_numpy(np.ascontiguousarray(big.T)).cuda()
    a = sb.run_batch_params(dev, SENSOR)
    perm = torch.randperm(len(big), device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    b = sb.run_batch_params(dev[:, perm].contiguous(), SENSOR)
    assert torch.equal(b, a[perm])
