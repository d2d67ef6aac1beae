"""CPU checks of geometry_kernel's hot-spot integral (tools/check_hotspot_series.py mirrors the kernel's series,
its per-lane stopping rule and its branch test) against adaptive quadrature."""
import re
import sys

import numpy as np

from conftest import ROOT

sys.path.insert(0, str(ROOT / "tools"))
import check_hotspot_series as hs  # noqa: E402


def test_mirror_constants_match_the_kernel():
    src = (ROOT / "spart-python_b200" / "csrc" / "spart_device.cuh").read_text()
    val = lambda name: float(re.search(rf"#define {name} (\S+)", src).group(1))  # noqa: E731
    assert val("SPART_HOTSPOT_SMAX") == hs.SMAX
    assert val("SPART_HOTSPOT_AMAX") == hs.AMAX
    assert val("SPART_HOTSPOT_TOL") == hs.SERIES_TOL
    assert val("SPART_HOTSPOT_NMAX") == hs.NMAX
    assert val("SPART_HOTSPOT_SPLIT") == hs.SPLIT


def check(inputs, n_quad, tol_series, tol_panels=None):
    K, k, LAI, q, dso = inputs
    A, Cq, alpha, _ = hs.setup(K, k, LAI, q, dso)
    I, ser, N = hs.hotspot(K, k, LAI, q, dso)
    sel = np.arange(min(n_quad, len(I)))
    ref = hs.quad_reference(A[sel], Cq[sel], alpha[sel])
    err = np.abs(I[sel] - ref) / ref
    assert err[ser[sel]].max(initial=0.0) < tol_series
    if tol_panels is not None:
        assert (~ser[sel]).any()
        assert err[~ser[sel]].max() < tol_panels
    return I, ser, N


def test_series_on_the_benchmark_distributions():
    """Configs 2 and 3 (bench.py): every sample takes the series, within 2e-15 of quadrature; the slowest lane
    of a 32-sample warp needs about 16 (config 2) and 22 (config 3) terms."""
    for config, warp_terms in ((2, 17), (3, 23)):
        _, ser, N = check(hs.config_inputs(config, 4096, 21 + config), 100, 2e-15)
        assert ser.all()
        assert N.reshape(-1, 32).max(1).mean() < warp_terms
        assert N.max() <= 70


def test_series_on_a_wide_domain():
    """Zenith 0-85, view 0-60 degrees, LAI 1e-3-20, q 1e-4-1: no cancellation for sparse canopies, at most 1 in
    1e4 samples so close to the hot spot (s > SMAX) that it takes the panels."""
    inputs = hs.wide_inputs(8192, 31)
    _, ser, N = check(inputs, 160, 2e-15)
    assert ser.mean() > 0.9999
    assert N.max() <= 70
    LAI = inputs[2]
    sparse = LAI < 1e-2                   # e^E within 2 % of 1: the two gamma series would cancel
    assert check(tuple(x[sparse] for x in inputs), 40, 2e-15)[1].all()


def test_branches_at_the_hot_spot_and_for_bare_soil():
    """Rows on both sides of s = SMAX next to the hot spot, the exact hot spot (dso = 0) and bare soil (A = 0, the
    integral is exactly 1).  Where the series stops the panels keep their accuracy."""
    K, k, dso = hs.geometry([30.0] * 6, [30.5, 30.02, 30.005, 30.0001, 0.0, 40.0], [0.0] * 6, np.ones(6),
                            np.zeros(6), np.zeros(6))
    LAI, q = np.full(6, 3.0), np.full(6, 0.1)
    I, ser, N = check((K[:4], k[:4], LAI[:4], q[:4], dso[:4]), 4, 2e-15, 1e-12)
    assert ser.tolist() == [True, True, False, False]
    # exact hot spot: pso = e^{(A - sqrt(Kk) LAI) x}
    I0, ser0, _ = hs.hotspot(K[4:5], k[4:5], LAI[4:5], q[4:5], np.zeros(1))
    Am = (K[4] + k[4] - np.sqrt(K[4] * k[4])) * LAI[4]
    assert not ser0[0] and abs(I0[0] - (-np.expm1(-Am) / Am)) < 1e-14 * I0[0]
    # bare soil
    Ib, serb, _ = hs.hotspot(K[5:], k[5:], np.zeros(1), q[5:], dso[5:])
    assert not serb[0] and abs(Ib[0] - 1.0) < 1e-14
    # NaN inputs take the panels, as before
    assert not hs.use_series(np.array([np.nan]), np.array([1.0]), np.array([1.0]))[0]


def test_sparse_canopies_next_to_the_hot_spot():
    """LAI -> 0 with the sun at nadir and the view 1e-9 .. 1e-17 degrees off it (K ~ k, h_0 ~ LAI): the stopping
    bound takes h_j <= 1, so these rows run the longest series, up to the NMAX cap.  The products stay finite
    (s <= SMAX), the capped sums are as accurate as the others, and rows with s > SMAX take the panels."""
    LAI = np.array([3.5e-7, 3.5e-7, 1e-6, 1e-9, 1e-12, 1e-15, 1e-40])
    vza = np.array([1e-9, 1e-8, 2.91e-8, 2.91e-11, 2.91e-14, 2.91e-17, 2.91e-42])
    K, k, dso = hs.geometry(np.zeros(len(LAI)), vza, np.zeros(len(LAI)), LAI, np.full(len(LAI), -0.35),
                            np.full(len(LAI), -0.15))
    I, ser, N = check((K, k, LAI, np.ones(len(LAI)), dso), len(LAI), 2e-15, 2e-13)
    assert ser.tolist() == [False] + [True] * 6
    assert N[-2:].tolist() == [hs.NMAX, hs.NMAX]
    assert np.isfinite(I).all() and (I > 0.99).all()
    A, _, alpha, _ = hs.setup(K, k, LAI, np.ones(len(LAI)), dso)
    s = A / alpha
    assert (A[ser] * np.prod(s[ser, None] + np.arange(1, hs.NMAX + 1), axis=1) < 1e305).all()
