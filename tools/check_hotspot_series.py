#!/usr/bin/env python
"""NumPy mirror / check of geometry_kernel's hot-spot integral (spart_device.cuh::hotspot_integrals).

The kernel needs I = int_{-1}^{0} exp(A x + z (1 - e^{alpha x})) dx, A = (K + k) LAI, z = sqrt(K k) LAI / alpha
(sailh.py:116-135).  With v = e^{alpha x}, s = A / alpha, v0 = e^{-alpha} and E = -A + z (1 - v0) <= 0:

    I = (1 / alpha) sum_{j>=0} z^j h_j / (s (s+1) ... (s+j)),   h_j = 1 - e^E v0^j

(the difference of two lower incomplete gamma series, merged term by term).  h_j follows from
h_0 = 1 - e^E (-expm1(E) for E > -0.5) and h_j = v0 h_{j-1} + (1 - v0), 1 - v0 = 1 - e^{-alpha} (-expm1(-alpha)
for alpha <= 0.5): every term is a sum of positive numbers, so nothing cancels however close e^E is to 1 (sparse
canopies).  The sum is accumulated without a division per term, R_m = R_{m-1} (s+m) + z^m h_m,
D_m = D_{m-1} (s+m), I = R_N / (A D_N), and each sample stops at its own N: the first even m at which the
bound z^{m+1} / (s+m+1-z) on the tail, in units of D_m, is at most SERIES_TOL R_m, or N = NMAX.  A >= 2 sqrt(K k) LAI gives s >= 2 z, so the terms fall at least by
half from one to the next.  The bound takes h_j <= 1, so for LAI -> 0 (h_0 << 1) a sample may run to the cap,
where the neglected tail is below 1e-25 of the sum.  s <= SMAX and A <= AMAX keep A D_N finite.

For s > SMAX (next to the hot spot), A > AMAX, dso == 0 and A == 0 (bare soil) the kernel keeps the
Gauss-Legendre panels, mirrored here by `panels`.

usage: python tools/check_hotspot_series.py [samples]   prints accuracy against adaptive quadrature, term counts
(per sample and per 32-sample warp) and the share of samples on each path for the benchmark configurations 2 and 3
and for a wide domain."""
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1] / "oracle"))
import spart_oracle as so  # noqa: E402

# must match SPART_HOTSPOT_* in spart_device.cuh
SMAX = 1e3
AMAX = 1e12
SERIES_TOL = 1e-17
NMAX = 96
SPLIT = 0.2


def setup(K, k, LAI, q, dso):
    """A, Cq, alpha as hotspot_integrals forms them (A = Amin and alpha = 0 where dso == 0)."""
    A0 = (K + k) * LAI
    S = np.sqrt(K * k) * LAI
    nz = dso != 0
    with np.errstate(all="ignore"):
        alpha = np.where(nz, dso / q * 2 / (k + K), 0.0)
        Cq = np.where(nz, S / alpha, 0.0)
    A = np.where(nz, A0, A0 - S)
    return A, Cq, alpha, A0 - S


def use_series(A, Cq, alpha):
    """The kernel's branch test; written so that NaN takes the panels."""
    with np.errstate(all="ignore"):
        s = A / alpha
        return (A > 0) & (A <= AMAX) & (alpha > 0) & (s <= SMAX)


def series(A, z, alpha):
    """The kernel's series, lane by lane: returns (I, N) -- the integral and the number of terms after j = 0."""
    A, z, alpha = (np.asarray(v, dtype=np.float64) for v in (A, z, alpha))
    s = A / alpha
    with np.errstate(all="ignore"):
        big = alpha > 0.5
        v0 = np.where(big, np.exp(-alpha), 1.0 + np.expm1(-alpha))
        omv0 = np.where(big, 1.0 - v0, -np.expm1(-alpha))
        E = z * omv0 - A
        h = np.where(E < -0.5, 1.0 - np.exp(E), -np.expm1(E))
    R = h.copy()
    D = np.ones_like(A)
    pz = z.copy()
    sm = s + 1.0
    live = np.ones(A.shape, bool)
    N = np.zeros(A.shape, int)
    for _ in range(0, NMAX, 2):
        if not live.any():
            break
        for _ in range(2):
            hn = h * v0 + omv0
            Rn = R * sm + pz * hn
            Dn = D * sm
            smn = sm + 1.0
            pn = pz * z
            h, R, D, sm, pz = (np.where(live, a, b) for a, b in ((hn, h), (Rn, R), (Dn, D), (smn, sm), (pn, pz)))
            N += live
        live &= ~(pz <= SERIES_TOL * R * (sm - z))
    return R / (A * D), N


def panels(A, Cq, alpha, Amin):
    """The Gauss-Legendre panels of the kernel (2 x 16 nodes on [-L, 0], analytic remainder below -L)."""
    x16, w16 = np.polynomial.legendre.leggauss(16)
    L = np.ones_like(A)
    with np.errstate(all="ignore"):
        L = np.where(alpha > 0, np.minimum(L, 40.0 / alpha), L)
        L = np.where(Amin > 0, np.minimum(L, 40.0 / Amin), L)
        total = np.zeros_like(A)
        for hw_f, xc_f in ((0.5 * SPLIT, -0.5 * SPLIT), (0.5 * (1 - SPLIT), -0.5 * (1 + SPLIT))):
            hw, xc = hw_f * L, xc_f * L
            x = xc[:, None] + hw[:, None] * x16[None, :]
            f = np.exp(A[:, None] * x + Cq[:, None] * (1 - np.exp(alpha[:, None] * x)))
            total = total + hw * (f * w16).sum(1)
        rem = (L < 1.0) & (alpha * L >= 40.0 * (1 - 1e-12))
        w = 1 - L
        xr = A * w
        f = np.where(xr < 1e-4, w * (1 + xr * (-0.5 + xr / 6)), (1 - np.exp(-xr)) / A)
        total = total + np.where(rem, np.exp(Cq - A * L) * f, 0.0)
    return total


def hotspot(K, k, LAI, q, dso):
    """int_{-1}^0 pso dx as geometry_kernel computes it; returns (I, series_mask, N)."""
    A, Cq, alpha, Amin = setup(*(np.asarray(v, dtype=np.float64) for v in (K, k, LAI, q, dso)))
    ser = use_series(A, Cq, alpha)
    I = panels(A, Cq, alpha, Amin)
    N = np.zeros(A.shape, int)
    if ser.any():
        Is, Ns = series(A[ser], Cq[ser], alpha[ser])
        I[ser] = Is
        N[ser] = Ns
    return I, ser, N


def quad_reference(A, Cq, alpha):
    """Adaptive quadrature (QUADPACK) on 80 panels graded towards the hot spot at x = 0."""
    from scipy import integrate
    edges = np.concatenate([-np.logspace(0, -10, 80), [0.0]])
    out = np.empty(len(A))
    for i, (a, c, al) in enumerate(zip(A, Cq, alpha)):
        f = lambda x: np.exp(a * x - c * np.expm1(al * x))  # noqa: E731
        out[i] = sum(integrate.quad(f, lo, hi, epsabs=0, epsrel=1.2e-14, limit=200)[0]
                      for lo, hi in zip(edges[:-1], edges[1:]))
    return out


def geometry(tts, tto, raa, LAI, a, b):
    """k, K, dso of SAILH (sailh.py:59-97) without the Pso layers of oracle.sail_geometry."""
    rd = np.pi / 180
    col = lambda v: np.asarray(v, dtype=np.float64).reshape(-1, 1)  # noqa: E731
    tts, tto, raa = col(tts), col(tto), col(raa)
    psi_rad = np.abs(raa - 360 * np.round(raa / 360)) * rd
    with np.errstate(invalid="ignore"):
        dso = np.sqrt(np.tan(tts * rd) ** 2 + np.tan(tto * rd) ** 2
                      - 2 * np.tan(tts * rd) * np.tan(tto * rd) * np.cos(psi_rad))
    chi_s, chi_o, _, _ = so.volscatt(np.sin(tts * rd), np.cos(tts * rd), np.sin(tto * rd), np.cos(tto * rd), psi_rad,
                                     np.sin(so.LITAB * rd)[None, :], np.cos(so.LITAB * rd)[None, :])
    lidf = so.leafangles(a, b)
    k = ((chi_s / np.cos(tts * rd)) * lidf).sum(1)
    K = ((chi_o / np.cos(tto * rd)) * lidf).sum(1)
    return K, k, dso.ravel()


def config_inputs(config, n, seed):
    """(K, k, LAI, q, dso) of oracle.synthetic_params(n, config, seed)."""
    P = so.synthetic_params(n, config, seed=seed)
    K, k, dso = geometry(P[:, so.SZA], P[:, so.VZA], P[:, so.RAA], P[:, so.LAI], P[:, so.LIDFA], P[:, so.LIDFB])
    return K, k, P[:, so.LAI], P[:, so.HOT_Q], dso


def wide_inputs(n, seed):
    """Zenith 0-85, view 0-60, azimuth 0-180 degrees, LAI 1e-3-20 and q 1e-4-1 log-uniform, |a|, |b| <= 0.5."""
    rng = np.random.default_rng(seed)
    u = rng.uniform
    LAI, q = 10 ** u(-3, np.log10(20), n), 10 ** u(-4, 0, n)
    K, k, dso = geometry(u(0, 85, n), u(0, 60, n), u(0, 180, n), LAI, u(-0.5, 0.5, n), u(-0.5, 0.5, n))
    return K, k, LAI, q, dso


def study(inputs, n_quad):
    """Accuracy against quadrature on the first n_quad samples, term counts and path shares on all of them."""
    K, k, LAI, q, dso = inputs
    I, ser, N = hotspot(K, k, LAI, q, dso)
    A, Cq, alpha, Amin = setup(K, k, LAI, q, dso)
    sel = np.arange(min(n_quad, len(I)))
    sel = sel[dso[sel] != 0]
    ref = quad_reference(A[sel], Cq[sel], alpha[sel])
    err = np.abs(I[sel] - ref) / ref
    old = panels(A, Cq, alpha, Amin)
    warps = len(N) // 32
    wN = N[:warps * 32].reshape(warps, 32).max(1)
    wfb = (~ser[:warps * 32]).reshape(warps, 32).any(1)
    return dict(err_series=float(err[ser[sel]].max(initial=0.0)), err_panels=float(err[~ser[sel]].max(initial=0.0)),
                n_series_checked=int(ser[sel].sum()), n_panels_checked=int((~ser[sel]).sum()),
                series_vs_panels=float((np.abs(I - old) / old)[ser].max(initial=0.0)),
                share_series=float(ser.mean()), terms_max=int(N.max()), terms_p50=float(np.median(N[ser])),
                warp_terms_mean=float(wN.mean()), warp_terms_max=int(wN.max()), warps_with_panels=float(wfb.mean()),
                z_max_series=float(Cq[ser].max(initial=0.0)))


def main(n=20000, n_quad=200):
    for name, inputs in (("config 2", config_inputs(2, n, 5)), ("config 3", config_inputs(3, n, 5)),
                         ("wide", wide_inputs(n, 3))):
        r = study(inputs, n_quad)
        print(name, " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in r.items()))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 20000)
