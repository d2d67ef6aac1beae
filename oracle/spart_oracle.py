"""CPU oracle for the SPART forward path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

This file is a NumPy restatement (vectorised over samples) of the algorithm in the
reference wirrell/SPART-python.  Only tests/, __graft_entry__.smoke() and the
`cpu_baseline` / `--impl reference` legs of bench.py may import it; the product package
(spart-python_b200/) never does and fails loudly when its CUDA library is missing.

Parity status: PINNED.  tools/make_golden.py runs the unmodified reference in the build
container (one fresh SPART object per sample, np.float64 scalar inputs) and commits its
outputs under tests/golden/; tests/test_oracle_golden.py checks this restatement against
them (O1 = raw reference, O2 = reference with only its quadrature-based expint swapped
for scipy.special.exp1, SURVEY.md section 8(c)).

Every function cites the reference file:line it follows.  Deliberate differences, all
below the 1e-9 gate and documented in DESIGN.md:
  * E1 is scipy.special.exp1 (what prospect_5d.py:186-188 documents) instead of a
    QUADPACK qagie call per wavelength (prospect_5d.py:192), i.e. the oracle is "O2";
  * the 61 hot-spot panel integrals (sailh.py:131-135) use one 21-point Gauss-Kronrod
    panel each, which is what QUADPACK qagse evaluates before it accepts (it accepts
    after one panel for every realistic input, SURVEY.md row a9).

Parameter layout of a batch: float64 array [n, 27], columns
  0..8   leaf    Cab Cdm Cw Cs Cca Cant N PROT CBC      (prospect_5d.py:73-81)
  9..14  soil    B lat lon SMp SMC film                 (bsm.py:269-287)
  15..18 canopy  LAI LIDFa LIDFb q                      (sailh.py:340-348)
  19..21 angles  sol_angle obs_angle rel_angle [deg]    (sailh.py:298-301)
  22..25 atm     aot550 uo3 uh2o Pa                     (smac.py:307-317)
  26     DOY                                            (SPART.py:83)
"""
from pathlib import Path

import numpy as np
from scipy.special import exp1 as _exp1

DATA_DIR = Path(__file__).resolve().parents[1] / "spart-python_b200" / "spart_b200" / "data"

NPAR = 27
(CAB, CDM, CW, CS, CCA, CANT, NSTRUCT, PROT, CBC,
 SOIL_B, SOIL_LAT, SOIL_LON, SMP, SMC, FILM,
 LAI, LIDFA, LIDFB, HOT_Q,
 SZA, VZA, RAA,
 AOT550, UO3, UH2O, PA,
 DOY) = range(NPAR)

NWL_P = 2001  # 400..2400 nm, SPART.py:303
NWL_T = 161   # thermal padding, SPART.py:307-309
NWL_S = NWL_P + NWL_T

SENSORS = [
    "TerraAqua-MODIS", "LANDSAT4-TM", "LANDSAT5-TM", "LANDSAT7-ETM", "LANDSAT8-OLI",
    "Sentinel2A-MSI", "Sentinel2B-MSI", "Sentinel3A-OLCI", "Sentinel3B-OLCI",
]


# ----------------------------------------------------------------------------- tables
def load_optical(data_dir=DATA_DIR):
    """optical_params.pkl + ET_irradiance.pkl content (SPART.py:399-416)."""
    with np.load(Path(data_dir) / "optical.npz") as z:
        return {k: z[k] for k in z.files}


def load_sensor(name, data_dir=DATA_DIR):
    """sensor_information/<name>.pkl content (SPART.py:419-424); raises FileNotFoundError
    for an unknown sensor exactly like the reference's open()."""
    path = Path(data_dir) / "sensors" / f"{name}.npz"
    if not path.exists():
        raise FileNotFoundError(str(path))
    with np.load(path) as z:
        coef = {k.split(".", 1)[1]: z[k] for k in z.files if k.startswith("SMAC_coef.")}
        return {
            "SMAC_coef": coef,
            "wl_smac": z["wl_smac"],
            "wl_srf_smac": z["wl_srf_smac"],
            "p_srf_smac": z["p_srf_smac"],
            "band_id_smac": [str(b) for b in z["band_id_smac"]],
        }


def spectral_wlS():
    """SpectralBands.wlS (SPART.py:303-310)."""
    wlO = np.arange(400, 2401, 1)
    wlT = np.concatenate([np.arange(2500, 15001, 100), np.arange(16000, 50001, 1000)])
    return np.concatenate([wlO, wlT])


# --------------------------------------------------------------------------- PROSPECT
def calculate_tav(alpha, nr):
    """Stern/Allen average interface transmissivity (prospect_5d.py:249-311)."""
    rd = np.pi / 180
    n2 = nr ** 2
    n_p = n2 + 1
    nm = n2 - 1
    a = (nr + 1) * (nr + 1) / 2
    k = -(n2 - 1) * (n2 - 1) / 4
    sa = np.sin(alpha * rd)
    b1 = 0
    if alpha != 90:
        b1 = np.sqrt((sa ** 2 - n_p / 2) * (sa ** 2 - n_p / 2) + k)
    b2 = sa ** 2 - n_p / 2
    b = b1 - b2
    b3 = b ** 3
    a3 = a ** 3
    ts = (k ** 2 / (6 * b3) + k / b - b / 2) - (k ** 2 / (6 * a3) + k / a - a / 2)
    tp1 = -2 * n2 * (b - a) / (n_p ** 2)
    tp2 = -2 * n2 * n_p * np.log(b / a) / (nm ** 2)
    tp3 = n2 * (1 / b - 1 / a) / 2
    tp4 = (16 * n2 ** 2 * (n2 ** 2 + 1)
           * np.log((2 * n_p * b - nm ** 2) / (2 * n_p * a - nm ** 2))
           / (n_p ** 3 * nm ** 2))
    tp5 = 16 * n2 ** 3 * (1 / (2 * n_p * b - nm ** 2) - 1 / (2 * n_p * a - nm ** 2)) / n_p ** 3
    tp = tp1 + tp2 + tp3 + tp4 + tp5
    return (ts + tp) / (2 * sa ** 2)


def _col(tab, idx):
    """Table column [2001,1] -> row vector [1, nl] at wavelength indices idx."""
    v = tab[:, 0] if tab.ndim == 2 else tab
    return v[idx][None, :]


def prospect(leaf, opt, idx=None, expint=_exp1):
    """PROSPECT-5D / PROSPECT-PRO (prospect_5d.py:117-246), batched.

    leaf: [n, 9] columns Cab Cdm Cw Cs Cca Cant N PROT CBC.
    Returns refl, tran, kChlrel, each [n, nl] at wavelength indices `idx` (all 2001 if None).
    """
    if idx is None:
        idx = np.arange(NWL_P)
    leaf = np.asarray(leaf, dtype=np.float64)
    Cab, Cdm, Cw, Cs, Cca, Cant, N, PROTc, CBCc = (leaf[:, i:i + 1] for i in range(9))
    # prospect_5d.py:148-155 -- PROSPECT-PRO switch zeroes Cdm
    pro = ((PROTc > 0.0) | (CBCc > 0.0)) & (Cdm > 0)
    Cdm = np.where(pro, 0.0, Cdm)

    nr = _col(opt["nr"], idx)
    Kab, Kca, Kdm, Kw, Ks, Kant = (_col(opt[k], idx) for k in ("Kab", "Kca", "Kdm", "Kw", "Ks", "Kant"))
    kcbc, kprot = _col(opt["cbc"], idx), _col(opt["prot"], idx)

    with np.errstate(all="ignore"):
        # prospect_5d.py:170-179
        Kall = (Cab * Kab + Cca * Kca + Cdm * Kdm + Cw * Kw + Cs * Ks + Cant * Kant
                + CBCc * kcbc + PROTc * kprot) / N
        pos = Kall > 0
        Ksafe = np.where(pos, Kall, 1.0)
        t1 = (1 - Kall) * np.exp(-Kall)
        t2 = Kall ** 2 * expint(Ksafe)
        tau = np.where(pos, t1 + t2, 1.0)                         # :195-196
        kChlrel = np.where(pos, Cab * Kab / (Ksafe * N), 0.0)     # :197-198

        t_alph = calculate_tav(40, nr)                            # :200-205
        r_alph = 1 - t_alph
        t12 = calculate_tav(90, nr)
        r12 = 1 - t12
        t21 = t12 / (nr ** 2)
        r21 = 1 - t21

        denom = 1 - r21 * r21 * tau ** 2                          # :208-214
        Ta = t_alph * tau * t21 / denom
        Ra = r_alph + r21 * tau * Ta
        t = t12 * tau * t21 / denom
        r = r12 + r21 * tau * t

        D = np.sqrt((1 + r + t) * (1 + r - t) * (1 - r + t) * (1 - r - t))   # :219-230
        rq = r ** 2
        tq = t ** 2
        a = (1 + rq - tq + D) / (2 * r)
        b = (1 - rq + tq + D) / (2 * t)
        bNm1 = b ** (N - 1)
        bN2 = bNm1 ** 2
        a2 = a ** 2
        denom = a2 * bN2 - 1
        Rsub = a * (bN2 - 1) / denom
        Tsub = bNm1 * (a2 - 1) / denom

        j = (r + t) >= 1                                          # :233-235
        Tsub0 = t / (t + (1 - t) * (N - 1))
        Tsub = np.where(j, Tsub0, Tsub)
        Rsub = np.where(j, 1 - Tsub0, Rsub)

        denom = 1 - Rsub * r                                      # :239-241
        tran = Ta * Tsub / denom
        refl = Ra + Ta * Rsub * t / denom
    return refl, tran, kChlrel


# -------------------------------------------------------------------------------- BSM
def _poisson_pmf(k, mu):
    """scipy.stats.poisson.pmf(k, mu) (bsm.py:121) = exp(-mu) mu^k / k!  (matches to 5e-15)."""
    fact = np.array([1.0, 1.0, 2.0, 6.0, 24.0, 120.0, 720.0])[k]
    return np.exp(-mu) * mu ** k / fact


def bsm(soil, opt, idx=None, rdry_user=None):
    """BSM soil reflectance (bsm.py:17-128), batched.  soil: [n, 6] B lat lon SMp SMC film.
    rdry_user: optional dry-soil spectrum [2001] replacing the soil-vector model (bsm.py:42-43).
    Returns (rwet, rdry), each [n, nl]."""
    if idx is None:
        idx = np.arange(NWL_P)
    soil = np.asarray(soil, dtype=np.float64)
    B, lat, lon, SMp, SMCc, film = (soil[:, i:i + 1] for i in range(6))
    GSV = opt["GSV"]
    f1 = B * np.sin(lat * np.pi / 180)                                     # bsm.py:49-52
    f2 = B * np.cos(lat * np.pi / 180) * np.sin(lon * np.pi / 180)
    f3 = B * np.cos(lat * np.pi / 180) * np.cos(lon * np.pi / 180)
    rdry = f1 * GSV[idx, 0][None, :] + f2 * GSV[idx, 1][None, :] + f3 * GSV[idx, 2][None, :]
    if rdry_user is not None:
        rdry = np.repeat(np.asarray(rdry_user, dtype=np.float64).reshape(-1)[idx][None, :], soil.shape[0], axis=0)
    kw = _col(opt["Kw"], idx)
    nw = _col(opt["nw"], idx)

    # soilwat, bsm.py:62-128
    mu = (SMp - 5) / SMCc
    wet = mu > 0
    mu_s = np.where(wet, mu, 1.0)
    rbac = 1 - (1 - rdry) * (rdry * calculate_tav(90, 2 / nw) / calculate_tav(90, 2) + 1 - rdry)
    p = 1 - calculate_tav(90, nw) / nw ** 2
    Rw = 1 - calculate_tav(40, nw)
    rwet = rdry * _poisson_pmf(0, mu_s)
    for k in range(1, 7):
        tw = np.exp(-2 * kw * film * k)
        Rwet_k = Rw + (1 - Rw) * (1 - p) * tw * rbac / (1 - p * tw * rbac)
        rwet = rwet + Rwet_k * _poisson_pmf(k, mu_s)
    rwet = np.where(wet, rwet, rdry)                                       # bsm.py:102-103
    return rwet, rdry


# ------------------------------------------------------------------------------ SAILH
LITAB = np.array([*range(5, 80, 10), *range(81, 91, 2)], dtype=np.float64)  # sailh.py:49


def leafangles(LIDFa, LIDFb):
    """calculate_leafangles (sailh.py:351-398), batched -> lidf [n, 13].

    The fixed-point loop of dcum (sailh.py:374-383) is reproduced iteration for
    iteration, including its stop at abs(dx) <= 1e-8 and the use of the *last computed*
    y (from x before its final update)."""
    a = np.asarray(LIDFa, dtype=np.float64).reshape(-1)
    b = np.asarray(LIDFb, dtype=np.float64).reshape(-1)
    n = a.shape[0]
    rd = np.pi / 180
    F = np.zeros((n, 14))
    thetas = [i * 10 for i in range(1, 9)] + [80 + (i - 8) * 2 for i in range(9, 13)]
    for i, theta in enumerate(thetas, start=1):
        x = np.full(n, 2 * rd * theta)
        theta2 = x.copy()
        y = np.zeros(n)
        delx = np.ones(n)
        act = delx > 1e-8
        while act.any():
            ynew = a * np.sin(x) + 0.5 * b * np.sin(2 * x)
            dx = 0.5 * (ynew - x + theta2)
            x = np.where(act, x + dx, x)
            y = np.where(act, ynew, y)
            delx = np.where(act, np.abs(dx), delx)
            act = delx > 1e-8
        f = (2 * y + theta2) / np.pi
        f = np.where(a > 1, 1 - np.cos(theta * rd), f)             # sailh.py:371-372
        F[:, i] = f
    F[:, 13] = 1
    return np.diff(F, axis=1)


def volscatt(sin_tts, cos_tts, sin_tto, cos_tto, psi_rad, sin_ttli, cos_ttli):
    """_volscatt (sailh.py:401-446); scalars are [n,1], leaf classes [1,13]."""
    cos_psi = np.cos(psi_rad)
    Cs = cos_ttli * cos_tts
    Ss = sin_ttli * sin_tts
    Co = cos_ttli * cos_tto
    So = sin_ttli * sin_tto
    As = np.maximum(Ss, Cs)
    Ao = np.maximum(So, Co)
    bts = np.arccos(-Cs / As)
    bto = np.arccos(-Co / Ao)
    chi_o = 2 / np.pi * ((bto - np.pi / 2) * Co + np.sin(bto) * So)
    chi_s = 2 / np.pi * ((bts - np.pi / 2) * Cs + np.sin(bts) * Ss)
    delta1 = np.abs(bts - bto)
    delta2 = np.pi - np.abs(bts + bto - np.pi)
    Tot = psi_rad + delta1 + delta2
    bt1 = np.minimum(psi_rad, delta1)
    bt3 = np.maximum(psi_rad, delta2)
    bt2 = Tot - bt1 - bt3
    T1 = 2 * Cs * Co + Ss * So * cos_psi
    T2 = np.sin(bt2) * (2 * As * Ao + Ss * So * np.cos(bt1) * np.cos(bt3))
    Jmin = bt2 * T1 - T2
    Jplus = (np.pi - bt2) * T1 + T2
    frho = np.maximum(0.0, Jplus / (2 * np.pi ** 2))
    ftau = np.maximum(0.0, -Jmin / (2 * np.pi ** 2))
    return chi_s, chi_o, frho, ftau


# 21-point Gauss-Kronrod rule (QUADPACK qk21): abscissae and weights on [-1, 1].
_XGK = np.array([
    0.995657163025808080735527280689003, 0.973906528517171720077964012084452,
    0.930157491355708226001207180059508, 0.865063366688984510732096688423493,
    0.780817726586416897063717578345042, 0.679409568299024406234327365114874,
    0.562757134668604683339000099272694, 0.433395394129247190799265943165784,
    0.294392862701460198131126603103866, 0.148874338981631210884826001129720,
    0.0])
_WGK = np.array([
    0.011694638867371874278064396062192, 0.032558162307964727478818972459390,
    0.054755896574351996031381300244580, 0.075039674810919952767043140916190,
    0.093125454583697605535065465083366, 0.109387158802297641899210590325805,
    0.123491976262065851077958109585166, 0.134709217311473325928054001771707,
    0.142775938577060080797094273138717, 0.147739104901338491374841515972068,
    0.149445554002916905664936468389821])
GK21_X = np.concatenate([-_XGK[:10], [0.0], _XGK[:10][::-1]])
GK21_W = np.concatenate([_WGK[:10], [_WGK[10]], _WGK[:10][::-1]])


def pso_panels(K, k, LAI, q, dso, nl=60):
    """Pso[j], j=0..nl (sailh.py:116-135): mean of Psofunction over [xl[j]-dx, xl[j]].
    Inputs [n,1]; returns [n, nl+1]."""
    dx = 1.0 / nl
    xl = np.arange(0, -1 - (1 / nl), -1 / nl)                        # sailh.py:52
    centr = (xl - dx / 2)[None, :, None]                              # [1, 61, 1]
    x = centr + (dx / 2) * GK21_X[None, None, :]                      # [1, 61, 21]
    K3, k3, L3 = K[:, :, None], k[:, :, None], LAI[:, :, None]
    nz = (dso != 0)[:, :, None]
    dso_s = np.where(dso != 0, dso, 1.0)[:, :, None]
    with np.errstate(all="ignore"):
        alpha = (dso_s / q[:, :, None]) * 2 / (k3 + K3)               # sailh.py:121
        p_a = np.exp((K3 + k3) * L3 * x + np.sqrt(K3 * k3) * L3 / alpha * (1 - np.exp(x * alpha)))
        p_b = np.exp((K3 + k3) * L3 * x - np.sqrt(K3 * k3) * L3 * x)  # sailh.py:127
    pso = np.where(nz, p_a, p_b)
    return (pso * GK21_W[None, None, :]).sum(axis=2) * (dx / 2) / dx


def sail_geometry(canopy, angles, lidf=None):
    """Per-sample (wavelength independent) part of SAILH (sailh.py:46-135)."""
    canopy = np.asarray(canopy, dtype=np.float64)
    angles = np.asarray(angles, dtype=np.float64)
    LAIc, LIDFa, LIDFb, q = (canopy[:, i:i + 1] for i in range(4))
    tts, tto, rel = (angles[:, i:i + 1] for i in range(3))
    if lidf is None:
        lidf = leafangles(LIDFa, LIDFb)
    deg2rad = np.pi / 180
    psi = np.abs(rel - 360 * np.round(rel / 360))                     # sailh.py:65
    psi_rad = psi * deg2rad
    sin_tts, cos_tts, tan_tts = np.sin(tts * deg2rad), np.cos(tts * deg2rad), np.tan(tts * deg2rad)
    sin_tto, cos_tto, tan_tto = np.sin(tto * deg2rad), np.cos(tto * deg2rad), np.tan(tto * deg2rad)
    sin_ttli = np.sin(LITAB * deg2rad)[None, :]
    cos_ttli = np.cos(LITAB * deg2rad)[None, :]
    with np.errstate(invalid="ignore"):
        dso = np.sqrt(tan_tts ** 2 + tan_tto ** 2 - 2 * tan_tts * tan_tto * np.cos(psi_rad))  # :78
    chi_s, chi_o, frho, ftau = volscatt(sin_tts, cos_tts, sin_tto, cos_tto, psi_rad, sin_ttli, cos_ttli)
    ksli = chi_s / cos_tts
    koli = chi_o / cos_tto
    sobli = frho * np.pi / (cos_tts * cos_tto)
    sofli = ftau * np.pi / (cos_tts * cos_tto)
    bfli = cos_ttli ** 2
    k = (ksli * lidf).sum(1, keepdims=True)                           # sailh.py:93-97
    K = (koli * lidf).sum(1, keepdims=True)
    bf = (bfli * lidf).sum(1, keepdims=True)
    sob = (sobli * lidf).sum(1, keepdims=True)
    sof = (sofli * lidf).sum(1, keepdims=True)
    Pso = pso_panels(K, k, LAIc, q, dso)
    return dict(LAI=LAIc, k=k, K=K, bf=bf, sob=sob, sof=sof, dso=dso, Pso=Pso, lidf=lidf)


def sailh(rs, rho, tau, canopy, angles, lidf=None, geo=None):
    """SAILH (sailh.py:14-237) on [n, nl] soil/leaf spectra -> rso, rdo, rsd, rdd [n, nl]."""
    g = geo if geo is not None else sail_geometry(canopy, angles, lidf)
    LAIc, k, K, bf, sob, sof, Pso = g["LAI"], g["k"], g["K"], g["bf"], g["sob"], g["sof"], g["Pso"]
    nl = 60
    iLAI = LAIc * (1 / nl)
    sdb = 0.5 * (k + bf)                                              # sailh.py:100-105
    sdf = 0.5 * (k - bf)
    ddb = 0.5 * (1 + bf)
    ddf = 0.5 * (1 - bf)
    dob = 0.5 * (K + bf)
    dof = 0.5 * (K - bf)
    with np.errstate(all="ignore"):
        sigb = ddb * rho + ddf * tau                                  # sailh.py:142-152
        sigf = ddf * rho + ddb * tau
        sb = sdb * rho + sdf * tau
        sf = sdf * rho + sdb * tau
        vb = dob * rho + dof * tau
        vf = dof * rho + dob * tau
        w = sob * rho + sof * tau
        a = 1 - sigf
        m = np.sqrt(a ** 2 - sigb ** 2)
        rinf = (a - m) / sigb
        rinf2 = rinf * rinf

        def calcJ1(x, m, k, LAI):                                     # sailh.py:154-170
            sing = np.abs((m - k) * LAI) < 1e-6
            JN = (np.exp(m * LAI * x) - np.exp(k * LAI * x)) / (k - m)
            JS = -0.5 * (np.exp(m * LAI * x) + np.exp(k * LAI * x)) * LAI * x * (
                1 - 1 / 12 * (k - m) ** 2 * LAI ** 2)
            return np.where(sing, JS, JN)

        def calcJ2(x, m, k, LAI):                                     # sailh.py:172-177
            return (np.exp(k * LAI * x) - np.exp(-k * LAI) * np.exp(-m * LAI * (1 + x))) / (k + m)

        J1k = calcJ1(-1, m, k, LAIc)                                  # sailh.py:180-233
        J2k = calcJ2(0, m, k, LAIc)
        J1K = calcJ1(-1, m, K, LAIc)
        J2K = calcJ2(0, m, K, LAIc)
        e1 = np.exp(-m * LAIc)
        e2 = e1 ** 2
        re = rinf * e1
        denom = 1 - rinf2 ** 2
        s1 = sf + rinf * sb
        s2 = sf * rinf + sb
        v1 = vf + rinf * vb
        v2 = vf * rinf + vb
        Pss = s1 * J1k
        Qss = s2 * J2k
        Poo = v1 * J1K
        Qoo = v2 * J2K
        tau_ss = np.exp(-k * LAIc)
        tau_oo = np.exp(-K * LAIc)
        Z = (1 - tau_ss * tau_oo) / (K + k)
        tau_dd = (1 - rinf2) * e1 / denom
        rho_dd = rinf * (1 - e2) / denom
        tau_sd = (Pss - re * Qss) / denom
        tau_do = (Poo - re * Qoo) / denom
        rho_sd = (Qss - re * Pss) / denom
        rho_do = (Qoo - re * Poo) / denom
        T1 = v2 * s1 * (Z - J1k * tau_oo) / (K + m) + v1 * s2 * (Z - J1K * tau_ss) / (k + m)
        T2 = -(Qoo * rho_sd + Poo * tau_sd) * rinf
        rho_sod = (T1 + T2) / (1 - rinf2)
        rho_sos = w * Pso[:, 0:nl].sum(1, keepdims=True) * iLAI
        rho_so = rho_sod + rho_sos
        Pso2w = Pso[:, nl:nl + 1]
        denom = 1 - rs * rho_dd
        rso = (rho_so + rs * Pso2w
               + ((tau_sd + tau_ss * rs * rho_dd) * tau_oo + (tau_sd + tau_ss) * tau_do) * rs / denom)
        rdo = rho_do + (tau_oo + tau_do) * rs * tau_dd / denom
        rsd = rho_sd + (tau_ss + tau_sd) * rs * tau_dd / denom
        rdd = rho_dd + tau_dd * rs * tau_dd / denom
    return rso, rdo, rsd, rdd


# ------------------------------------------------------------------------------- SMAC
def smac(angles, atm, coefs, terms=False):
    """SMAC (smac.py:14-213), batched: angles [n,3], atm [n,4] (aot550 uo3 uh2o Pa),
    coefs = dict of [1, nb] arrays in their native dtype.  Returns dict of nine [n, nb].
    terms=True adds the summands the sums Ra_so, Ta_s and Ta_o are formed of (lists under "Ra_so_terms",
    "Ta_s_terms", "Ta_o_terms"): what a test needs to judge how ill-conditioned those sums are."""
    angles = np.asarray(angles, dtype=np.float64)
    atm = np.asarray(atm, dtype=np.float64)
    tts, tto, psi = (angles[:, i:i + 1] for i in range(3))
    taup550, uo3, uh2o, Pa = (atm[:, i:i + 1] for i in range(4))
    c = coefs
    cdr = np.pi / 180
    crd = 180 / np.pi
    with np.errstate(all="ignore"):
        us = np.cos(tts * cdr)
        uv = np.cos(tto * cdr)
        Peq = Pa / 1013.25
        m = 1 / us + 1 / uv
        taup = c["a0taup"] + c["a1taup"] * taup550
        uo2 = Peq ** c["po2"]
        uco2 = Peq ** c["pco2"]
        uch4 = Peq ** c["pch4"]
        uno2 = Peq ** c["pno2"]
        uco = Peq ** c["pco"]
        to3 = np.exp(c["ao3"] * (uo3 * m) ** c["no3"])
        th2o = np.exp(c["ah2o"] * (uh2o * m) ** c["nh2o"])
        to2 = np.exp(c["ao2"] * (uo2 * m) ** c["no2"])
        tco2 = np.exp(c["aco2"] * (uco2 * m) ** c["nco2"])
        tch4 = np.exp(c["ach4"] * (uch4 * m) ** c["nch4"])
        tno2 = np.exp(c["ano2"] * (uno2 * m) ** c["nno2"])
        tco = np.exp(c["aco"] * (uco * m) ** c["nco"])
        tg = th2o * to3 * to2 * tco2 * tch4 * tco * tno2
        s = c["a0s"] * Peq + c["a3s"] + c["a1s"] * taup550 + c["a2s"] * taup550 ** 2
        ttetas = c["a0T"] + c["a1T"] * taup550 / us + (c["a2T"] * Peq + c["a3T"]) / (1 + us)
        ttetav = c["a0T"] + c["a1T"] * taup550 / uv + (c["a2T"] * Peq + c["a3T"]) / (1 + uv)
        # smac.py:129-131 -- note cos(psi * crd): degrees multiplied by 180/pi (sic)
        cksi = -((us * uv) + (np.sqrt(1 - us * us) * np.sqrt(1 - uv * uv) * np.cos(psi * crd)))
        cksi = np.where(cksi < -1, -1.0, cksi)
        ksiD = crd * np.arccos(cksi)
        ray_phase = 0.7190443 * (1 + (cksi * cksi)) + 0.0412742
        taur = c["taur"]
        ray_ref = (taur * ray_phase) / (4 * us * uv)
        ray_ref = ray_ref * Pa / 1013.25
        taurz = taur * Peq
        aer_phase = (c["a0P"] + c["a1P"] * ksiD + c["a2P"] * ksiD * ksiD
                     + c["a3P"] * ksiD ** 3 + c["a4P"] * ksiD ** 4)
        wo, gc = c["wo"], c["gc"]
        ak2 = (1 - wo) * (3 - wo * 3 * gc)
        ak = np.sqrt(ak2)
        e = -3 * us * us * wo / (4 * (1 - ak2 * us * us))
        f = -(1 - wo) * 3 * gc * us * us * wo / (4 * (1 - ak2 * us * us))
        dp = e / (3 * us) + us * f
        d = e + f
        b = 2 * ak / (3 - wo * 3 * gc)
        delta = np.exp(ak * taup) * (1 + b) ** 2 - np.exp(-ak * taup) * (1 - b) ** 2
        ww = wo / 4
        ss = us / (1 - ak2 * us * us)
        q1 = 2 + 3 * us + (1 - wo) * 3 * gc * us * (1 + 2 * us)
        q2 = 2 - 3 * us - (1 - wo) * 3 * gc * us * (1 - 2 * us)
        q3 = q2 * np.exp(-taup / us)
        c1 = ((ww * ss) / delta) * (q1 * np.exp(ak * taup) * (1 + b) + q3 * (1 - b))
        c2 = -((ww * ss) / delta) * (q1 * np.exp(-ak * taup) * (1 - b) + q3 * (1 + b))
        cp1 = c1 * ak / (3 - wo * 3 * gc)
        cp2 = -c2 * ak / (3 - wo * 3 * gc)
        z = d - wo * 3 * gc * uv * dp + wo * aer_phase / 4
        x = c1 - wo * 3 * gc * uv * cp1
        y = c2 - wo * 3 * gc * uv * cp2
        aa1 = uv / (1 + ak * uv)
        aa2 = uv / (1 - ak * uv)
        aa3 = us * uv / (us + uv)
        aer_ref1 = x * aa1 * (1 - np.exp(-taup / aa1))
        aer_ref2 = y * aa2 * (1 - np.exp(-taup / aa2))
        aer_ref3 = z * aa3 * (1 - np.exp(-taup / aa3))
        aer_ref = (aer_ref1 + aer_ref2 + aer_ref3) / (us * uv)
        Res_ray = (c["Resr1"] + c["Resr2"] * taur * ray_phase / (us * uv)
                   + c["Resr3"] * ((taur * ray_phase / (us * uv)) ** 2))
        Res_aer = ((c["Resa1"] + c["Resa2"] * (taup * m * cksi) + c["Resa3"] * ((taup * m * cksi) ** 2))
                   + c["Resa4"] * (taup * m * cksi) ** 3)
        tautot = taup + taurz
        Res_6s = ((c["Rest1"] + c["Rest2"] * (tautot * m * cksi) + c["Rest3"] * ((tautot * m * cksi) ** 2))
                  + c["Rest4"] * ((tautot * m * cksi) ** 3))
        atm_ref = ray_ref - Res_ray + aer_ref - Res_aer + Res_6s
        tdir_tts = np.exp(-tautot / us)
        tdir_ttv = np.exp(-tautot / uv)
        tdif_tts = ttetas - tdir_tts
        tdif_ttv = ttetav - tdir_ttv
    out = dict(Ta_s=ttetas, Ta_o=ttetav, Tg=tg, Ra_dd=s, Ra_so=atm_ref,
               Ta_ss=tdir_tts, Ta_sd=tdif_tts, Ta_oo=tdir_ttv, Ta_do=tdif_ttv)
    if terms:
        with np.errstate(all="ignore"):
            out["Ra_so_terms"] = [ray_ref, Res_ray, aer_ref1 / (us * uv), aer_ref2 / (us * uv), aer_ref3 / (us * uv),
                                  Res_aer, Res_6s]
            out["Ta_s_terms"] = [c["a0T"], c["a1T"] * taup550 / us, (c["a2T"] * Peq + c["a3T"]) / (1 + us)]
            out["Ta_o_terms"] = [c["a0T"], c["a1T"] * taup550 / uv, (c["a2T"] * Peq + c["a3T"]) / (1 + uv)]
    return out


# ----------------------------------------------------- ET irradiance + SRF convolution
def closest_index(wl_srf, wl_hi):
    """get_closest_index (SPART.py:381-387): for every SRF wavelength (column-major
    flattening) the index of the nearest entry of wl_hi; first minimum on ties, 0 for NaN."""
    V = np.reshape(wl_srf, (wl_srf.shape[0] * wl_srf.shape[1],), order="F")
    N = np.asarray(wl_hi, dtype=np.float64).reshape(-1)
    out = np.empty(V.shape[0], dtype=np.int64)
    with np.errstate(invalid="ignore"):
        for s in range(0, V.shape[0], 512):
            A = np.abs(N[:, None] - V[None, s:s + 512])
            out[s:s + 512] = np.argmin(A, 0)
    return out.reshape(wl_srf.shape, order="F")


def et_correction(doy):
    """Sun-earth distance factor (SPART.py:345-352, DOY / 365)."""
    b = 2 * np.pi * doy / 365
    return (1.00011 + 0.034221 * np.cos(b) + 0.00128 * np.sin(b)
            + 0.000719 * np.cos(2 * b) + 0.000077 * np.sin(2 * b))


def et_band_radiance(doy, tts, opt, sensor):
    """calculate_ET_radiance + calculate_spectral_convolution (SPART.py:318-396), batched
    and faithful: the per-sample spectrum is gathered and SRF-weighted.  -> La [n, nb]."""
    doy = np.asarray(doy, dtype=np.float64).reshape(-1, 1)
    tts = np.asarray(tts, dtype=np.float64).reshape(-1, 1)
    Ea = opt["Ea"][:, 0][None, :]
    Ra = Ea * et_correction(doy) * np.cos(tts * np.pi / 180) / np.pi        # [n, 2001]
    idx = closest_index(sensor["wl_srf_smac"], opt["wl_Ea"])
    p = sensor["p_srf_smac"]
    rad = Ra[:, idx]                                                         # [n, n_srf, nb]
    return np.sum(rad * p[None], axis=1) / np.sum(p, axis=0)[None, :]


# ------------------------------------------------------------------ thermal padding
def pad_soil(rs):
    """set_soil_refl_trans_assumptions (SPART.py:427-442): thermal = value at 2400 nm."""
    return np.concatenate([rs, np.repeat(rs[:, -1:], NWL_T, axis=1)], axis=1)


def pad_leaf(x, thermal=0.01):
    """set_leaf_refl_trans_assumptions (SPART.py:445-470): thermal rho = tau = 0.01."""
    return np.concatenate([x, np.full((x.shape[0], NWL_T), thermal)], axis=1)


# ------------------------------------------------------------------------ full chain
def band_sample_points(wl_smac):
    """Indices/weights np.interp(wl_smac, wlS, .) touches (SPART.py:216-223).
    Returns lo index, hi index, fractional offset (x - xp[lo]) for each band."""
    wlS = spectral_wlS().astype(np.float64)
    x = np.asarray(wl_smac, dtype=np.float64).reshape(-1)
    lo = np.clip(np.searchsorted(wlS, x, side="right") - 1, 0, NWL_S - 1)
    frac = x - wlS[lo]
    hi = np.where(frac == 0, lo, np.minimum(lo + 1, NWL_S - 1))   # a knot hit needs no neighbour
    return lo, hi, frac


def toc_to_toa(rv_so, rv_do, rv_dd, rv_sd, atmo, La):
    """TOC -> TOA algebra (SPART.py:235-252)."""
    ta_ss, ta_sd, ta_oo, ta_do = atmo["Ta_ss"], atmo["Ta_sd"], atmo["Ta_oo"], atmo["Ta_do"]
    ra_dd, ra_so, T_g = atmo["Ra_dd"], atmo["Ra_so"], atmo["Tg"]
    with np.errstate(all="ignore"):
        rtoa0 = ra_so + ta_ss * rv_so * ta_oo
        rtoa1 = ((ta_sd * rv_do + ta_ss * rv_sd * ra_dd * rv_do) * ta_oo / (1 - rv_dd * ra_dd))
        rtoa2 = (ta_ss * rv_sd + ta_sd * rv_dd) * ta_do / (1 - rv_dd * ra_dd)
        R_TOC = (ta_ss * rv_so + ta_sd * rv_do) / (ta_ss + ta_sd)
        R_TOA = T_g * (rtoa0 + rtoa1 + rtoa2)
        L_TOA = La * R_TOA
    return R_TOC, R_TOA, L_TOA


def canopy_spectra(params, opt=None, expint=_exp1, soil_rdry=None):
    """leafopt/soilopt/canopyopt of SPART.run() (SPART.py:189-214) over all 2162
    wavelengths.  Returns dict of [n, 2162] arrays (kChlrel [n, 2001])."""
    params = np.atleast_2d(np.asarray(params, dtype=np.float64))
    opt = opt or load_optical()
    refl, tran, kchl = prospect(params[:, CAB:CBC + 1], opt, expint=expint)
    rwet, rdry = bsm(params[:, SOIL_B:FILM + 1], opt, rdry_user=soil_rdry)
    rho, tau, rs = pad_leaf(refl), pad_leaf(tran), pad_soil(rwet)
    rso, rdo, rsd, rdd = sailh(rs, rho, tau, params[:, LAI:HOT_Q + 1], params[:, SZA:RAA + 1])
    return dict(leaf_refl=rho, leaf_tran=tau, kChlrel=kchl, soil_refl=rs, soil_refl_dry=rdry,
                rso=rso, rdo=rdo, rsd=rsd, rdd=rdd)


def srf_convolve(spectrum, opt, sensor):
    """calculate_spectral_convolution (SPART.py:358-396) applied to [n, >=2001] spectra on the
    400..2400 nm grid -> [n, nb]."""
    idx = closest_index(sensor["wl_srf_smac"], opt["wl_Ea"])
    p = sensor["p_srf_smac"]
    rad = spectrum[:, idx]
    with np.errstate(all="ignore"):
        return np.sum(rad * p[None], axis=1) / np.sum(p, axis=0)[None, :]


def spart_bands(params, sensor, opt=None, faithful=False, expint=_exp1, return_canopy=False, soil_rdry=None,
                band_mode="interp", lidf=None):
    """SPART(...).run() (SPART.py:162-269) for a batch -> [n, nb, 3] = (R_TOC, R_TOA, L_TOA).

    `sensor` is a sensor name or a sensorinfo dict.  faithful=True evaluates the whole
    2162-wavelength spectrum and calls np.interp / the gather-based SRF convolution like
    the reference does; faithful=False evaluates only the wavelengths np.interp touches
    and uses the linearity of the SRF convolution in Ea (identical to ~1e-15).
    return_canopy=True also returns the band-sampled canopy reflectances [n, nb, 4].
    lidf [n, 13]: a leaf inclination distribution assigned to CanopyStructure.lidf after construction, which
    SAILH then uses as is (sailh.py:81-97 read canopy.lidf); default band mode only."""
    params = np.atleast_2d(np.asarray(params, dtype=np.float64))
    opt = opt or load_optical()
    if isinstance(sensor, str):
        sensor = load_sensor(sensor)
    wl = sensor["wl_smac"].T[0]
    if band_mode == "srf":     # extension: SRF-weighted band means of the canopy reflectances
        cs = canopy_spectra(params, opt, expint=expint, soil_rdry=soil_rdry)
        rv = {k: srf_convolve(cs[k], opt, sensor) for k in ("rso", "rdo", "rdd", "rsd")}
        La = et_band_radiance(params[:, DOY], params[:, SZA], opt, sensor)
    elif faithful:
        cs = canopy_spectra(params, opt, expint=expint, soil_rdry=soil_rdry)
        wlS = spectral_wlS()
        rv = {k: np.stack([np.interp(wl, wlS, row) for row in cs[k]]) for k in ("rso", "rdo", "rdd", "rsd")}
        La = et_band_radiance(params[:, DOY], params[:, SZA], opt, sensor)
    else:
        lo, hi, frac = band_sample_points(wl)
        if hi.max() >= NWL_P:
            raise ValueError("band centres beyond 2400 nm need faithful=True")
        idx = np.concatenate([lo, hi])
        refl, tran, _ = prospect(params[:, CAB:CBC + 1], opt, idx, expint=expint)
        rwet, _ = bsm(params[:, SOIL_B:FILM + 1], opt, idx, rdry_user=soil_rdry)
        r4 = sailh(rwet, refl, tran, params[:, LAI:HOT_Q + 1], params[:, SZA:RAA + 1], lidf=lidf)
        nb = lo.shape[0]
        rv = {}
        for name, r in zip(("rso", "rdo", "rsd", "rdd"), r4):
            f0, f1 = r[:, :nb], r[:, nb:]
            # np.interp: exact sample at a knot, else slope * (x - xp[j]) + fp[j], knots 1 nm apart
            with np.errstate(all="ignore"):
                rv[name] = np.where(frac[None, :] == 0, f0, (f1 - f0) / 1.0 * frac[None, :] + f0)
        idxE = closest_index(sensor["wl_srf_smac"], opt["wl_Ea"])
        p = sensor["p_srf_smac"]
        convEa = np.sum(opt["Ea"][:, 0][idxE] * p, axis=0) / np.sum(p, axis=0)
        scale = (et_correction(params[:, DOY:DOY + 1]) * np.cos(params[:, SZA:SZA + 1] * np.pi / 180) / np.pi)
        La = convEa[None, :] * scale
    atmo = smac(params[:, SZA:RAA + 1], params[:, AOT550:PA + 1], sensor["SMAC_coef"])
    R_TOC, R_TOA, L_TOA = toc_to_toa(rv["rso"], rv["rdo"], rv["rdd"], rv["rsd"], atmo, La)
    out = np.stack([R_TOC, R_TOA, L_TOA], axis=2)
    if return_canopy:
        # band-sampled rso, rdo, rsd, rdd [n, nb, 4]: lets tests tell physically valid SAILH
        # output (all four in (0, 1)) from the reference's out-of-range results
        return out, np.stack([rv["rso"], rv["rdo"], rv["rsd"], rv["rdd"]], axis=2)
    return out


# ------------------------------------------------------------ synthetic sensor (config 4)
def synthetic_fullspectrum_sensor():
    """The 2001-band synthetic sensor of SURVEY.md section 8(d): band centres 400..2400 nm,
    SMAC coefficients linearly interpolated in wavelength from TerraAqua-MODIS (sorted by
    wl_smac), top-hat single-wavelength SRF.  Fed unchanged to the reference (as a plain
    sensorinfo dict) and to the CUDA path."""
    modis = load_sensor("TerraAqua-MODIS")
    wl_m = modis["wl_smac"].T[0].astype(np.float64)
    order = np.argsort(wl_m)
    grid = np.arange(400, 2401, 1).astype(np.float64)
    coef = {k: np.interp(grid, wl_m[order], v[0].astype(np.float64)[order])[None, :]
            for k, v in modis["SMAC_coef"].items()}
    return {
        "SMAC_coef": coef,
        "wl_smac": grid[:, None],
        "wl_srf_smac": grid[None, :].copy(),
        "p_srf_smac": np.ones((1, NWL_P)),
        "band_id_smac": [f"{int(w)} nm" for w in grid],
    }


# ------------------------------------------------------------ synthetic parameter batches
def synthetic_params(n, config=2, seed=None):
    """Seeded synthetic parameter batch [n, 27] for BASELINE.json config 2..5
    (distributions of SURVEY.md section 8(d))."""
    rng = np.random.default_rng(20261018 + config if seed is None else seed)
    P = np.zeros((n, NPAR))
    u = rng.uniform
    P[:, CAB] = u(5, 80, n)
    P[:, CCA] = u(1, 25, n)
    P[:, CANT] = u(0, 10, n)
    P[:, CS] = u(0, 0.5, n)
    P[:, CW] = u(0.005, 0.05, n)
    P[:, NSTRUCT] = u(1, 3, n)
    if config == 3:
        P[:, CDM] = 0.0
        P[:, PROT] = u(0, 0.003, n)
        P[:, CBC] = u(0, 0.01, n)
    else:
        P[:, CDM] = u(0.002, 0.02, n)
    P[:, SOIL_B] = u(0.2, 0.8, n)
    P[:, SOIL_LAT] = u(0, 25, n)
    P[:, SOIL_LON] = u(90, 115, n)
    smp = u(5, 55, n)
    dry = u(0, 1, n) < 0.05
    P[:, SMP] = np.where(dry, u(0, 5, n), smp)
    P[:, SMC] = 25.0
    P[:, FILM] = 0.015
    P[:, LAI] = u(0.1, 8, n)
    a = u(-0.5, 0.5, n)
    b = u(-0.5, 0.5, n)
    P[:, LIDFA], P[:, LIDFB] = a, b
    P[:, HOT_Q] = u(0.01, 0.2, n)
    if config == 3:
        P[:, SZA] = u(0, 65, n)
        P[:, VZA] = u(0, 40, n)
        P[:, RAA] = u(0, 180, n)
    else:
        P[:, SZA], P[:, VZA], P[:, RAA] = 40.0, 0.0, 0.0
    P[:, AOT550] = u(0.05, 0.6, n)
    P[:, UO3] = u(0.25, 0.45, n)
    P[:, UH2O] = u(0.5, 4, n)
    P[:, PA] = u(900, 1030, n)
    P[:, DOY] = rng.integers(1, 366, n).astype(np.float64)
    return P
