// spart_device_f32.cuh -- FP32 arithmetic variant of the per-point physics (SPART_FP32 mode).
//
// Target: relative error <= 1e-4 on R_TOC / R_TOA / L_TOA against the FP64 oracle
// (BASELINE.json north_star).  Same equations and reference citations as spart_device.cuh;
// the differences are the ones single precision needs:
//   * the leaf-angle fixed point is solved with a safeguarded Newton iteration (6 steps,
//     |error| < 1e-6) instead of reproducing the reference's 1e-8-truncated iteration, which
//     is below float resolution anyway (sailh.py:374-383);
//   * exp / log / reciprocal use the SFU approximations (MUFU.EX2 / LG2 / RCP);
//   * calcJ1's near-singular series (sailh.py:154-170) takes over at |(m-k) LAI| < 2e-2;
//   * the per-sample SMAC scattering-angle terms stay in FP64 (cos of a ~1e4 rad argument).
#pragma once
#include "spart_device.cuh"

namespace spart {
namespace f32 {

#define SPART_PI_F 3.14159265358979323846f

__constant__ float c_gl10_xf[10] = SPART_GL10_X;
__constant__ float c_gl10_wf[10] = SPART_GL10_W;
__constant__ float c_gl4_xf[4] = SPART_GL4_X;
__constant__ float c_gl4_wf[4] = SPART_GL4_W;

// SFU reciprocal / square root (1-2 ulp, no slow path)
__device__ __forceinline__ float rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float fsqrt(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// 1 - e^z for z <= 0 without cancellation near z = 0
__device__ __forceinline__ float one_minus_exp(float z) {
  if (fabsf(z) < 0.05f) return -z * (1.0f + z * (0.5f + z * (1.0f / 6.0f + z * (1.0f / 24.0f))));
  return 1.0f - __expf(z);
}
__device__ __forceinline__ float fexp(float x) { return __expf(x); }
__device__ __forceinline__ float flog(float x) { return __logf(x); }

// Degree-7 Chebyshev interpolants on the intervals of the FP64 tables (tools/gen_tau_coeffs.py:
// relative error <= 9e-8 with float coefficients, i.e. float epsilon; the FP64 tables are degree 16).
__constant__ float c_tauf_coef[SPART_TAU_NINT][SPART_TAUF_DEG + 1];

struct TauTableF {
  float coef[SPART_TAU_NINT][SPART_TAUF_DEG + 1];
  float mid[SPART_TAU_NINT];
  float invhalf[SPART_TAU_NINT];
};

__device__ __forceinline__ void load_tau_table_f(TauTableF* s) {
  float* dst = reinterpret_cast<float*>(s);
  const int ncoef = SPART_TAU_NINT * (SPART_TAUF_DEG + 1);
  for (int i = threadIdx.x; i < ncoef + 2 * SPART_TAU_NINT; i += blockDim.x) {
    float v;
    if (i < ncoef) v = (&c_tauf_coef[0][0])[i];
    else if (i < ncoef + SPART_TAU_NINT) v = (float)c_tau_mid[i - ncoef];
    else v = (float)c_tau_invhalf[i - ncoef - SPART_TAU_NINT];
    dst[i] = v;
  }
}

// tau(K) = (1-K) e^-K + K^2 E1(K), prospect_5d.py:182-196 (see plate_tau in spart_device.cuh).
// Returns tau and sets omt = 1 - tau, each formed where it has no cancellation.  For a weakly absorbing plate
// (K < 1) 1 - tau is the quantity the leaf absorptance hangs on: (1 - e^-K) + K e^-K - K^2 E1(K).  For a strongly
// absorbing one (K >= 1) tau = e^-K t H(t) is small (7e-11 at K = 21) and a float 1 - (1 - tau) would lose it, down
// to 0 for K > ~14.5, where the N-layer solution then divides by zero.
__device__ __forceinline__ float plate_tau_f(float K, const TauTableF* tab, float& omt) {
  const float emk = fexp(-K);
  int idx;
  float u, t = 0.0f;
  if (K < 1.0f) {
    idx = 0;
    u = 2.0f * K - 1.0f;
  } else {
    t = rcp(K);
    const int e = (__float_as_int(K) >> 23) - 127;
    idx = min(e + 1, SPART_TAU_NINT - 1);
    u = (t - tab->mid[idx]) * tab->invhalf[idx];
  }
  const float* c = tab->coef[idx];
  float p = c[SPART_TAUF_DEG];
#pragma unroll
  for (int i = SPART_TAUF_DEG - 1; i >= 0; --i) p = fmaf(p, u, c[i]);
  if (K < 1.0f) {
    const float e1 = fmaf(K, p, -0.57721566490153286061f - flog(K));
    const float ome = (K < 0.05f) ? K * (1.0f - K * (0.5f - K * (1.0f / 6.0f - K * (1.0f / 24.0f)))) : 1.0f - emk;
    omt = fmaf(K, emk - K * e1, ome);
    return 1.0f - omt;
  }
  const float tau = emk * t * p;
  omt = 1.0f - tau;
  return tau;
}

struct LeafParF {
  float Cab, Cca, Cdm, Cw, Cs, Cant, CBC, PROT, N, invN;
};

template <typename T>
__device__ __forceinline__ LeafParF load_leaf_f(const ParamsT<T>& P, int64_t s) {
  LeafParF L;
  L.Cab = (float)P.at(P_CAB, s);
  L.Cdm = (float)P.at(P_CDM, s);
  L.Cw = (float)P.at(P_CW, s);
  L.Cs = (float)P.at(P_CS, s);
  L.Cca = (float)P.at(P_CCA, s);
  L.Cant = (float)P.at(P_CANT, s);
  L.N = (float)P.at(P_N, s);
  L.PROT = (float)P.at(P_PROT, s);
  L.CBC = (float)P.at(P_CBC, s);
  if ((L.PROT > 0.0f || L.CBC > 0.0f) && L.Cdm > 0.0f) L.Cdm = 0.0f;   // prospect_5d.py:148-155
  L.invN = rcp(L.N);
  return L;
}

// prospect_5d.py:117-246 at one wavelength.  Besides refl / tran the leaf absorptance
// absorb = 1 - refl - tran is returned: the canopy solution depends on it (m^2 = absorb (a + sigb),
// sailh.py:151) and for near-conservative leaves (NIR plateau, refl + tran > 0.98) a float difference of
// refl and tran would lose it.  When the single plate is near-conservative (r + t > 0.9) the N-layer
// Stokes system (prospect_5d.py:219-241), ill-conditioned in 1 - r - t, is solved in FP64 from the
// float plate transmissivity (B200 runs FP64 at half the FP32 rate, and only the NIR bands take this path).
__device__ __forceinline__ void prospect_point_f(const LeafParF& L, const float* lc, const TauTableF* tab,
                                                 float& refl, float& tran, float& absorb) {
  const float Ksum = L.Cab * lc[LC_KAB] + L.Cca * lc[LC_KCA] + L.Cdm * lc[LC_KDM] + L.Cw * lc[LC_KW] +
                     L.Cs * lc[LC_KS] + L.Cant * lc[LC_KANT] + L.CBC * lc[LC_CBC] + L.PROT * lc[LC_PROT];
  const float Kall = Ksum * L.invN;
  float omt = 0.0f, tau = 1.0f;
  if (Kall > 0.0f) tau = plate_tau_f(Kall, tab, omt);
  const float t_alph = lc[LC_TALPH], t12 = lc[LC_T12], t21 = lc[LC_T21];
  const float r_alph = 1.0f - t_alph, r12 = 1.0f - t12, r21 = 1.0f - t21;
  const float tt21 = tau * t21;
  const float inv_d1 = rcp(1.0f - r21 * r21 * tau * tau);
  const float t = t12 * tt21 * inv_d1;
  const float r = r12 + r21 * tau * t;
  if (r + t > 0.9f) {
    double rd, td;
    leaf_from_tau(1.0 - (double)omt, (double)t_alph, (double)t12, (double)t21, (double)L.N, rd, td);
    refl = (float)rd;
    tran = (float)td;
    absorb = (float)(1.0 - rd - td);
    return;
  }
  const float Ta = t_alph * tt21 * inv_d1;
  const float Ra = r_alph + r21 * tau * Ta;
  const float Nm1 = L.N - 1.0f;
  const float D = fsqrt((1.0f + r + t) * (1.0f + r - t) * (1.0f - r + t) * (1.0f - r - t));
  const float rq = r * r, tq = t * t;
  const float a = (1.0f + rq - tq + D) * rcp(2.0f * r);
  const float b = (1.0f - rq + tq + D) * rcp(2.0f * t);
  const float bNm1 = (Nm1 == 0.0f) ? 1.0f : fexp(Nm1 * flog(b));
  const float bN2 = bNm1 * bNm1;
  const float a2 = a * a;
  const float inv_d2 = rcp(a2 * bN2 - 1.0f);
  const float Rsub = a * (bN2 - 1.0f) * inv_d2;
  const float Tsub = bNm1 * (a2 - 1.0f) * inv_d2;
  const float inv_d3 = rcp(1.0f - Rsub * r);
  tran = Ta * Tsub * inv_d3;
  refl = Ra + Ta * Rsub * t * inv_d3;
  absorb = 1.0f - refl - tran;
}

struct SoilParF {
  float f1, f2, f3, mu, emu, film;
};

// bsm.py:99-124 at one wavelength: wet soil from a given dry reflectance
__device__ __forceinline__ float bsm_wet_f(const SoilParF& S, const float* lc, float rdry) {
  if (!(S.mu > 0.0f)) return rdry;
  const float rbac = 1.0f - (1.0f - rdry) * (rdry * lc[LC_SOILC1] + 1.0f - rdry);
  const float p = lc[LC_SOILP], Rw = lc[LC_SOILRW];
  const float tw1 = fexp(-2.0f * lc[LC_KW] * S.film);
  float fk = S.emu;
  float acc = rdry * fk;
  float tw = 1.0f;
  const float g = (1.0f - Rw) * (1.0f - p);
#pragma unroll
  for (int k = 1; k <= 6; ++k) {
    tw *= tw1;
    fk = fk * S.mu * (1.0f / (float)k);
    const float x = tw * rbac;
    acc += (Rw + g * x * rcp(1.0f - p * x)) * fk;
  }
  return acc;
}

// bsm.py:49-52, 99-124 at one wavelength
__device__ __forceinline__ float bsm_point_f(const SoilParF& S, const float* lc) {
  return bsm_wet_f(S, lc, S.f1 * lc[LC_GSV0] + S.f2 * lc[LC_GSV1] + S.f3 * lc[LC_GSV2]);
}

struct CanopyGeoF {
  float LAI, k, K, bf, sob, sof, tau_ss, tau_oo, sumpso, pso2w, Z;
};

__device__ __forceinline__ float sail_J1_f(float m, float k, float LAI, float em, float ek) {
  const float d = (k - m) * LAI;
  if (fabsf(d) < 2e-2f) return 0.5f * (em + ek) * LAI * (1.0f - (1.0f / 12.0f) * d * d);
  return (em - ek) * rcp(k - m);
}

// sailh.py:99-105, 142-233 at one wavelength
// Single-precision forms (tools/fp32_study.py measures each against the float64 oracle): rinf =
// sigb / (a + m) and 1 - rinf^2 = 2 m / (a + m) * rinf replace (a - m) / sigb and the difference, which
// cancel for dark (a ~ m) and for bright (rinf ~ 1) leaves; 1 - e^-x terms switch to their series for
// small x; m^2 = absorb (a + sigb) takes the leaf absorptance from PROSPECT instead of 1 - rho - tau.
__device__ __forceinline__ float omx(float z, float ez) {   // 1 - e^z for z <= 0, ez = e^z already known
  return (z > -0.05f) ? -z * (1.0f + z * (0.5f + z * (1.0f / 6.0f + z * (1.0f / 24.0f)))) : 1.0f - ez;
}

__device__ __forceinline__ void sailh_point_f(const CanopyGeoF& G, float rho, float tau, float absorb, float rs,
                                              float& rso, float& rdo, float& rsd, float& rdd) {
  const float k = G.k, K = G.K, bf = G.bf, LAI = G.LAI;
  const float sdb = 0.5f * (k + bf), sdf = 0.5f * (k - bf);
  const float ddb = 0.5f * (1.0f + bf), ddf = 0.5f * (1.0f - bf);
  const float dob = 0.5f * (K + bf), dof = 0.5f * (K - bf);
  const float sigb = ddb * rho + ddf * tau;
  const float sigf = ddf * rho + ddb * tau;
  const float sb = sdb * rho + sdf * tau;
  const float sf = sdf * rho + sdb * tau;
  const float vb = dob * rho + dof * tau;
  const float vf = dof * rho + dob * tau;
  const float w = G.sob * rho + G.sof * tau;
  const float a = 1.0f - sigf;
  // a^2 - sigb^2 = (1 - rho - tau)(a + sigb) (sigf + sigb = rho + tau)
  const float m = fsqrt(absorb * (a + sigb));
  const float inv_apm = rcp(a + m);
  const float rinf = sigb * inv_apm;                 // (a - m) / sigb, since (a - m)(a + m) = sigb^2
  const float rinf2 = rinf * rinf;
  const float omr2 = 2.0f * m * inv_apm;             // 1 - rinf^2 = ((a + m)^2 - sigb^2) / (a + m)^2 = 2 m / (a + m)
  const float e1 = fexp(-m * LAI);
  const float e2 = e1 * e1;
  const float tau_ss = G.tau_ss, tau_oo = G.tau_oo;
  const float inv_km = rcp(k + m), inv_Km = rcp(K + m);
  const float J1k = sail_J1_f(m, k, LAI, e1, tau_ss);
  const float J2k = omx(-(k + m) * LAI, tau_ss * e1) * inv_km;
  const float J1K = sail_J1_f(m, K, LAI, e1, tau_oo);
  const float J2K = omx(-(K + m) * LAI, tau_oo * e1) * inv_Km;
  const float re = rinf * e1;
  const float inv_den = rcp(omr2 * (1.0f + rinf2));
  const float s1 = sf + rinf * sb, s2 = sf * rinf + sb;
  const float v1 = vf + rinf * vb, v2 = vf * rinf + vb;
  const float Pss = s1 * J1k, Qss = s2 * J2k;
  const float Poo = v1 * J1K, Qoo = v2 * J2K;
  const float Z = G.Z;
  const float tau_dd = omr2 * e1 * inv_den;
  const float rho_dd = rinf * omx(-2.0f * m * LAI, e2) * inv_den;
  const float tau_sd = (Pss - re * Qss) * inv_den;
  const float tau_do = (Poo - re * Qoo) * inv_den;
  const float rho_sd = (Qss - re * Pss) * inv_den;
  const float rho_do = (Qoo - re * Poo) * inv_den;
  const float T1 = v2 * s1 * (Z - J1k * tau_oo) * inv_Km + v1 * s2 * (Z - J1K * tau_ss) * inv_km;
  const float T2 = -(Qoo * rho_sd + Poo * tau_sd) * rinf;
  const float rho_sod = (T1 + T2) * rcp(omr2);
  const float rho_so = rho_sod + w * G.sumpso;
  const float rs_den = rs * rcp(1.0f - rs * rho_dd);
  rso = rho_so + rs * G.pso2w + ((tau_sd + tau_ss * rs * rho_dd) * tau_oo + (tau_sd + tau_ss) * tau_do) * rs_den;
  rdo = rho_do + (tau_oo + tau_do) * tau_dd * rs_den;
  rsd = rho_sd + (tau_ss + tau_sd) * tau_dd * rs_den;
  rdd = rho_dd + tau_dd * tau_dd * rs_den;
}

// sin / cos for |x| up to a few pi: fold to [-pi/2, pi/2] and use the SFU sine / cosine there
// (absolute error ~4e-7), which is what the Newton solve below needs
__device__ __forceinline__ void sincos_sfu(float x, float& s, float& c) {
  const float kf = rintf(x * (1.0f / SPART_PI_F));
  float r = fmaf(-kf, 3.140625f, x);                    // pi = 3.140625 + 9.67653589793e-4 (Cody-Waite)
  r = fmaf(-kf, 9.67653589793e-4f, r);
  const int odd = ((int)kf) & 1;
  const float s0 = __sinf(r), c0 = __cosf(r);
  s = odd ? -s0 : s0;
  c = odd ? -c0 : c0;
}

// Cumulative leaf-angle value F(theta) = (2 y(x*) + theta2) / pi with x* the root of
// y(x) - x + theta2 = 0, y = a sin x + b/2 sin 2x (the fixed point of sailh.py:378-382).
// y - x is monotone decreasing for |a| + |b| <= 1, so Newton is safeguarded by the bracket
// [theta2 - 1.6, theta2 + 1.6]; 6 steps give |F error| < 1e-6 over the whole (a, b) domain.
__device__ __forceinline__ float dcum_newton_f(float a, float b, float theta2) {
  if (a > 1.0f) return 1.0f - cosf(0.5f * theta2);   // sailh.py:371-372
  float lo = theta2 - 1.6f, hi = theta2 + 1.6f, x = theta2;
#pragma unroll 1
  for (int it = 0; it < 6; ++it) {
    float s, c;
    sincos_sfu(x, s, c);
    const float f = s * fmaf(b, c, a) - x + theta2;
    const float fp = fmaf(a, c, b * (2.0f * c * c - 1.0f)) - 1.0f;
    lo = (f > 0.0f) ? x : lo;
    hi = (f < 0.0f) ? x : hi;
    const float xn = x - f * rcp(fp);
    x = (xn >= lo && xn <= hi) ? xn : 0.5f * (lo + hi);
  }
  float s, c;
  sincos_sfu(x, s, c);
  return (2.0f * s * fmaf(b, c, a) + theta2) * (1.0f / SPART_PI_F);
}

// sailh.py:401-446
__device__ __forceinline__ void volscatt_class_f(float sin_tts, float cos_tts, float sin_tto, float cos_tto,
                                                 float psi_rad, float sin_psi, float cos_psi, float sin_ttli,
                                                 float cos_ttli, float& chi_s, float& chi_o, float& frho,
                                                 float& ftau) {
  const float Cs = cos_ttli * cos_tts, Ss = sin_ttli * sin_tts;
  const float Co = cos_ttli * cos_tto, So = sin_ttli * sin_tto;
  const float As = fmaxf(Ss, Cs), Ao = fmaxf(So, Co);
  // flat leaf classes: C >= S in every lane of the warp -> beta = pi, sin beta = 0 (see volscatt_class)
  float cbs = -1.0f, cbo = -1.0f, bts = SPART_PI_F, bto = SPART_PI_F, sbs = 0.0f, sbo = 0.0f;
  const unsigned active = __activemask();
  if (!__all_sync(active, Cs >= Ss)) {
    cbs = -Cs / As;                               // exact: the quotient must be exactly -1 when As == Cs
    bts = acosf(cbs);
    sbs = fsqrt(fmaxf(0.0f, 1.0f - cbs * cbs));   // sin(acos z) = sqrt(1 - z^2)
  }
  if (!__all_sync(active, Co >= So)) {
    cbo = -Co / Ao;
    bto = acosf(cbo);
    sbo = fsqrt(fmaxf(0.0f, 1.0f - cbo * cbo));
  }
  chi_o = 2.0f / SPART_PI_F * ((bto - SPART_PI_F / 2.0f) * Co + sbo * So);
  chi_s = 2.0f / SPART_PI_F * ((bts - SPART_PI_F / 2.0f) * Cs + sbs * Ss);
  const float delta1 = fabsf(bts - bto);
  const float delta2 = SPART_PI_F - fabsf(bts + bto - SPART_PI_F);
  const float Tot = psi_rad + delta1 + delta2;
  const float bt1 = fminf(psi_rad, delta1);
  const float bt3 = fmaxf(psi_rad, delta2);
  const float bt2 = Tot - bt1 - bt3;
  const float T1 = 2.0f * Cs * Co + Ss * So * cos_psi;
  // (bt1, bt2, bt3) = (psi, delta1, delta2) sorted: sines / cosines by the addition theorems, see volscatt_class
  const float cc = cbs * cbo, ss = sbs * sbo, sc = sbs * cbo, cs = cbs * sbo;
  const bool lo = psi_rad <= delta1, hi = psi_rad > delta2;
  const float c1 = lo ? cos_psi : cc + ss;
  const float c3 = hi ? cos_psi : cc - ss;
  const float s2 = lo ? fabsf(sc - cs) : (hi ? fabsf(sc + cs) : sin_psi);
  const float T2 = s2 * (2.0f * As * Ao + Ss * So * c1 * c3);
  const float Jmin = bt2 * T1 - T2;
  const float Jplus = (SPART_PI_F - bt2) * T1 + T2;
  frho = fmaxf(0.0f, Jplus * (1.0f / (2.0f * SPART_PI_F * SPART_PI_F)));
  ftau = fmaxf(0.0f, -Jmin * (1.0f / (2.0f * SPART_PI_F * SPART_PI_F)));
}

// hot-spot integrals, see hotspot_integrals in spart_device.cuh (sailh.py:116-135, 216-219)
__device__ __forceinline__ void hotspot_integrals_f(float K, float k, float LAI, float q, float dso,
                                                    float& sumpso_ilai, float& pso2w) {
  const float A0 = (K + k) * LAI;
  const float S = fsqrt(K * k) * LAI;
  const float Amin = A0 - S;
  float A = A0, Cq = 0.0f, alpha = 0.0f;
  if (dso != 0.0f) {
    alpha = (dso * rcp(q)) * 2.0f * rcp(k + K);
    Cq = S * rcp(alpha);
  } else {
    A = Amin;
  }
  float L = 1.0f;
  if (alpha > 0.0f) L = fminf(L, 20.0f * rcp(alpha));     // e^-20 = 2e-9 is below float resolution of the integral
  if (Amin > 0.0f) L = fminf(L, 20.0f * rcp(Amin));
  // two graded panels, [-L/5, 0] and [-L, -L/5], of a 10-point Gauss-Legendre rule: relative error
  // <= 1e-8 on the benchmark distributions, see hotspot_integrals
  float total = 0.0f;
#pragma unroll 1
  for (int j = 0; j < 2; ++j) {
    const float hw = (j == 0 ? 0.1f : 0.4f) * L;
    const float xc = (j == 0 ? -0.1f : -0.6f) * L;
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      const float x = fmaf(hw, c_gl10_xf[i], xc);
      const float arg = fmaf(A, x, Cq * one_minus_exp(alpha * x));
      acc = fmaf(c_gl10_wf[i], fexp(arg), acc);
    }
    total = fmaf(hw, acc, total);
  }
  if (L < 1.0f && alpha * L >= 20.0f * (1.0f - 1e-6f)) {
    // e^{Cq - A L} (1 - e^{-A (1 - L)}) / A, finite for A -> 0 (bare soil): one_minus_exp switches to its series
    const float w = 1.0f - L, xr = A * w;
    const float f = (xr < 1e-3f) ? w * fmaf(xr, fmaf(xr, 1.0f / 6.0f, -0.5f), 1.0f) : one_minus_exp(-xr) * rcp(A);
    total += fexp(Cq - A * L) * f;
  }
  sumpso_ilai = total * LAI;
  const float dx = 1.0f / 60.0f;
  const float xc = -1.0f - 0.5f * dx;
  float acc = 0.0f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {      // the layer is 1/60 wide: 4 points resolve it to 1e-7
    const float x = fmaf(0.5f * dx, c_gl4_xf[i], xc);
    const float arg = fmaf(A, x, Cq * one_minus_exp(alpha * x));
    acc = fmaf(c_gl4_wf[i], fexp(arg), acc);
  }
  pso2w = 0.5f * acc;
}

struct AtmSampleF {
  float us, uv, m, Peq, lo3, lh2o, lm, lpeq, cksi, ksiD, ray_phase, taup550;
  float inv_us, inv_uv, inv_1pus, inv_1puv, aa3;
};

// smac.py:94-207 + SPART.py:235-252 at one band; c = the SM_* constants as float
__device__ __forceinline__ void smac_toa_band_f(const AtmSampleF& S, const float* c, float conv_ea, float etscale,
                                                float rv_so, float rv_do, float rv_dd, float rv_sd, float& R_TOC,
                                                float& R_TOA, float& L_TOA) {
  const float us = S.us, uv = S.uv, m = S.m, Peq = S.Peq, taup550 = S.taup550;
  const float inv_us = S.inv_us, inv_uv = S.inv_uv;
  const float taup = c[SM_A0TAUP] + c[SM_A1TAUP] * taup550;
  float gsum = 0.0f;
  if (c[SM_AO3] != 0.0f) gsum += c[SM_AO3] * fexp(c[SM_NO3] * S.lo3);
  if (c[SM_AH2O] != 0.0f) gsum += c[SM_AH2O] * fexp(c[SM_NH2O] * S.lh2o);
  if (c[SM_AO2] != 0.0f) gsum += c[SM_AO2] * fexp(fmaf(c[SM_NPO2], S.lpeq, c[SM_NO2] * S.lm));
  if (c[SM_ACO2] != 0.0f) gsum += c[SM_ACO2] * fexp(fmaf(c[SM_NPCO2], S.lpeq, c[SM_NCO2] * S.lm));
  if (c[SM_ACH4] != 0.0f) gsum += c[SM_ACH4] * fexp(fmaf(c[SM_NPCH4], S.lpeq, c[SM_NCH4] * S.lm));
  if (c[SM_ANO2] != 0.0f) gsum += c[SM_ANO2] * fexp(fmaf(c[SM_NPNO2], S.lpeq, c[SM_NNO2] * S.lm));
  if (c[SM_ACO] != 0.0f) gsum += c[SM_ACO] * fexp(fmaf(c[SM_NPCO], S.lpeq, c[SM_NCO] * S.lm));
  const float tg = fexp(gsum);
  const float s = c[SM_A0S] * Peq + c[SM_A3S] + c[SM_A1S] * taup550 + c[SM_A2S] * taup550 * taup550;
  const float tnum = c[SM_A2T] * Peq + c[SM_A3T];
  const float ttetas = c[SM_A0T] + c[SM_A1T] * taup550 * inv_us + tnum * S.inv_1pus;
  const float ttetav = c[SM_A0T] + c[SM_A1T] * taup550 * inv_uv + tnum * S.inv_1puv;
  const float cksi = S.cksi, ksiD = S.ksiD;
  const float taur = c[SM_TAUR];
  const float inv_usuv = inv_us * inv_uv;
  const float rr = taur * S.ray_phase * inv_usuv;
  const float ray_ref = 0.25f * rr * Peq;
  const float taurz = taur * Peq;
  const float ksi2 = ksiD * ksiD;
  const float aer_phase = c[SM_A0P] + c[SM_A1P] * ksiD + c[SM_A2P] * ksi2 + c[SM_A3P] * (ksi2 * ksiD) +
                          c[SM_A4P] * (ksi2 * ksi2);
  const float wo = c[SM_WO], ak2 = c[SM_AK2], ak = c[SM_AK];
  const float opb = c[SM_OPB], omb = c[SM_OMB], g3 = c[SM_G3], h3 = c[SM_H3], akd3 = c[SM_AKD3];
  const float us2 = us * us;
  const float inv_q = rcp(1.0f - ak2 * us2);
  const float e = -0.75f * us2 * wo * inv_q;
  const float f = -0.25f * h3 * us2 * wo * inv_q;
  const float dp = e * inv_us * (1.0f / 3.0f) + us * f;
  const float d = e + f;
  const float eak = fexp(ak * taup);
  const float emak = rcp(eak);
  const float inv_delta = rcp(eak * c[SM_OPB2] - emak * c[SM_OMB2]);
  const float ss = us * inv_q;
  const float q1 = 2.0f + 3.0f * us + h3 * us * (1.0f + 2.0f * us);
  const float q2 = 2.0f - 3.0f * us - h3 * us * (1.0f - 2.0f * us);
  const float Eu = fexp(-taup * inv_us), Ev = fexp(-taup * inv_uv);
  const float q3 = q2 * Eu;
  const float wsd = c[SM_WW] * ss * inv_delta;
  const float c1 = wsd * (q1 * eak * opb + q3 * omb);
  const float c2 = -wsd * (q1 * emak * omb + q3 * opb);
  const float cp1 = c1 * akd3;
  const float cp2 = -c2 * akd3;
  const float g3uv = g3 * uv;
  const float z = d - g3uv * dp + wo * aer_phase * 0.25f;
  const float x = c1 - g3uv * cp1;
  const float y = c2 - g3uv * cp2;
  const float aa1 = uv * rcp(1.0f + ak * uv);
  const float aa2 = uv * rcp(1.0f - ak * uv);
  const float aer_ref1 = x * aa1 * (1.0f - Ev * emak);
  const float aer_ref2 = y * aa2 * (1.0f - Ev * eak);
  const float aer_ref3 = z * S.aa3 * (1.0f - Ev * Eu);
  const float aer_ref = (aer_ref1 + aer_ref2 + aer_ref3) * inv_usuv;
  const float Res_ray = c[SM_RESR1] + c[SM_RESR2TAUR] * S.ray_phase * inv_usuv + c[SM_RESR3] * (rr * rr);
  const float ta = taup * m * cksi;
  const float Res_aer = (c[SM_RESA1] + c[SM_RESA2] * ta + c[SM_RESA3] * (ta * ta)) + c[SM_RESA4] * (ta * ta * ta);
  const float tautot = taup + taurz;
  const float tt = tautot * m * cksi;
  const float Res_6s = (c[SM_REST1] + c[SM_REST2] * tt + c[SM_REST3] * (tt * tt)) + c[SM_REST4] * (tt * tt * tt);
  const float atm_ref = ray_ref - Res_ray + aer_ref - Res_aer + Res_6s;
  const float ta_ss = fexp(-tautot * inv_us);
  const float ta_oo = fexp(-tautot * inv_uv);
  const float ta_sd = ttetas - ta_ss;
  const float ta_do = ttetav - ta_oo;
  const float ra_dd = s, ra_so = atm_ref;
  const float inv_ms = rcp(1.0f - rv_dd * ra_dd);
  const float rtoa0 = ra_so + ta_ss * rv_so * ta_oo;
  const float rtoa1 = (ta_sd * rv_do + ta_ss * rv_sd * ra_dd * rv_do) * ta_oo * inv_ms;
  const float rtoa2 = (ta_ss * rv_sd + ta_sd * rv_dd) * ta_do * inv_ms;
  R_TOC = (ta_ss * rv_so + ta_sd * rv_do) * rcp(ta_ss + ta_sd);
  R_TOA = tg * (rtoa0 + rtoa1 + rtoa2);
  L_TOA = (conv_ea * etscale) * R_TOA;
}

}  // namespace f32
}  // namespace spart
