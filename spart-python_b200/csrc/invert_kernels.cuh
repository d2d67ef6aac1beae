// invert_kernels.cuh -- per-observation retrieval by bounded Levenberg-Marquardt: the design of one iteration's
// forward batch, the per-track step, and the pick of the best start per observation with its covariance.
//
// A track is one start of one observation (track t belongs to observation t / n_starts), iterated in normalised
// coordinates u in [0, 1]^P with x = lo + (hi - lo) u (each operation rounded once, no FMA).  Its state is a
// column of the [inv_rows(P)][n_tracks] state array (layout below).  One iteration = design -> forward -> step:
//   design: for each active track, P + 1 samples: sample 0 at the trial point, sample p + 1 with u_p moved by
//     h = 2^-17 (up if u_p + h <= 1, else down);
//   step: C(trial) = sum_b w_b (f_b - y_b)^2 in band order; accept if C(trial) < C (strict), then take the
//     trial's J^T W J and J^T W r (J column p = (f_{p+1} - f_0) / du_p, du_p the difference of the two written x
//     over hi - lo, so J is d f / d u); lambda / 10 (>= 1e-15) on acceptance, x 10 on rejection; then solve
//     (J^T W J + lambda D) delta = -J^T W r, D = diag(max(J^T W J_pp, 1e-30)), by Cholesky, lambda x 10 and
//     again while the factorisation fails; next trial = clip(u + delta, 0, 1).
// The step's Cholesky factor lives in a shared-memory column per thread (element k of thread i at
// smem[k * kInvThreads + i]), so no per-thread array is indexed at run time and nothing goes to local memory.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spart {

constexpr int kInvMaxVary = 16;
constexpr int kInvThreads = 32;              // step / finish: 32 columns of <= 184 doubles = 47 KB of shared memory
constexpr double kInvStep = 0x1p-17;
constexpr double kInvLambdaMin = 1e-15, kInvLambdaMax = 1e16, kInvDiagFloor = 1e-30;

// status codes (spart_b200.h SPART_INV_*)
constexpr int kInvActive = 0, kInvConvergedCost = 1, kInvConvergedStep = 2, kInvMaxIter = 3, kInvStalled = 4,
              kInvInvalid = 5;

// state rows of a track with P varied parameters: u [P], trial [P], J^T W J [P (P + 1) / 2] (lower triangle,
// row-major: (i, j <= i) at i (i + 1) / 2 + j), J^T W r [P], C, lambda, status, forward calls
__host__ __device__ constexpr int inv_tri(int P) { return P * (P + 1) / 2; }
__host__ __device__ constexpr int inv_rows(int P) { return 3 * P + inv_tri(P) + 4; }
__host__ __device__ constexpr int inv_shared(int P) { return inv_tri(P) + 3 * P; }

struct InvertArgs {
  double lo[kInvMaxVary], hi[kInvMaxVary];
  double base[27];                           // values of the broadcast rows, written at element 0
  int row[kInvMaxVary];
  int obs_row[27];                           // rows given per observation
  int bcast_row[27];                         // rows written at element 0 only
  int n_vary, n_obs_rows, n_bcast, n_starts;
};

__device__ __forceinline__ double inv_x(double lo, double hi, double u) {
  return __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u));
}

// u_p of sample p + 1 of a trial u_p
__device__ __forceinline__ double inv_moved(double u) {
  return __dadd_rn(u, kInvStep) <= 1.0 ? __dadd_rn(u, kInvStep) : __dsub_rn(u, kInvStep);
}

// thread = one sample (active slot a, sample s) of the batch [27][ld], column a (P + 1) + s
__global__ void __launch_bounds__(256)
invert_design_kernel(const InvertArgs a, const double* __restrict__ obs_values, int64_t ld_values,
                     const double* __restrict__ state, int64_t n_tracks, const int32_t* __restrict__ active,
                     int64_t n_active, double* __restrict__ params, int64_t ld) {
  const int P = a.n_vary;
  // n_tracks (P + 1) < 2^31 (checked by the caller): 32-bit index arithmetic, no 64-bit division
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= n_active * (P + 1)) return;
  const int slot = col / (P + 1), s = col - slot * (P + 1);
  const int t = active[slot];
  const double* trial = state + (int64_t)P * n_tracks + t;
  for (int p = 0; p < P; ++p) {
    const double u = trial[(int64_t)p * n_tracks];
    params[(int64_t)a.row[p] * ld + col] = inv_x(a.lo[p], a.hi[p], s == p + 1 ? inv_moved(u) : u);
  }
  const int o = t / a.n_starts;
  for (int k = 0; k < a.n_obs_rows; ++k) params[(int64_t)a.obs_row[k] * ld + col] = obs_values[k * ld_values + o];
  if (col == 0)
    for (int k = 0; k < a.n_bcast; ++k) params[(int64_t)a.bcast_row[k] * ld] = a.base[a.bcast_row[k]];
}

// Cholesky of M = A + lambda diag(max(A_pp, 1e-30)) (lambda = 0: of A itself) into the shared column L (packed
// lower triangle); A is read from the state column.  Returns false where a pivot is not > 0 (or is NaN).
__device__ __forceinline__ bool inv_cholesky(const double* A, int64_t ld, int P, double lambda, double* L) {
  for (int j = 0; j < P; ++j) {
    const int jj = inv_tri(j);
    const double ajj = A[(int64_t)(jj + j) * ld];
    double s = lambda > 0.0 ? ajj + lambda * fmax(ajj, kInvDiagFloor) : ajj;
    for (int k = 0; k < j; ++k) s -= L[(jj + k) * kInvThreads] * L[(jj + k) * kInvThreads];
    if (!(s > 0.0)) return false;
    const double d = sqrt(s);
    L[(jj + j) * kInvThreads] = d;
    for (int i = j + 1; i < P; ++i) {
      const int ii = inv_tri(i);
      double v = A[(int64_t)(ii + j) * ld];
      for (int k = 0; k < j; ++k) v -= L[(ii + k) * kInvThreads] * L[(jj + k) * kInvThreads];
      L[(ii + j) * kInvThreads] = v / d;
    }
  }
  return true;
}

// thread = one active track; dynamic shared memory kInvThreads * inv_shared(P) doubles
__global__ void __launch_bounds__(kInvThreads)
invert_step_kernel(const InvertArgs a, const double* __restrict__ f, int n_bands, int column,
                   const double* __restrict__ obs, const double* __restrict__ weights, double ftol, double xtol,
                   int max_iter, double* __restrict__ state, int64_t n_tracks, const int32_t* __restrict__ active,
                   int64_t n_active) {
  extern __shared__ double inv_smem[];
  const int64_t slot = (int64_t)blockIdx.x * kInvThreads + threadIdx.x;
  if (slot >= n_active) return;
  const int P = a.n_vary, NA = inv_tri(P);
  const int64_t ld = n_tracks, t = active[slot];
  double* u = state + t;
  double* trial = u + P * ld;
  double* A = trial + P * ld;
  double* g = A + NA * ld;
  double* st = g + P * ld;                   // C, lambda, status, forward calls
  double* L = inv_smem + threadIdx.x;        // [NA] factor / J^T W J being summed
  double* gs = L + NA * kInvThreads;         // [P] J^T W r being summed
  double* J = gs + P * kInvThreads;          // [P] one band's Jacobian row
  double* z = J + P * kInvThreads;           // [P] du, then the solve's vector
  const double* y = obs + (int64_t)((int)t / a.n_starts) * n_bands;
  const int64_t row0 = slot * (P + 1);       // sample 0 of this track in the batch
  const double* f0 = f + row0 * n_bands * 3 + column;

  const int calls = (int)st[3 * ld] + 1;
  st[3 * ld] = (double)calls;
  double c = 0.0;
  bool finite_y = true;
  for (int b = 0; b < n_bands; ++b) {
    const double w = weights ? weights[b] : 1.0;
    const double d = __dsub_rn(f0[b * 3], y[b]);
    c = __dadd_rn(c, __dmul_rn(w, __dmul_rn(d, d)));
    finite_y = finite_y && isfinite(y[b]);
  }
  const bool first = calls == 1;
  if (first && !(finite_y && isfinite(c))) {
    st[2 * ld] = kInvInvalid;
    return;
  }
  const double c_old = st[0];
  double lambda = st[ld];
  if (first || c < c_old) {
    for (int p = 0; p < P; ++p) {
      const double up = trial[p * ld];
      u[p * ld] = up;
      z[p * kInvThreads] = __dsub_rn(inv_x(a.lo[p], a.hi[p], inv_moved(up)), inv_x(a.lo[p], a.hi[p], up)) /
                           __dsub_rn(a.hi[p], a.lo[p]);
      gs[p * kInvThreads] = 0.0;
    }
    for (int k = 0; k < NA; ++k) L[k * kInvThreads] = 0.0;
    for (int b = 0; b < n_bands; ++b) {
      const double w = weights ? weights[b] : 1.0;
      const double fb = f0[b * 3];
      const double d = fb - y[b];
      for (int p = 0; p < P; ++p) J[p * kInvThreads] = (f0[((p + 1) * n_bands + b) * 3] - fb) / z[p * kInvThreads];
      for (int i = 0; i < P; ++i) {
        const double wj = w * J[i * kInvThreads];
        gs[i * kInvThreads] += wj * d;
        for (int j = 0; j <= i; ++j) L[(inv_tri(i) + j) * kInvThreads] += wj * J[j * kInvThreads];
      }
    }
    for (int k = 0; k < NA; ++k) A[k * ld] = L[k * kInvThreads];
    for (int p = 0; p < P; ++p) g[p * ld] = gs[p * kInvThreads];
    st[0] = c;
    if (!first) {
      lambda = fmax(lambda / 10.0, kInvLambdaMin);
      if (c_old - c <= ftol * c_old) {
        st[ld] = lambda;
        st[2 * ld] = kInvConvergedCost;
        return;
      }
    }
  } else {
    lambda *= 10.0;
  }
  int status = kInvActive;
  if (lambda > kInvLambdaMax) status = kInvStalled;
  else if (calls >= max_iter) status = kInvMaxIter;
  while (status == kInvActive && !inv_cholesky(A, ld, P, lambda, L)) {
    lambda *= 10.0;
    if (lambda > kInvLambdaMax) status = kInvStalled;
  }
  st[ld] = lambda;
  if (status != kInvActive) {
    st[2 * ld] = status;
    return;
  }
  // L y = -g, then L^T delta = y (z holds y, then delta)
  for (int i = 0; i < P; ++i) {
    const int ii = inv_tri(i);
    double v = -g[i * ld];
    for (int k = 0; k < i; ++k) v -= L[(ii + k) * kInvThreads] * z[k * kInvThreads];
    z[i * kInvThreads] = v / L[(ii + i) * kInvThreads];
  }
  for (int i = P - 1; i >= 0; --i) {
    double v = z[i * kInvThreads];
    for (int k = i + 1; k < P; ++k) v -= L[(inv_tri(k) + i) * kInvThreads] * z[k * kInvThreads];
    z[i * kInvThreads] = v / L[(inv_tri(i) + i) * kInvThreads];
  }
  double step = 0.0;
  for (int p = 0; p < P; ++p) {
    const double up = u[p * ld];
    const double next = fmin(fmax(up + z[p * kInvThreads], 0.0), 1.0);
    trial[p * ld] = next;
    step = fmax(step, fabs(next - up));
  }
  if (step <= xtol) st[2 * ld] = kInvConvergedStep;
}

// thread = one observation: the track with the lowest finite cost (ties to the lowest start), its x, cost,
// status, start and forward calls, the forward runs of all its tracks, and std_p = (hi_p - lo_p)
// sqrt(scale (A^-1)_pp) from the Cholesky factor of its J^T W J (scale = C / (n_bands - P), or 1 with
// absolute_sigma); NaN where J^T W J is not positive definite or, scaled, where n_bands <= P.
__global__ void __launch_bounds__(kInvThreads)
invert_finish_kernel(const InvertArgs a, int n_bands, int absolute_sigma, const double* __restrict__ state,
                     int64_t n_obs, double* __restrict__ x, double* __restrict__ cost, double* __restrict__ sd,
                     int32_t* __restrict__ status, int32_t* __restrict__ start, int32_t* __restrict__ iterations,
                     int64_t* __restrict__ n_forward) {
  extern __shared__ double inv_smem[];
  const int64_t o = (int64_t)blockIdx.x * kInvThreads + threadIdx.x;
  if (o >= n_obs) return;
  const int P = a.n_vary, NA = inv_tri(P), S = a.n_starts;
  const int64_t ld = n_obs * S;
  const double* C = state + (int64_t)(3 * P + NA) * ld;
  int best = -1;
  int64_t runs = 0;
  for (int s = 0; s < S; ++s) {
    const int64_t t = o * S + s;
    runs += (int64_t)C[3 * ld + t] * (P + 1);
    if (isfinite(C[t]) && (best < 0 || C[t] < C[o * S + best])) best = s;
  }
  n_forward[o] = runs;
  if (best < 0) {
    for (int p = 0; p < P; ++p) x[o * P + p] = sd[o * P + p] = nan("");
    cost[o] = nan("");
    status[o] = kInvInvalid;
    start[o] = -1;
    iterations[o] = 0;
    return;
  }
  const int64_t t = o * S + best;
  const double c = C[t];
  for (int p = 0; p < P; ++p) x[o * P + p] = inv_x(a.lo[p], a.hi[p], state[p * ld + t]);
  cost[o] = c;
  status[o] = (int32_t)C[2 * ld + t];
  start[o] = best;
  iterations[o] = (int32_t)C[3 * ld + t];
  double* L = inv_smem + threadIdx.x;
  double* z = L + NA * kInvThreads;
  const double scale = absolute_sigma ? 1.0 : (n_bands > P ? c / (double)(n_bands - P) : nan(""));
  const bool pd = inv_cholesky(state + (int64_t)2 * P * ld + t, ld, P, 0.0, L);
  for (int p = 0; p < P; ++p) {
    double var = nan("");
    if (pd) {
      // column p of L^-1: z_p = 1 / L_pp, z_i = -(sum_{k=p}^{i-1} L_ik z_k) / L_ii; (A^-1)_pp = sum_i z_i^2
      var = 0.0;
      for (int i = p; i < P; ++i) {
        double v = i == p ? 1.0 : 0.0;
        for (int k = p; k < i; ++k) v -= L[(inv_tri(i) + k) * kInvThreads] * z[k * kInvThreads];
        const double zi = v / L[(inv_tri(i) + i) * kInvThreads];
        z[i * kInvThreads] = zi;
        var += zi * zi;
      }
    }
    sd[o * P + p] = __dsub_rn(a.hi[p], a.lo[p]) * sqrt(scale * var);
  }
}

}  // namespace spart
