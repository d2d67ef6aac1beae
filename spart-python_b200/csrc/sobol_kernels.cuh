// sobol_kernels.cuh -- variance-based sensitivity analysis on the device: a scrambled Sobol' design written in the
// batch layout, and the Saltelli (2010) estimators of the first-order and total indices over its outputs.
//
// Design: point i of dimension d is k_d(i) = XOR of v'[d][j] over the set bits j of gray(i) = i ^ (i >> 1), XOR
// s_d, and u = k_d(i) * 2^-32 (direction numbers v of sobol_dirs.h; v' = L_d v and s_d come from the host, see
// spart_sobol_design in spart_b200.h).  Every point is evaluated from its index alone, so any index range can be
// produced and shards need no state.
//   thread = one base point j, block = 256 base points x one varied parameter p (blockIdx.y)
//   Saltelli layout: blocks A, B, AB_1 .. AB_d of `count` samples each; the thread writes parameter p of its base
//   point in every block (AB_i takes p from B when i == p, from A otherwise).
//
// Estimators (scipy.stats.sobol_indices, method "saltelli_2010", which centres the outputs on their mean): per
// output o and varied parameter i, over base points j (f_X = output of block X at j)
//   t = (f_B - mean) (f_ABi - f_A),  u = (f_A - f_ABi)^2,  V = population variance of f_A and f_B together,
//   S_i = mean(t) / V,  ST_i = mean(u) / (2 V).
// Sums are taken of values shifted by their value at base point 0 of the whole design (ref), so that an output
// whose mean is far above its spread keeps its variance, and so that the accumulator is a plain sum that shards
// merge by adding.
//   block = one slice of the chunk's base points x one varied parameter (blockIdx.x; x = d: the f sums);
//   thread (r, o): output o, base points j = r, r + R, ... of the slice, so a warp reads consecutive addresses;
//   the R partial sums of each output are added in r order, and the slice's total is added to its own slot of
//   the accumulator: every sum has a fixed order, so a run is bit-reproducible.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sobol_dirs.h"

namespace spart {

constexpr int kSobolMaxVary = 27;             // = SPART_NPAR
constexpr int kSobolThreads = 256;
constexpr int kSobolSlices = 128;             // accumulator slots per (parameter, output)

// Everything the design kernel needs, passed by value (kernel parameter space, ~8.9 KB): a per-call constant
// upload would race between host threads with different seeds.
struct SobolDesignArgs {
  unsigned v[2 * kSobolMaxVary][32];           // scrambled direction numbers v' of the dimensions used
  unsigned shift[2 * kSobolMaxVary];           // digital shift s_d
  double lo[kSobolMaxVary], hi[kSobolMaxVary];
  int row[kSobolMaxVary];
};

__device__ __forceinline__ unsigned sobol_point(const unsigned (&v)[32], unsigned shift, unsigned i) {
  const unsigned g = i ^ (i >> 1);
  unsigned k = shift;
#pragma unroll
  for (int j = 0; j < 32; ++j) k ^= v[j] & (0u - ((g >> j) & 1u));
  return k;
}

// x = lo + (hi - lo) u without FMA contraction (NumPy reproduces it bit for bit); a value rounded up to hi is
// moved to the double below it, so x is in [lo, hi)
__device__ __forceinline__ double sobol_value(unsigned k, double lo, double hi) {
  const double x = __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), (double)k * 0x1p-32));
  return x < hi ? x : nextafter(hi, lo);
}

__global__ void __launch_bounds__(kSobolThreads)
sobol_design_kernel(const SobolDesignArgs a, int n_vary, int64_t first, int64_t count, int saltelli,
                    double* __restrict__ params, int64_t ld) {
  const int64_t j = (int64_t)blockIdx.x * kSobolThreads + threadIdx.x;
  if (j >= count) return;
  const int p = blockIdx.y;
  const unsigned i = (unsigned)(first + j);
  double* out = params + (int64_t)a.row[p] * ld + j;
  const double xa = sobol_value(sobol_point(a.v[p], a.shift[p], i), a.lo[p], a.hi[p]);
  out[0] = xa;
  if (!saltelli) return;
  const double xb = sobol_value(sobol_point(a.v[n_vary + p], a.shift[n_vary + p], i), a.lo[p], a.hi[p]);
  out[count] = xb;
  for (int b = 0; b < n_vary; ++b) out[(2 + b) * count] = (b == p) ? xb : xa;
}

constexpr int kSobolSums = 8;                 // doubles per accumulator slot

// acc layout: [kSobolSlices][n_vary + 1][n_out][kSobolSums] doubles.  With a = f_B - f_ref, D = f_ABi - f_A,
// p = a D and u = D^2, slot (s, i < n_vary, o) holds the sums of (p - p_ref), (p - p_ref)^2, (D - D_ref),
// (D - D_ref)^2, (p - p_ref)(D - D_ref), (u - u_ref), (u - u_ref)^2 and a zero; slot (s, n_vary, o) holds those of
// (f - f_ref) and (f - f_ref)^2 over f_A and f_B, then zeros.  (f_B - mean) D = p - (mean - f_ref) D is then
// formed in the finish, once the mean is known.
__global__ void __launch_bounds__(kSobolThreads)
sobol_accumulate_kernel(const double* __restrict__ f, int64_t n, int n_out, int n_vary, const double* __restrict__ ref,
                        double* __restrict__ acc) {
  __shared__ double part[kSobolThreads][kSobolSums - 1];
  const int i = blockIdx.x, s = blockIdx.y;
  const int cols = n_out < kSobolThreads ? n_out : kSobolThreads;
  const int R = kSobolThreads / cols;
  const int r = threadIdx.x / cols, oc = threadIdx.x % cols;
  const int64_t j0 = n * s / kSobolSlices, j1 = n * (s + 1) / kSobolSlices;
  for (int o0 = 0; o0 < n_out; o0 += cols) {
    const int o = o0 + oc;
    double z[kSobolSums - 1] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (r < R && o < n_out) {
      const double* fa = f + o;
      const double* fb = f + n * n_out + o;
      const double ra = ref[o];
      if (i == n_vary) {
#pragma unroll 4
        for (int64_t j = j0 + r; j < j1; j += R) {
          const double da = fa[j * n_out] - ra, db = fb[j * n_out] - ra;
          z[0] += da;
          z[1] = fma(da, da, z[1]);
          z[0] += db;
          z[1] = fma(db, db, z[1]);
        }
      } else {
        const double* fab = f + (2 + i) * n * n_out + o;
        const double qr = ref[(2 + i) * n_out + o] - ra;
        const double pr = __dmul_rn(ref[n_out + o] - ra, qr), ur = __dmul_rn(qr, qr);
#pragma unroll 4
        for (int64_t j = j0 + r; j < j1; j += R) {
          const double xa = fa[j * n_out], D = fab[j * n_out] - xa;
          const double dp = __dsub_rn(__dmul_rn(fb[j * n_out] - ra, D), pr);
          const double dq = D - qr;
          const double du = __dsub_rn(__dmul_rn(D, D), ur);
          z[0] += dp;
          z[1] = fma(dp, dp, z[1]);
          z[2] += dq;
          z[3] = fma(dq, dq, z[3]);
          z[4] = fma(dp, dq, z[4]);
          z[5] += du;
          z[6] = fma(du, du, z[6]);
        }
      }
    }
#pragma unroll
    for (int c = 0; c < kSobolSums - 1; ++c) part[threadIdx.x][c] = z[c];
    __syncthreads();
    if (r == 0 && o < n_out) {
      double t[kSobolSums - 1] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      for (int q = 0; q < R; ++q)
#pragma unroll
        for (int c = 0; c < kSobolSums - 1; ++c) t[c] += part[q * cols + oc][c];
      double* dst = acc + (((int64_t)s * (n_vary + 1) + i) * n_out + o) * kSobolSums;
#pragma unroll
      for (int c = 0; c < kSobolSums - 1; ++c) dst[c] += t[c];
    }
    __syncthreads();
  }
}

// thread = (output o, varied parameter i); i == 0 also writes mean and var of output o.  As in
// scipy.stats.sobol_indices, f_B is centred on the mean of f_A and f_B: t = (f_B - mean) D = p - m D with
// m = mean - f_ref, so mean(t) = mean(p) - m mean(D) and var(t) = var(p) - 2 m cov(p, D) + m^2 var(D).
__global__ void sobol_finish_kernel(const double* __restrict__ acc, const double* __restrict__ ref, int64_t n_total,
                                    int n_out, int n_vary, double* __restrict__ mean, double* __restrict__ var,
                                    double* __restrict__ first, double* __restrict__ total,
                                    double* __restrict__ first_se, double* __restrict__ total_se) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n_out * n_vary) return;
  const int o = (int)(idx / n_vary), i = (int)(idx % n_vary);
  double sf = 0.0, sff = 0.0, z[kSobolSums - 1] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int s = 0; s < kSobolSlices; ++s) {
    const double* a = acc + (((int64_t)s * (n_vary + 1) + n_vary) * n_out + o) * kSobolSums;
    const double* b = acc + (((int64_t)s * (n_vary + 1) + i) * n_out + o) * kSobolSums;
    sf += a[0];
    sff += a[1];
#pragma unroll
    for (int c = 0; c < kSobolSums - 1; ++c) z[c] += b[c];
  }
  const double N = (double)n_total, ra = ref[o];
  const double m = sf / (2.0 * N);
  const double V = fmax(sff / (2.0 * N) - m * m, 0.0);
  const double qr = ref[(2 + i) * n_out + o] - ra;
  const double pr = __dmul_rn(ref[n_out + o] - ra, qr), ur = __dmul_rn(qr, qr);
  const double mp = z[0] / N, mq = z[2] / N, mu = z[5] / N;
  const double vp = z[1] / N - mp * mp, vq = z[3] / N - mq * mq, cpq = z[4] / N - mp * mq;
  const double vt = fmax(vp - 2.0 * m * cpq + m * m * vq, 0.0), vu = fmax(z[6] / N - mu * mu, 0.0);
  const double mt = (pr + mp) - m * (qr + mq);
  const double sq = sqrt(N);
  first[(int64_t)o * n_vary + i] = mt / V;
  total[(int64_t)o * n_vary + i] = (ur + mu) / (2.0 * V);
  first_se[(int64_t)o * n_vary + i] = sqrt(vt) / (sq * V);
  total_se[(int64_t)o * n_vary + i] = sqrt(vu) / (2.0 * sq * V);
  if (i == 0) {
    mean[o] = ra + m;
    var[o] = V;
  }
}

}  // namespace spart
