// Test harness for the device math functions of spart_device.cuh / spart_device_f32.cuh, compiled at test time
// into a shared library (tests/test_gpu_device_math.py) and called through ctypes on device pointers.
// The plate-transmissivity tables are uploaded the way spart_create does.
#include <stdint.h>

#include "spart_device_f32.cuh"

using namespace spart;

enum Fn64 { F_EXP_FAST = 0, F_EXP_CLAMP, F_EXP_NEG, F_EXP_BOUNDED, F_LOG, F_RCP, F_SQRT, F_SIN, F_COS, F_PLATE_TAU };
enum Fn32 { G_ONE_MINUS_TAU = 0, G_EXP, G_LOG, G_RCP, G_SQRT, G_TAU };

__global__ void eval64(int fn, const double* __restrict__ x, double* __restrict__ y, int64_t n) {
  __shared__ TauTable s_tau;
  load_tau_table(&s_tau);
  exp_table_load();
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double v = x[i] * 1.0;    // an arithmetic result, as at every call site (canonical NaN)
  double r = 0.0, c;
  switch (fn) {
    case F_EXP_FAST: r = exp_fast(v); break;
    case F_EXP_CLAMP: r = exp_clamp(v); break;
    case F_EXP_NEG: r = exp_neg(v); break;
    case F_EXP_BOUNDED: r = exp_bounded(v); break;
    case F_LOG: r = log_fast(v); break;
    case F_RCP: r = rcp_fast(v); break;
    case F_SQRT: r = sqrt_fast(v); break;
    case F_SIN: sincos_small(v, r, c); break;
    case F_COS: sincos_small(v, c, r); break;
    case F_PLATE_TAU: r = plate_tau(v, &s_tau); break;
  }
  y[i] = r;
}

__global__ void eval32(int fn, const float* __restrict__ x, float* __restrict__ y, int64_t n) {
  __shared__ f32::TauTableF s_tau;
  f32::load_tau_table_f(&s_tau);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = x[i];
  float r = 0.0f, omt = 0.0f;
  switch (fn) {
    case G_ONE_MINUS_TAU: f32::plate_tau_f(v, &s_tau, omt); r = omt; break;
    case G_TAU: r = f32::plate_tau_f(v, &s_tau, omt); break;
    case G_EXP: r = f32::fexp(v); break;
    case G_LOG: r = f32::flog(v); break;
    case G_RCP: r = f32::rcp(v); break;
    case G_SQRT: r = f32::fsqrt(v); break;
  }
  y[i] = r;
}

extern "C" {

// 0 on success, else the CUDA error code
int dm_init() {
  cudaError_t e = cudaMemcpyToSymbol(c_tau_coef, SPART_TAU_COEF_H, sizeof(SPART_TAU_COEF_H));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_tau_mid, SPART_TAU_MID_H, sizeof(SPART_TAU_MID_H));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_tau_invhalf, SPART_TAU_INVHALF_H, sizeof(SPART_TAU_INVHALF_H));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(f32::c_tauf_coef, SPART_TAUF_COEF_H, sizeof(SPART_TAUF_COEF_H));
  return (int)e;
}

int dm_eval64(int fn, const double* x, double* y, int64_t n) {
  if (n > 0) eval64<<<(unsigned)((n + 255) / 256), 256>>>(fn, x, y, n);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  return (int)e;
}

int dm_eval32(int fn, const float* x, float* y, int64_t n) {
  if (n > 0) eval32<<<(unsigned)((n + 255) / 256), 256>>>(fn, x, y, n);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  return (int)e;
}

}  // extern "C"
