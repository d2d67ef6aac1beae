// lut_kernels.cuh -- nearest look-up-table entry (the consumer of a SPART LUT, SURVEY.md 8(f)2).
//
// For every observed band vector o (m of them) find the LUT entry l (n of them, produced by
// spart_forward_bands) that minimises the weighted squared distance sum_b w_b (o_b - l_b)^2.
// Arithmetic is FP32 SIMT: with 6..26 bands the contraction dimension is far too short to feed
// tensor cores, and the expanded form |o|^2 + |l|^2 - 2 o.l would cancel catastrophically in
// low precision for the near-identical spectra a retrieval compares.
//   thread  = one observation (its scaled band values live in registers)
//   block   = kLutObs observations x one slice of the LUT (blockIdx.y), walked in shared-memory
//             tiles of kLutTile entries; every lane reads the same LUT value (broadcast LDS.128)
//   result  = atomicMin on a packed (cost bits << 32 | index) word per observation, so ties go to
//             the lowest index and the result is deterministic
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spart {

constexpr int kLutObs = 256;
constexpr int kLutTile = 128;

template <int NB4>   // bands padded to 4 * NB4
__global__ void __launch_bounds__(kLutObs)
lut_nearest_kernel(const float* __restrict__ lut, int64_t n, int nb, const float* __restrict__ obs, int64_t m,
                   const float* __restrict__ sqrt_w, int64_t per_slice, unsigned index_offset,
                   unsigned long long* __restrict__ best) {
  constexpr int NBP = 4 * NB4;
  __shared__ __align__(16) float s_l[kLutTile][NBP];
  __shared__ float s_w[NBP];
  for (int b = threadIdx.x; b < NBP; b += blockDim.x) s_w[b] = (b < nb) ? (sqrt_w ? sqrt_w[b] : 1.0f) : 0.0f;
  __syncthreads();
  const int64_t oi = (int64_t)blockIdx.x * kLutObs + threadIdx.x;
  const int64_t oc = oi < m ? oi : m - 1;
  float o[NBP];
#pragma unroll
  for (int b = 0; b < NBP; ++b) o[b] = (b < nb) ? obs[oc * nb + b] * s_w[b] : 0.0f;
  const int64_t e0 = (int64_t)blockIdx.y * per_slice;
  const int64_t e1 = (e0 + per_slice < n) ? e0 + per_slice : n;
  float best_cost = 3.0e38f;
  unsigned best_idx = 0xffffffffu;
  for (int64_t t0 = e0; t0 < e1; t0 += kLutTile) {
    const int cnt = (int)((e1 - t0 < kLutTile) ? (e1 - t0) : kLutTile);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * NBP; i += blockDim.x) {
      const int e = i / NBP, b = i % NBP;
      s_l[e][b] = (b < nb) ? lut[(t0 + e) * nb + b] * s_w[b] : 0.0f;
    }
    __syncthreads();
#pragma unroll 2
    for (int e = 0; e < cnt; ++e) {
      const float4* row = reinterpret_cast<const float4*>(s_l[e]);
      float c0 = 0.0f, c1 = 0.0f;
#pragma unroll
      for (int q = 0; q < NB4; ++q) {
        const float4 l = row[q];
        const float d0 = o[4 * q] - l.x, d1 = o[4 * q + 1] - l.y, d2 = o[4 * q + 2] - l.z, d3 = o[4 * q + 3] - l.w;
        c0 = fmaf(d0, d0, c0);
        c1 = fmaf(d1, d1, c1);
        c0 = fmaf(d2, d2, c0);
        c1 = fmaf(d3, d3, c1);
      }
      const float c = c0 + c1;
      if (c < best_cost) {
        best_cost = c;
        best_idx = (unsigned)(t0 + e);
      }
    }
  }
  if (oi < m && best_idx != 0xffffffffu) {
    // index_offset: position of this LUT (shard) inside a larger table split over several GPUs
    const unsigned long long packed = ((unsigned long long)__float_as_uint(best_cost) << 32) | (best_idx + index_offset);
    atomicMin(&best[oi], packed);
  }
}

__global__ void lut_unpack_kernel(const unsigned long long* __restrict__ best, int64_t m, int64_t* __restrict__ idx,
                                  float* __restrict__ cost) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const unsigned long long p = best[i];
  idx[i] = (int64_t)(p & 0xffffffffu);
  cost[i] = __uint_as_float((unsigned)(p >> 32));
}

// ---- k nearest entries ----------------------------------------------------------------------------------------
// lut_topk_kernel: the search of lut_nearest_kernel (same FP32 cost: weighting, padding, c0 / c1 interleaving and
// fmaf order, so k = 1 gives its index and cost bit for bit), keeping the k smallest words (cost bits << 32 | global
// index) per observation instead of one.  Costs are >= 0, so unsigned word order is (cost, index) order.
//   heap   = each thread's k words as a max-heap in a column of dynamic shared memory ([k][blockDim.x], conflict-free);
//            the root is the k-th best so far and starts as the all-ones "no entry" word
//   filter = an entry enters only if its cost is below the root's (below 3e38 while a "no entry" word is the root):
//            a slice is walked in ascending index order, so an equal cost loses to the root's lower index and the
//            compare is the word order.  After the first k entries the inner loop is the nearest kernel's loop;
//            the heap is entered ~k ln(n_slice / k) times per observation and slice (replace root, sift down);
//            4 entries per unrolled step keep enough independent cost chains in flight at the lower occupancy the
//            heaps leave (measured +2..9 % at k = 16..50 over 2)
//   result = each list heap-sorted ascending and written to lists [slice][m][k]; lut_topk_merge_kernel reduces them
constexpr int kLutTopkMax = 128;

// replace the root of the max-heap h[0..size) (element i at h[i * stride]) by w and restore the heap order
__device__ __forceinline__ void topk_sift_down(unsigned long long* h, int stride, int size, unsigned long long w) {
  int i = 0;
  for (int c = 1; c < size; c = 2 * i + 1) {
    unsigned long long cv = h[c * stride];
    if (c + 1 < size) {
      const unsigned long long r = h[(c + 1) * stride];
      if (r > cv) {
        cv = r;
        ++c;
      }
    }
    if (cv <= w) break;
    h[i * stride] = cv;
    i = c;
  }
  h[i * stride] = w;
}

template <int NB4>   // bands padded to 4 * NB4
__global__ void __launch_bounds__(kLutObs)
lut_topk_kernel(const float* __restrict__ lut, int64_t n, int nb, const float* __restrict__ obs, int64_t m,
                const float* __restrict__ sqrt_w, int64_t per_slice, unsigned index_offset, int k,
                unsigned long long* __restrict__ lists) {
  constexpr int NBP = 4 * NB4;
  __shared__ __align__(16) float s_l[kLutTile][NBP];
  __shared__ float s_w[NBP];
  extern __shared__ unsigned long long s_heap[];
  const int nt = blockDim.x;
  unsigned long long* h = s_heap + threadIdx.x;
  for (int j = 0; j < k; ++j) h[j * nt] = ~0ull;
  for (int b = threadIdx.x; b < NBP; b += blockDim.x) s_w[b] = (b < nb) ? (sqrt_w ? sqrt_w[b] : 1.0f) : 0.0f;
  __syncthreads();
  const int64_t oi = (int64_t)blockIdx.x * nt + threadIdx.x;
  const int64_t oc = oi < m ? oi : m - 1;
  float o[NBP];
#pragma unroll
  for (int b = 0; b < NBP; ++b) o[b] = (b < nb) ? obs[oc * nb + b] * s_w[b] : 0.0f;
  const int64_t e0 = (int64_t)blockIdx.y * per_slice;
  const int64_t e1 = (e0 + per_slice < n) ? e0 + per_slice : n;
  float thr = 3.0e38f;
  for (int64_t t0 = e0; t0 < e1; t0 += kLutTile) {
    const int cnt = (int)((e1 - t0 < kLutTile) ? (e1 - t0) : kLutTile);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt * NBP; i += blockDim.x) {
      const int e = i / NBP, b = i % NBP;
      s_l[e][b] = (b < nb) ? lut[(t0 + e) * nb + b] * s_w[b] : 0.0f;
    }
    __syncthreads();
#pragma unroll 4
    for (int e = 0; e < cnt; ++e) {
      const float4* row = reinterpret_cast<const float4*>(s_l[e]);
      float c0 = 0.0f, c1 = 0.0f;
#pragma unroll
      for (int q = 0; q < NB4; ++q) {
        const float4 l = row[q];
        const float d0 = o[4 * q] - l.x, d1 = o[4 * q + 1] - l.y, d2 = o[4 * q + 2] - l.z, d3 = o[4 * q + 3] - l.w;
        c0 = fmaf(d0, d0, c0);
        c1 = fmaf(d1, d1, c1);
        c0 = fmaf(d2, d2, c0);
        c1 = fmaf(d3, d3, c1);
      }
      const float c = c0 + c1;
      if (c < thr) {
        topk_sift_down(h, nt, k, ((unsigned long long)__float_as_uint(c) << 32) | ((unsigned)(t0 + e) + index_offset));
        thr = fminf(__uint_as_float((unsigned)(h[0] >> 32)), 3.0e38f);   // a "no entry" root has cost bits NaN
      }
    }
  }
  for (int end = k - 1; end > 0; --end) {   // heap sort: ascending words
    const unsigned long long top = h[0];
    topk_sift_down(h, nt, end, h[end * nt]);
    h[end * nt] = top;
  }
  if (oi < m) {
    unsigned long long* out = lists + ((int64_t)blockIdx.y * m + oi) * k;
    for (int j = 0; j < k; ++j) out[j] = h[j * nt];
  }
}

// L ascending lists of k words per observation (lists [L][m][k]) -> the k smallest words, ascending.  One warp per
// observation: each lane owns lists lane, lane + 32, ... and keeps the smallest of their heads; per output slot a
// warp min picks the winner, whose owner (the lowest such lane) advances that list and re-scans its heads.  Heads
// and cursors live in dynamic shared memory: [warps][L] words, then [warps][L] bytes.  Once the winner is the
// "no entry" word every list is exhausted and the remaining slots are filled with it.  Writes each output that is
// not NULL: idx / cost (unpacked as lut_unpack_kernel does) and packed.
__global__ void lut_topk_merge_kernel(const unsigned long long* __restrict__ lists, int L, int64_t m, int k,
                                      int64_t* __restrict__ idx, float* __restrict__ cost,
                                      unsigned long long* __restrict__ packed) {
  extern __shared__ unsigned long long s_merge[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  const int64_t o = (int64_t)blockIdx.x * warps + warp;
  if (o >= m) return;                                  // whole warps leave together
  unsigned long long* head = s_merge + (int64_t)warp * L;
  unsigned char* cur = reinterpret_cast<unsigned char*>(s_merge + (int64_t)warps * L) + (int64_t)warp * L;
  const unsigned long long* base = lists + o * k;
  const int64_t lstride = m * k;
  unsigned long long mine = ~0ull;
  int mine_l = 0;
  for (int l = lane; l < L; l += 32) {
    const unsigned long long v = base[l * lstride];
    head[l] = v;
    cur[l] = 0;
    if (v < mine) {
      mine = v;
      mine_l = l;
    }
  }
  const int64_t out0 = o * k;
  for (int r = 0; r < k; ++r) {
    unsigned long long w = mine;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long x = __shfl_xor_sync(0xffffffffu, w, d);
      w = x < w ? x : w;
    }
    if (w == ~0ull) {                                  // warp-uniform
      for (int j = r + lane; j < k; j += 32) {
        if (idx) idx[out0 + j] = 0xffffffffLL;
        if (cost) cost[out0 + j] = __uint_as_float(0xffffffffu);
        if (packed) packed[out0 + j] = ~0ull;
      }
      return;
    }
    if (lane == 0) {
      if (idx) idx[out0 + r] = (int64_t)(w & 0xffffffffu);
      if (cost) cost[out0 + r] = __uint_as_float((unsigned)(w >> 32));
      if (packed) packed[out0 + r] = w;
    }
    const unsigned own = __ballot_sync(0xffffffffu, mine == w);
    if (lane == __ffs(own) - 1) {
      const int c = ++cur[mine_l];
      head[mine_l] = c < k ? base[mine_l * lstride + c] : ~0ull;
      mine = ~0ull;
      for (int l = lane; l < L; l += 32) {
        const unsigned long long v = head[l];
        if (v < mine) {
          mine = v;
          mine_l = l;
        }
      }
    }
    __syncwarp();
  }
}

// ---- moments of the parameters of the chosen entries ---------------------------------------------------------
// Thread = (observation o, column p of acc [m][P + 1]).  Over the neighbours j of o in index order, those whose index
// lies in this table piece [index_offset, index_offset + n_local) add x = params[p * stride_param + e * stride_entry]
// (e = local index) -- or (x - centre[o][p])^2 with a centre -- in FP64; column P adds 1 per such neighbour (the
// count).  The sum is added to acc, so pieces of a sharded table accumulate into one buffer.
template <typename T>
__global__ void lut_moments_kernel(const T* __restrict__ params, int P, int64_t stride_param, int64_t stride_entry,
                                   int64_t index_offset, int64_t n_local, const int64_t* __restrict__ index,
                                   int64_t m, int k, const double* __restrict__ centre, double* __restrict__ acc) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m * (P + 1)) return;
  const int64_t o = t / (P + 1);
  const int p = (int)(t - o * (P + 1));
  const double c = (centre && p < P) ? centre[o * P + p] : 0.0;
  double s = 0.0;
  for (int j = 0; j < k; ++j) {
    const int64_t e = index[o * k + j] - index_offset;
    if (e < 0 || e >= n_local) continue;
    if (p == P) {
      s += 1.0;
    } else {
      const double x = (double)params[p * stride_param + e * stride_entry];
      if (centre) {
        const double d = x - c;
        s += d * d;
      } else {
        s += x;
      }
    }
  }
  acc[t] += s;
}

// mean = sum / count, std = sqrt(sum of squared deviations / count) (population); count 0 gives NaN for both.
// Without sq only mean and count are written.
__global__ void lut_moments_finish_kernel(const double* __restrict__ sum, const double* __restrict__ sq, int64_t m,
                                          int P, double* __restrict__ mean, double* __restrict__ sd,
                                          int64_t* __restrict__ count) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m * (P + 1)) return;
  const int64_t o = t / (P + 1);
  const int p = (int)(t - o * (P + 1));
  const double cnt = sum[o * (P + 1) + P];
  if (p == P) {
    count[o] = (int64_t)cnt;
    return;
  }
  mean[o * P + p] = sum[t] / cnt;
  if (sq) sd[o * P + p] = sqrt(sq[t] / cnt);
}

}  // namespace spart

// ---- tensor-core variant ------------------------------------------------------------------------
// The same search as a skinny GEMM on the tensor cores: C[obs, entry] = |l|^2 - 2 o.l (the |o|^2 term is
// constant per observation), K = the band axis padded to 16 with two spare slots carrying |l|^2 (split in
// two TF32 halves) against a constant 1 on the observation side.  Operands are split 3xTF32
// (a = a_hi + a_lo, C += a_hi b_hi + a_lo b_hi + a_hi b_lo), which brings the products to ~2^-21 of
// |o||l| -- plain TF32 / BF16 would lose the distances between the near-identical spectra a retrieval
// compares.  mma.sync.m16n8k8 (the warp-level MMA path; K = 16 is far too short to feed a tcgen05 pipeline,
// and the kernel is bound by the min / index bookkeeping of the epilogue, 3 instructions per pair, not by
// the MMAs).  The winner of the approximate search is re-costed exactly in FP32 (lut_refine_kernel), so the
// reported cost is exact; the chosen entry is optimal up to the 3xTF32 error of the comparison
// (~1e-6 |o||l|), which is why the exact SIMT kernel stays the default.
constexpr int kTcWarps = 4;
constexpr int kTcTile = 128;                       // LUT entries staged per shared-memory tile

__device__ __forceinline__ unsigned tf32_hi(float x) {
  unsigned r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ void mma_tf32(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// KS: k-steps of 8 (bands + 2 <= 8 KS); MT: M-tiles of 16 observations per warp
template <int KS, int MT>
__global__ void __launch_bounds__(kTcWarps * 32)
lut_nearest_tc_kernel(const float* __restrict__ lut, int64_t n, int nb, const float* __restrict__ obs, int64_t m,
                      const float* __restrict__ sqrt_w, int64_t per_slice, unsigned index_offset,
                      unsigned long long* __restrict__ best) {
  constexpr int K = 8 * KS;
  constexpr int kStride = K + 4;                     // + 4 padding: conflict-free B fragment loads
  constexpr int kObsPerWarp = 16 * MT;
  __shared__ __align__(16) unsigned s_hi[kTcTile][kStride], s_lo[kTcTile][kStride];
  __shared__ float s_w[K];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, q = lane & 3;             // fragment row group / column group
  for (int b = threadIdx.x; b < K; b += blockDim.x) s_w[b] = (b < nb) ? (sqrt_w ? sqrt_w[b] : 1.0f) : 0.0f;
  __syncthreads();
  // A fragments: 4 M-tiles x 2 k-steps x {hi, lo}; row r of tile t is observation base + 16 t + r.
  // A[row][k] = -2 w_k o_k for k < nb, 1 for the two |l|^2 slots (13, 14 -> here nb, nb + 1), 0 beyond.
  const int64_t obase = ((int64_t)blockIdx.x * kTcWarps + warp) * kObsPerWarp;
  unsigned ah[MT][KS][4], al[MT][KS][4];
  float o2[MT][2];
#pragma unroll
  for (int t = 0; t < MT; ++t) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {                    // the two rows of this thread in tile t: g and g + 8
      const int64_t oi = obase + 16 * t + g + 8 * h;
      const int64_t oc = oi < m ? oi : m - 1;
      float acc = 0.0f;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {                // columns q and q + 4 of k-step ks
          const int k = 8 * ks + q + 4 * c;
          float v;
          if (k < nb) {
            const float ow = obs[oc * nb + k] * s_w[k];
            acc = fmaf(ow, ow, acc);
            v = -2.0f * ow;
          } else {
            v = (k == nb || k == nb + 1) ? 1.0f : 0.0f;
          }
          const unsigned hi = tf32_hi(v);
          ah[t][ks][h + 2 * c] = hi;
          al[t][ks][h + 2 * c] = tf32_hi(v - __uint_as_float(hi));
        }
      }
      o2[t][h] = acc;                                // partial |o|^2 over this thread's columns
    }
  }
#pragma unroll
  for (int t = 0; t < MT; ++t)
#pragma unroll
    for (int h = 0; h < 2; ++h) {                    // complete |o|^2 over the 4 lanes of a row group
      o2[t][h] += __shfl_xor_sync(0xffffffffu, o2[t][h], 1);
      o2[t][h] += __shfl_xor_sync(0xffffffffu, o2[t][h], 2);
    }
  float bv[MT][2];
  unsigned bi[MT][2];
#pragma unroll
  for (int t = 0; t < MT; ++t)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      bv[t][h] = 3.0e38f;
      bi[t][h] = 0xffffffffu;
    }
  const int64_t e0 = (int64_t)blockIdx.y * per_slice;
  const int64_t e1 = (e0 + per_slice < n) ? e0 + per_slice : n;
  for (int64_t t0 = e0; t0 < e1; t0 += kTcTile) {
    const int cnt = (int)((e1 - t0 < kTcTile) ? (e1 - t0) : kTcTile);
    __syncthreads();
    // stage the tile: one thread per entry builds its padded, weighted row and |l|^2 (entries beyond cnt
    // get |l|^2 = NaN: their comparisons are false, so they never win, not even against NaN-only entries)
    for (int e = threadIdx.x; e < kTcTile; e += blockDim.x) {
      float l2 = 0.0f;
      for (int k = 0; k < K; ++k) {
        float v = 0.0f;
        if (k < nb && e < cnt) {
          v = lut[(t0 + e) * nb + k] * s_w[k];
          l2 = fmaf(v, v, l2);
        }
        if (k < nb) {
          const unsigned hi = tf32_hi(v);
          s_hi[e][k] = hi;
          s_lo[e][k] = tf32_hi(v - __uint_as_float(hi));
        }
      }
      if (e >= cnt) l2 = __int_as_float(0x7fc00000);
      const unsigned h2 = tf32_hi(l2);
      s_hi[e][nb] = h2;                              // |l|^2 = h2 + rest, both meet the constant 1 of A
      s_lo[e][nb] = 0u;
      const float rest = l2 - __uint_as_float(h2);
      const unsigned h3 = tf32_hi(rest);
      s_hi[e][nb + 1] = h3;
      s_lo[e][nb + 1] = tf32_hi(rest - __uint_as_float(h3));
      for (int k = nb + 2; k < K; ++k) {
        s_hi[e][k] = 0u;
        s_lo[e][k] = 0u;
      }
    }
    __syncthreads();
#pragma unroll 2
    for (int nt = 0; nt < kTcTile / 8; ++nt) {       // 8 entries per MMA tile: column g of B is entry 8 nt + g
      const int e = 8 * nt + g;
      unsigned bh[KS][2], bl[KS][2];
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        bh[ks][0] = s_hi[e][8 * ks + q];
        bh[ks][1] = s_hi[e][8 * ks + q + 4];
        bl[ks][0] = s_lo[e][8 * ks + q];
        bl[ks][1] = s_lo[e][8 * ks + q + 4];
      }
      const unsigned col0 = (unsigned)(t0 + 8 * nt + 2 * q);        // C columns of this thread: 2 q and 2 q + 1
#pragma unroll
      for (int t = 0; t < MT; ++t) {
        float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
          mma_tf32(c, al[t][ks], bh[ks][0], bh[ks][1]);
          mma_tf32(c, ah[t][ks], bl[ks][0], bl[ks][1]);
          mma_tf32(c, ah[t][ks], bh[ks][0], bh[ks][1]);
        }
        // c[0], c[1]: row g, columns 2q, 2q+1;  c[2], c[3]: row g + 8
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float v0 = c[2 * h], v1 = c[2 * h + 1];
          if (v0 < bv[t][h]) { bv[t][h] = v0; bi[t][h] = col0; }
          if (v1 < bv[t][h]) { bv[t][h] = v1; bi[t][h] = col0 + 1; }
        }
      }
    }
  }
  // per row: minimum over the 4 lanes of the row group (ties to the lower index), then one atomicMin
#pragma unroll
  for (int t = 0; t < MT; ++t)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v = fmaxf(bv[t][h] + o2[t][h], 0.0f);
      unsigned long long p = ((unsigned long long)__float_as_uint(v) << 32) | (bi[t][h] + (bi[t][h] == 0xffffffffu ? 0u : index_offset));
      for (int d = 1; d <= 2; d <<= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, p, d);
        p = o < p ? o : p;
      }
      const int64_t oi = obase + 16 * t + g + 8 * h;
      if (q == 0 && oi < m && bi[t][h] != 0xffffffffu) atomicMin(&best[oi], p);
    }
}

// exact FP32 cost of the entry the tensor-core search picked (same arithmetic as lut_nearest_kernel)
__global__ void lut_refine_kernel(const float* __restrict__ lut, int nb, const float* __restrict__ obs, int64_t m,
                                  const float* __restrict__ sqrt_w, unsigned index_offset,
                                  unsigned long long* __restrict__ best) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const unsigned idx = (unsigned)(best[i] & 0xffffffffu);
  if (idx == 0xffffffffu) return;
  const float* l = lut + (int64_t)(idx - index_offset) * nb;
  float c0 = 0.0f, c1 = 0.0f;
  for (int b = 0; b < nb; ++b) {
    const float w = sqrt_w ? sqrt_w[b] : 1.0f;
    const float d = obs[i * nb + b] * w - l[b] * w;
    if (b & 1) c1 = fmaf(d, d, c1);
    else c0 = fmaf(d, d, c0);
  }
  best[i] = ((unsigned long long)__float_as_uint(c0 + c1) << 32) | idx;
}
