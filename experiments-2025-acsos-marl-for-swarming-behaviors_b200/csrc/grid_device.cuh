// grid_device.cuh -- the uniform-grid broad phase of large swarms (one CTA per env, n_agents <= 4096) and the monotone
// float key of the sorted-source kernels, shared by grid_kernels.cu and stack_large_kernels.cu.
#ifndef SWARM_GRID_DEVICE_CUH
#define SWARM_GRID_DEVICE_CUH

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace swarm {

constexpr int kGridThreads = 512;
constexpr int kGridMax = 64;            // cells per axis
constexpr int kGridCells = kGridMax * kGridMax;
constexpr int kIdxBits = 12;            // n_agents <= 4096
constexpr uint32_t kIdxMask = (1u << kIdxBits) - 1u;

struct CellGrid {
  float x0, y0, inv;
  int nx, ny;
  __device__ __forceinline__ int cx(float x) const {
    const int c = (int)fminf(__fmul_rn(__fsub_rn(x, x0), inv), (float)(kGridMax - 1));
    return c < 0 ? 0 : (c >= nx ? nx - 1 : c);
  }
  __device__ __forceinline__ int cy(float y) const {
    const int c = (int)fminf(__fmul_rn(__fsub_rn(y, y0), inv), (float)(kGridMax - 1));
    return c < 0 ? 0 : (c >= ny ? ny - 1 : c);
  }
};

__host__ __device__ inline int grid_pow2(int n) {
  int p = 64;
  while (p < n) p <<= 1;
  return p;
}

// Bins and sorts the env's agents.  Every thread of the CTA calls it (block barriers inside).
//   keys  uint32[P]  (cell << 12 | agent), ascending; P = grid_pow2(N), padded with 0xFFFFFFFF
//   cbeg / cend uint16[kGridCells]: the key range of every cell (empty: 0, 0)
//   sred  float[64] scratch
// Two agents within `radius` of each other (rounded 2-norm) land in the same or in adjacent cells: the cell is 0.1 %
// wider than the radius, the float error of a cell coordinate is below 64 * 2e-7.
template <typename Pos>
__device__ __forceinline__ CellGrid grid_build(Pos pos, int N, int P, float radius, uint32_t* keys, uint16_t* cbeg,
                                               uint16_t* cend, float* sred) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
  for (int j = tid; j < N; j += kGridThreads) {
    const float2 q = pos(j);
    xmin = fminf(xmin, q.x); xmax = fmaxf(xmax, q.x);
    ymin = fminf(ymin, q.y); ymax = fmaxf(ymax, q.y);
  }
#pragma unroll
  for (int sh = 16; sh > 0; sh >>= 1) {
    xmin = fminf(xmin, __shfl_xor_sync(0xffffffffu, xmin, sh));
    xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, sh));
    ymin = fminf(ymin, __shfl_xor_sync(0xffffffffu, ymin, sh));
    ymax = fmaxf(ymax, __shfl_xor_sync(0xffffffffu, ymax, sh));
  }
  if (lane == 0) {
    sred[warp * 4 + 0] = xmin; sred[warp * 4 + 1] = xmax;
    sred[warp * 4 + 2] = ymin; sred[warp * 4 + 3] = ymax;
  }
  for (int c = tid; c < kGridCells; c += kGridThreads) { cbeg[c] = 0; cend[c] = 0; }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kGridThreads / 32; ++w) {
    xmin = fminf(xmin, sred[w * 4 + 0]); xmax = fmaxf(xmax, sred[w * 4 + 1]);
    ymin = fminf(ymin, sred[w * 4 + 2]); ymax = fmaxf(ymax, sred[w * 4 + 3]);
  }
  CellGrid g;
  const float ex = xmax - xmin, ey = ymax - ymin;            // NaN / inf extents collapse the grid to few cells: still exact
  float cell = fmaxf(radius * 1.001f, fmaxf(ex, ey) * (1.0f / kGridMax));
  cell = fmaxf(cell, 1e-20f);
  g.x0 = xmin;
  g.y0 = ymin;
  g.inv = 1.0f / cell;
  g.nx = (int)fminf(ex * g.inv, (float)(kGridMax - 1)) + 1;
  g.ny = (int)fminf(ey * g.inv, (float)(kGridMax - 1)) + 1;
  g.nx = g.nx < 1 ? 1 : g.nx;
  g.ny = g.ny < 1 ? 1 : g.ny;
  for (int j = tid; j < P; j += kGridThreads) {
    uint32_t key = 0xFFFFFFFFu;
    if (j < N) {
      const float2 q = pos(j);
      key = ((uint32_t)(g.cy(q.y) * g.nx + g.cx(q.x)) << kIdxBits) | (uint32_t)j;
    }
    keys[j] = key;
  }
  __syncthreads();
  // bitonic network; a warp's 32 pairs of a stage with distance <= 32 stay inside its own 64-key window, so those
  // stages only need a warp barrier
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < (P >> 1); t += kGridThreads) {
        const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int hi = lo | j;
        const bool up = (lo & k) == 0;
        const uint32_t a = keys[lo], b = keys[hi];
        if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
      }
      const int jn = (j > 1) ? (j >> 1) : k;              // distance of the next stage
      if (j > 32 || jn > 32) __syncthreads(); else __syncwarp();
    }
  }
  __syncthreads();
  for (int p = tid; p < N; p += kGridThreads) {
    const uint32_t c = keys[p] >> kIdxBits;
    if (p == 0 || (keys[p - 1] >> kIdxBits) != c) cbeg[c] = (uint16_t)p;
    if (p == N - 1 || (keys[p + 1] >> kIdxBits) != c) cend[c] = (uint16_t)(p + 1);
  }
  __syncthreads();
  return g;
}

__device__ __forceinline__ bool grid_hit(const float2& pj, const float2& neg, float qmax_r) {
  const float2 d = __fadd2_rn(pj, neg);
  return __fmaf_rn(d.y, d.y, __fmul_rn(d.x, d.x)) <= qmax_r;
}

// monotone map float -> uint32 (ascending)
__device__ __forceinline__ uint32_t float_order_key(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// ascending bitonic sort of P (power of two) uint32 keys carrying uint16 payloads, in shared memory (the barrier scheme
// of grid_build; the network gatq_large_sorted_kernel open-codes).  Every thread of the CTA calls it; ends with a block
// barrier.
__device__ __forceinline__ void bitonic_sort_pairs(uint32_t* keys, uint16_t* perm, int P) {
  const int tid = threadIdx.x;
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < (P >> 1); t += kGridThreads) {
        const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int hi = lo | j;
        const bool up = (lo & k) == 0;
        const uint32_t ka = keys[lo], kb = keys[hi];
        if ((ka > kb) == up) {
          keys[lo] = kb; keys[hi] = ka;
          const uint16_t pa = perm[lo];
          perm[lo] = perm[hi]; perm[hi] = pa;
        }
      }
      const int jn = (j > 1) ? (j >> 1) : k;
      if (j > 32 || jn > 32) __syncthreads(); else __syncwarp();
    }
  }
  __syncthreads();
}

}  // namespace swarm
#endif
