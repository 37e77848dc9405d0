// csr_kernels.cu -- GCN.forward on an arbitrary graph (the nn.Module seam, train_gcn_dqn.py:59-70, for
// Data / Batch inputs that did not come from the structured per-env builders) and the stable grouping
// of an edge list by target node that gives the aggregation its reference (edge-list) order.
#include <cub/device/device_radix_sort.cuh>

#include <string>

#include "gatq_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kCsrThreads = 128;
constexpr int kRow = 36;   // workspace row: h[32], alpha_src, alpha_dst, pad

__global__ void __launch_bounds__(kCsrThreads) csr_project_kernel(int n, const float* __restrict__ weights,
                                                                  const float* __restrict__ x,
                                                                  float* __restrict__ rows) {
  __shared__ __align__(16) float sw[TW_COUNT];
  stage_weights(weights, sw, threadIdx.x, kCsrThreads);
  __syncthreads();
  const int i = blockIdx.x * kCsrThreads + threadIdx.x;
  if (i >= n) return;
  float xi[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) xi[k] = x[(long long)i * 7 + k];
  float h[32], asrc, adst;
  gat_project(xi, sw, h, asrc, adst);
  float4* r = reinterpret_cast<float4*>(rows + (long long)i * kRow);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) r[c4] = make_float4(h[4 * c4], h[4 * c4 + 1], h[4 * c4 + 2], h[4 * c4 + 3]);
  r[8] = make_float4(asrc, adst, 0.0f, 0.0f);
}

// HEAD = true: the whole Q-network (aggregate + bias -> tanh -> lin1 -> ReLU -> lin2); HEAD = false: the GATConv layer
// alone, q_out = float[n][32] = aggregate + conv1.bias (torch_geometric GATConv.forward)
template <bool HEAD>
__global__ void __launch_bounds__(kCsrThreads) csr_aggregate_kernel(int n, const float* __restrict__ weights,
                                                                    const float* __restrict__ rows,
                                                                    const int32_t* __restrict__ row_ptr,
                                                                    const int32_t* __restrict__ src,
                                                                    float* __restrict__ q_out,
                                                                    int32_t* __restrict__ act_out) {
  __shared__ __align__(16) float sw[TW_COUNT];
  stage_weights(weights, sw, threadIdx.x, kCsrThreads);
  __syncthreads();
  const int i = blockIdx.x * kCsrThreads + threadIdx.x;
  if (i >= n) return;
  const int e0 = row_ptr[i], e1 = row_ptr[i + 1];
  const float adst = rows[(long long)i * kRow + 33];
  float m = -INFINITY;
  for (int e = e0; e < e1; ++e) m = fmaxf(m, gat_logit(rows[(long long)src[e] * kRow + 32], adst));
  float den = 0.0f;
  for (int e = e0; e < e1; ++e)
    den = __fadd_rn(den, expf(__fsub_rn(gat_logit(rows[(long long)src[e] * kRow + 32], adst), m)));
  den = __fadd_rn(den, 1e-16f);
  float a1[32];
#pragma unroll
  for (int cc = 0; cc < 32; ++cc) a1[cc] = 0.0f;
  for (int e = e0; e < e1; ++e) {
    const long long j = src[e];
    const float w = expf(__fsub_rn(gat_logit(rows[j * kRow + 32], adst), m));
    gat_accumulate(a1, __fdiv_rn(w, den), reinterpret_cast<const float4*>(rows + j * kRow));
  }
  if (!HEAD) {
    float4* o = reinterpret_cast<float4*>(q_out + (long long)i * 32);
    const float* b0 = sw + TW_B0;
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4)
      o[c4] = make_float4(__fadd_rn(a1[4 * c4], b0[4 * c4]), __fadd_rn(a1[4 * c4 + 1], b0[4 * c4 + 1]),
                          __fadd_rn(a1[4 * c4 + 2], b0[4 * c4 + 2]), __fadd_rn(a1[4 * c4 + 3], b0[4 * c4 + 3]));
    return;
  }
  float q[9];
  const int action = gat_head(a1, sw, q);
  if (q_out) {
#pragma unroll
    for (int a = 0; a < 9; ++a) q_out[(long long)i * 9 + a] = q[a];
  }
  if (act_out) act_out[i] = action;
}

// ---- edge list -> CSR by target, stable ---------------------------------------------------------
__global__ void csr_prepare_kernel(long long E, const int64_t* __restrict__ dst, int32_t* __restrict__ keys,
                                   int32_t* __restrict__ vals) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
    keys[e] = (int32_t)dst[e];
    vals[e] = (int32_t)e;
  }
}

__global__ void csr_finish_kernel(int n, long long E, const int32_t* __restrict__ keys_sorted,
                                  const int32_t* __restrict__ perm, const int64_t* __restrict__ edge_src,
                                  int32_t* __restrict__ row_ptr, int32_t* __restrict__ src) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = t; i <= n; i += stride) {
    // row_ptr[i] = first position whose key >= i
    long long lo = 0, hi = E;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (keys_sorted[mid] < i) lo = mid + 1;
      else hi = mid;
    }
    row_ptr[i] = (int32_t)lo;
  }
  for (long long e = t; e < E; e += stride) src[e] = (int32_t)edge_src[perm[e]];
}

static int key_bits(int n) {
  int b = 1;
  while ((1LL << b) < n) ++b;
  return b;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static size_t cub_temp_bytes(long long E, int n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, (int)E, 0, key_bits(n));
  return bytes;
}

long long csr_workspace_bytes(int n, long long E) {
  return (long long)(3 * align256((size_t)E * 4) + align256(cub_temp_bytes(E, n)) + 256);
}

cudaError_t launch_csr_from_edges(int n, long long E, const int64_t* edge_src, const int64_t* edge_dst, int32_t* row_ptr,
                                  int32_t* src, int32_t* perm, void* workspace, long long workspace_bytes,
                                  cudaStream_t stream) {
  if (workspace_bytes < csr_workspace_bytes(n, E)) return cudaErrorInvalidValue;
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  const size_t seg = align256((size_t)E * 4);
  int32_t* keys_in = reinterpret_cast<int32_t*>(base);
  int32_t* keys_out = reinterpret_cast<int32_t*>(base + seg);
  int32_t* vals_in = reinterpret_cast<int32_t*>(base + 2 * seg);
  void* temp = base + 3 * seg;
  size_t temp_bytes = cub_temp_bytes(E, n);
  long long blocks = (E + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  if (E > 0) {                                       // an edgeless graph: row_ptr = 0 everywhere, nothing to sort
    csr_prepare_kernel<<<(int)blocks, 256, 0, stream>>>(E, edge_dst, keys_in, vals_in);
    cudaError_t err = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, vals_in, perm, (int)E, 0,
                                                      key_bits(n), stream);
    if (err != cudaSuccess) return err;
  }
  long long work = E > n + 1 ? E : n + 1;
  blocks = (work + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  csr_finish_kernel<<<(int)blocks, 256, 0, stream>>>(n, E, keys_out, perm, edge_src, row_ptr, src);
  return cudaGetLastError();
}

cudaError_t launch_gatq_csr(int n, const float* weights, const float* x, const int32_t* row_ptr, const int32_t* src,
                            float* q, int32_t* actions, float* rows, cudaStream_t stream, bool conv_only) {
  const int blocks = (n + kCsrThreads - 1) / kCsrThreads;
  csr_project_kernel<<<blocks, kCsrThreads, 0, stream>>>(n, weights, x, rows);
  if (conv_only) csr_aggregate_kernel<false><<<blocks, kCsrThreads, 0, stream>>>(n, weights, rows, row_ptr, src, q, nullptr);
  else csr_aggregate_kernel<true><<<blocks, kCsrThreads, 0, stream>>>(n, weights, rows, row_ptr, src, q, actions);
  return cudaGetLastError();
}

cudaError_t launch_csr_project(int n, const float* weights, const float* x, float* rows, cudaStream_t stream) {
  const int blocks = (n + kCsrThreads - 1) / kCsrThreads;
  csr_project_kernel<<<blocks, kCsrThreads, 0, stream>>>(n, weights, x, rows);
  return cudaGetLastError();
}

long long gatq_workspace_bytes(int n) { return (long long)n * kRow * 4 + 256; }

}  // namespace swarm
