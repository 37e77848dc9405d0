// gatlayer_kernels.cu -- one single-head GATConv layer of any small width (in_channels, out_channels <= 64) on an
// arbitrary graph, forward and full backward (parameters AND node features), so that stacks of attention layers can be
// assembled and trained through torch autograd (SURVEY.md 8f rank 4: the older Flocking checkpoints of the reference,
// data/models/experiment_Flocking-seed_*.pth, hold three such layers of width 8).  Semantics = torch_geometric 2.5.3
// GATConv(in, out, heads=1, add_self_loops=False, bias=True).forward as train_gcn_dqn.py:53,61 uses it:
//   h = x W^T; e_(j->i) = LeakyReLU_0.2(h_j . a_src + h_i . a_dst); alpha = softmax over the edges into i (max-subtracted,
//   denominator + 1e-16); out_i = sum_j alpha h_j (edge-list order) + bias.
// Gather-only, no atomics, every reduction in a fixed order -> bit-reproducible results:
//   project        thread = node                 rows[n][CO_T + 4] = (h, h.a_src, h.a_dst)
//   aggregate      thread = target node          softmax over its in-edge group, weighted sum
//   bwd_target     thread = target node          alpha_e, d(raw logit)_e per in-edge, d(h_i . a_dst)
//   bwd_source     thread = source node          d h_j from its out-edges (CSR by source), d x_j = d h_j W
//   param_partial  CTA = contiguous node range,  thread = parameter element: sums over the range
//   param_reduce   thread = parameter element:   sums the partials in CTA order
// CO_T (8 / 16 / 32 / 64) is the compile-time row width the runtime out_channels is padded to.
#include <cstdint>

#include "gatq_device.cuh"
#include "swarm_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kGlThreads = 128;

struct GatLayerParams {
  int n, ci, co;
  long long E;
  const float* W;            // [co][ci]
  const float* a_src;        // [co]
  const float* a_dst;        // [co]
  const float* bias;         // [co]
  const float* x;            // [n][ci]
  const int32_t* row_ptr;    // CSR by target, edge-list order inside a group
  const int32_t* src;
  const int32_t* row_ptr_s;  // CSR by source
  const int32_t* tgt_s;
  const int32_t* pos_s;      // by-target position of out-edge q
  const float* grad_out;     // [n][co]
  float* out;                // [n][co]
  float* rows;               // [n][CO_T + 4]
  float* alpha;              // [E] by-target order
  float* draw;               // [E] by-target order
  float* dd;                 // [n]
  float* ds;                 // [n]
  float* dh;                 // [n][CO_T]
  float* grad_x;             // [n][ci] or NULL
  float* partials;           // [P][n_params]
  int nodes_per_cta;
};

template <int CO_T>
__global__ void __launch_bounds__(kGlThreads) gl_project_kernel(const __grid_constant__ GatLayerParams p) {
  extern __shared__ __align__(16) float gl_smem[];
  float* sW = gl_smem;                    // [ci][CO_T] (transposed, zero padded)
  float* sas = sW + p.ci * CO_T;
  float* sad = sas + CO_T;
  for (int e = threadIdx.x; e < p.ci * CO_T; e += blockDim.x) {
    const int k = e / CO_T, c = e - k * CO_T;
    sW[e] = c < p.co ? p.W[c * p.ci + k] : 0.0f;
  }
  for (int c = threadIdx.x; c < CO_T; c += blockDim.x) {
    sas[c] = c < p.co ? p.a_src[c] : 0.0f;
    sad[c] = c < p.co ? p.a_dst[c] : 0.0f;
  }
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  float h[CO_T];
#pragma unroll
  for (int c = 0; c < CO_T; ++c) h[c] = 0.0f;
  const float* xr = p.x + (long long)i * p.ci;
  for (int k = 0; k < p.ci; ++k) {
    const float xv = xr[k];
    const float4* w4 = reinterpret_cast<const float4*>(sW + k * CO_T);
#pragma unroll
    for (int c4 = 0; c4 < CO_T / 4; ++c4) {
      const float4 w = w4[c4];
      h[4 * c4 + 0] = fmaf(xv, w.x, h[4 * c4 + 0]);
      h[4 * c4 + 1] = fmaf(xv, w.y, h[4 * c4 + 1]);
      h[4 * c4 + 2] = fmaf(xv, w.z, h[4 * c4 + 2]);
      h[4 * c4 + 3] = fmaf(xv, w.w, h[4 * c4 + 3]);
    }
  }
  float s = 0.0f, d = 0.0f;
#pragma unroll
  for (int c = 0; c < CO_T; ++c) {
    s = fmaf(h[c], sas[c], s);
    d = fmaf(h[c], sad[c], d);
  }
  float4* row = reinterpret_cast<float4*>(p.rows + (long long)i * (CO_T + 4));
#pragma unroll
  for (int c4 = 0; c4 < CO_T / 4; ++c4) row[c4] = make_float4(h[4 * c4], h[4 * c4 + 1], h[4 * c4 + 2], h[4 * c4 + 3]);
  row[CO_T / 4] = make_float4(s, d, 0.0f, 0.0f);
}

// softmax statistics of the in-edge group of node i: max logit and denominator (+ 1e-16), PyG utils.softmax
template <int CO_T>
__device__ __forceinline__ void gl_softmax_stats(const GatLayerParams& p, int e0, int e1, float adst, float& m, float& den) {
  constexpr int RS = CO_T + 4;
  m = -INFINITY;
  for (int e = e0; e < e1; ++e) m = fmaxf(m, gat_logit(p.rows[(long long)p.src[e] * RS + CO_T], adst));
  den = 0.0f;
  for (int e = e0; e < e1; ++e)
    den = __fadd_rn(den, expf(__fsub_rn(gat_logit(p.rows[(long long)p.src[e] * RS + CO_T], adst), m)));
  den = __fadd_rn(den, 1e-16f);
}

template <int CO_T>
__global__ void __launch_bounds__(kGlThreads) gl_aggregate_kernel(const __grid_constant__ GatLayerParams p) {
  constexpr int RS = CO_T + 4;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const int e0 = p.row_ptr[i], e1 = p.row_ptr[i + 1];
  const float adst = p.rows[(long long)i * RS + CO_T + 1];
  float m, den;
  gl_softmax_stats<CO_T>(p, e0, e1, adst, m, den);
  float acc[CO_T];
#pragma unroll
  for (int c = 0; c < CO_T; ++c) acc[c] = 0.0f;
  for (int e = e0; e < e1; ++e) {
    const long long j = p.src[e];
    const float a = __fdiv_rn(expf(__fsub_rn(gat_logit(p.rows[j * RS + CO_T], adst), m)), den);
    const float4* hj = reinterpret_cast<const float4*>(p.rows + j * RS);
#pragma unroll
    for (int c4 = 0; c4 < CO_T / 4; ++c4) {
      const float4 hv = hj[c4];
      acc[4 * c4 + 0] = __fadd_rn(acc[4 * c4 + 0], __fmul_rn(a, hv.x));     // message rounded, then scatter-added
      acc[4 * c4 + 1] = __fadd_rn(acc[4 * c4 + 1], __fmul_rn(a, hv.y));
      acc[4 * c4 + 2] = __fadd_rn(acc[4 * c4 + 2], __fmul_rn(a, hv.z));
      acc[4 * c4 + 3] = __fadd_rn(acc[4 * c4 + 3], __fmul_rn(a, hv.w));
    }
  }
  float* o = p.out + (long long)i * p.co;
#pragma unroll
  for (int c = 0; c < CO_T; ++c)
    if (c < p.co) o[c] = __fadd_rn(acc[c], p.bias[c]);
}

template <int CO_T>
__global__ void __launch_bounds__(kGlThreads) gl_bwd_target_kernel(const __grid_constant__ GatLayerParams p) {
  constexpr int RS = CO_T + 4;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  const int e0 = p.row_ptr[i], e1 = p.row_ptr[i + 1];
  const float adst = p.rows[(long long)i * RS + CO_T + 1];
  float m, den;
  gl_softmax_stats<CO_T>(p, e0, e1, adst, m, den);
  float g[CO_T];
  const float* gr = p.grad_out + (long long)i * p.co;
#pragma unroll
  for (int c = 0; c < CO_T; ++c) g[c] = c < p.co ? gr[c] : 0.0f;
  float dot_sum = 0.0f;
  for (int e = e0; e < e1; ++e) {
    const long long j = p.src[e];
    const float a = __fdiv_rn(expf(__fsub_rn(gat_logit(p.rows[j * RS + CO_T], adst), m)), den);
    p.alpha[e] = a;
    const float4* hj = reinterpret_cast<const float4*>(p.rows + j * RS);
    float da = 0.0f;
#pragma unroll
    for (int c4 = 0; c4 < CO_T / 4; ++c4) {
      const float4 hv = hj[c4];
      da = fmaf(g[4 * c4 + 0], hv.x, da);
      da = fmaf(g[4 * c4 + 1], hv.y, da);
      da = fmaf(g[4 * c4 + 2], hv.z, da);
      da = fmaf(g[4 * c4 + 3], hv.w, da);
    }
    p.draw[e] = da;
    dot_sum = fmaf(a, da, dot_sum);
  }
  float dd_i = 0.0f;
  for (int e = e0; e < e1; ++e) {
    const float dz = p.alpha[e] * (p.draw[e] - dot_sum);
    const float raw = __fadd_rn(p.rows[(long long)p.src[e] * RS + CO_T], adst);
    const float dzz = raw > 0.0f ? dz : 0.2f * dz;
    p.draw[e] = dzz;
    dd_i += dzz;
  }
  p.dd[i] = dd_i;
}

template <int CO_T>
__global__ void __launch_bounds__(kGlThreads) gl_bwd_source_kernel(const __grid_constant__ GatLayerParams p) {
  extern __shared__ __align__(16) float gl_smem[];
  float* sW = gl_smem;                    // [CO_T][ci] zero padded rows
  float* sas = sW + CO_T * p.ci;
  float* sad = sas + CO_T;
  for (int e = threadIdx.x; e < CO_T * p.ci; e += blockDim.x) sW[e] = e < p.co * p.ci ? p.W[e] : 0.0f;
  for (int c = threadIdx.x; c < CO_T; c += blockDim.x) {
    sas[c] = c < p.co ? p.a_src[c] : 0.0f;
    sad[c] = c < p.co ? p.a_dst[c] : 0.0f;
  }
  __syncthreads();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.n) return;
  float dh[CO_T];
#pragma unroll
  for (int c = 0; c < CO_T; ++c) dh[c] = 0.0f;
  float ds_j = 0.0f;
  const int q0 = p.row_ptr_s[j], q1 = p.row_ptr_s[j + 1];
  for (int q = q0; q < q1; ++q) {
    const int pp = p.pos_s[q];
    const float a = p.alpha[pp];
    ds_j += p.draw[pp];
    const float* gr = p.grad_out + (long long)p.tgt_s[q] * p.co;
#pragma unroll
    for (int c = 0; c < CO_T; ++c)
      if (c < p.co) dh[c] = fmaf(a, gr[c], dh[c]);
  }
  const float dd_j = p.dd[j];
#pragma unroll
  for (int c = 0; c < CO_T; ++c) dh[c] = fmaf(ds_j, sas[c], fmaf(dd_j, sad[c], dh[c]));
  p.ds[j] = ds_j;
  float4* o = reinterpret_cast<float4*>(p.dh + (long long)j * CO_T);
#pragma unroll
  for (int c4 = 0; c4 < CO_T / 4; ++c4) o[c4] = make_float4(dh[4 * c4], dh[4 * c4 + 1], dh[4 * c4 + 2], dh[4 * c4 + 3]);
  if (p.grad_x) {
    float* gx = p.grad_x + (long long)j * p.ci;
    for (int k = 0; k < p.ci; ++k) {
      float acc = 0.0f;
#pragma unroll
      for (int c = 0; c < CO_T; ++c) acc = fmaf(dh[c], sW[c * p.ci + k], acc);
      gx[k] = acc;
    }
  }
}

// parameter element e of the layer: [0, co*ci) lin.weight, then att_src, att_dst, bias (co each)
template <int CO_T>
__global__ void __launch_bounds__(256) gl_param_partial_kernel(const __grid_constant__ GatLayerParams p) {
  constexpr int RS = CO_T + 4;
  const int n_params = p.co * p.ci + 3 * p.co;
  const int lo = blockIdx.x * p.nodes_per_cta;
  const int hi = min(p.n, lo + p.nodes_per_cta);
  float* out = p.partials + (long long)blockIdx.x * n_params;
  for (int e = threadIdx.x; e < n_params; e += blockDim.x) {
    float acc = 0.0f;
    if (e < p.co * p.ci) {                                   // dW[c][k] = sum_j dh_j[c] x_j[k]
      const int c = e / p.ci, k = e - c * p.ci;
      for (int j = lo; j < hi; ++j) acc = fmaf(p.dh[(long long)j * CO_T + c], p.x[(long long)j * p.ci + k], acc);
    } else {
      const int r = e - p.co * p.ci;
      const int which = r / p.co, c = r - which * p.co;
      if (which == 0) {                                      // d att_src[c] = sum_j ds_j h_j[c]
        for (int j = lo; j < hi; ++j) acc = fmaf(p.ds[j], p.rows[(long long)j * RS + c], acc);
      } else if (which == 1) {                               // d att_dst[c] = sum_i dd_i h_i[c]
        for (int j = lo; j < hi; ++j) acc = fmaf(p.dd[j], p.rows[(long long)j * RS + c], acc);
      } else {                                               // d bias[c] = sum_i d out_i[c]
        for (int j = lo; j < hi; ++j) acc += p.grad_out[(long long)j * p.co + c];
      }
    }
    out[e] = acc;
  }
}

__global__ void gl_param_reduce_kernel(const float* __restrict__ partials, int n_ctas, int n_params, int co, int ci,
                                       float* __restrict__ gW, float* __restrict__ gas, float* __restrict__ gad,
                                       float* __restrict__ gb) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_params) return;
  float acc = 0.0f;
  for (int b = 0; b < n_ctas; ++b) acc += partials[(long long)b * n_params + e];
  if (e < co * ci) gW[e] = acc;
  else {
    const int r = e - co * ci;
    const int which = r / co, c = r - which * co;
    (which == 0 ? gas : which == 1 ? gad : gb)[c] = acc;
  }
}

// original edge id -> position in the by-target order (phase 0), then by-source slot -> by-target position (phase 1)
__global__ void gl_edge_positions_kernel(long long E, const int32_t* __restrict__ perm_t,
                                         const int32_t* __restrict__ perm_s, int32_t* __restrict__ inv,
                                         int32_t* __restrict__ pos_s, int phase) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
    if (phase == 0) inv[perm_t[e]] = (int32_t)e;
    else pos_s[e] = inv[perm_s[e]];
  }
}

// ---- host side ------------------------------------------------------------------------------------------------

static size_t gl_align(size_t v) { return (v + 255) & ~(size_t)255; }
static int gl_width(int co) { return co <= 8 ? 8 : co <= 16 ? 16 : co <= 32 ? 32 : 64; }
static int gl_param_ctas(int n, int* nodes_per_cta) {
  int ctas = (n + 255) / 256;
  if (ctas > 148 * 4) ctas = 148 * 4;
  if (ctas < 1) ctas = 1;
  *nodes_per_cta = (n + ctas - 1) / ctas;
  return (n + *nodes_per_cta - 1) / *nodes_per_cta;
}

long long gat_layer_workspace_bytes(int n, long long E, int ci, int co, bool backward) {
  const int cot = gl_width(co);
  size_t bytes = 512 + gl_align((size_t)n * (cot + 4) * 4);
  if (backward) {
    int npc;
    const int ctas = gl_param_ctas(n, &npc);
    bytes += 4 * gl_align((size_t)E * 4) + 2 * gl_align((size_t)n * 4) + gl_align((size_t)n * cot * 4) +
             gl_align((size_t)ctas * (co * ci + 3 * co) * 4);
  }
  return (long long)bytes;
}

template <int CO_T>
static cudaError_t gl_forward(GatLayerParams& p, cudaStream_t stream) {
  const int blocks = (p.n + kGlThreads - 1) / kGlThreads;
  const int smem = (p.ci * CO_T + 2 * CO_T) * 4;
  gl_project_kernel<CO_T><<<blocks, kGlThreads, smem, stream>>>(p);
  if (p.out) gl_aggregate_kernel<CO_T><<<blocks, kGlThreads, 0, stream>>>(p);
  return cudaGetLastError();
}

template <int CO_T>
static cudaError_t gl_backward(GatLayerParams& p, const int32_t* perm, const int32_t* perm_s, int32_t* inv, int32_t* pos_s,
                               float* gW, float* gas, float* gad, float* gb, cudaStream_t stream) {
  cudaError_t err = gl_forward<CO_T>(p, stream);               // p.out == NULL: projection only
  if (err != cudaSuccess) return err;
  if (p.E > 0) {
    long long blocks = (p.E + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    gl_edge_positions_kernel<<<(int)blocks, 256, 0, stream>>>(p.E, perm, perm_s, inv, pos_s, 0);
    gl_edge_positions_kernel<<<(int)blocks, 256, 0, stream>>>(p.E, perm, perm_s, inv, pos_s, 1);
  }
  const int blocks = (p.n + kGlThreads - 1) / kGlThreads;
  gl_bwd_target_kernel<CO_T><<<blocks, kGlThreads, 0, stream>>>(p);
  const int smem = (p.ci * CO_T + 2 * CO_T) * 4;
  gl_bwd_source_kernel<CO_T><<<blocks, kGlThreads, smem, stream>>>(p);
  const int ctas = gl_param_ctas(p.n, &p.nodes_per_cta);
  gl_param_partial_kernel<CO_T><<<ctas, 256, 0, stream>>>(p);
  const int n_params = p.co * p.ci + 3 * p.co;
  gl_param_reduce_kernel<<<(n_params + 255) / 256, 256, 0, stream>>>(p.partials, ctas, n_params, p.co, p.ci, gW, gas, gad,
                                                                     gb);
  return cudaGetLastError();
}

cudaError_t launch_gat_layer_forward(int n, int ci, int co, const float* W, const float* a_src, const float* a_dst,
                                     const float* bias, const float* x, const int32_t* row_ptr, const int32_t* src,
                                     float* out, void* workspace, cudaStream_t stream) {
  GatLayerParams p{};
  p.n = n; p.ci = ci; p.co = co;
  p.W = W; p.a_src = a_src; p.a_dst = a_dst; p.bias = bias; p.x = x;
  p.row_ptr = row_ptr; p.src = src; p.out = out;
  p.rows = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  switch (gl_width(co)) {
    case 8: return gl_forward<8>(p, stream);
    case 16: return gl_forward<16>(p, stream);
    case 32: return gl_forward<32>(p, stream);
    default: return gl_forward<64>(p, stream);
  }
}

cudaError_t launch_gat_layer_backward(int n, long long E, int ci, int co, const float* W, const float* a_src,
                                      const float* a_dst, const float* x, const int32_t* row_ptr, const int32_t* src,
                                      const int32_t* perm, const int32_t* row_ptr_s, const int32_t* tgt_s,
                                      const int32_t* perm_s, const float* grad_out, float* gW, float* gas, float* gad,
                                      float* gb, float* grad_x, void* workspace, cudaStream_t stream) {
  const int cot = gl_width(co);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  auto take = [&](size_t bytes) { char* q = base; base += gl_align(bytes); return q; };
  GatLayerParams p{};
  p.n = n; p.ci = ci; p.co = co; p.E = E;
  p.W = W; p.a_src = a_src; p.a_dst = a_dst; p.x = x;
  p.row_ptr = row_ptr; p.src = src; p.row_ptr_s = row_ptr_s; p.tgt_s = tgt_s;
  p.grad_out = grad_out; p.grad_x = grad_x; p.out = nullptr;
  p.rows = reinterpret_cast<float*>(take((size_t)n * (cot + 4) * 4));
  p.alpha = reinterpret_cast<float*>(take((size_t)E * 4));
  p.draw = reinterpret_cast<float*>(take((size_t)E * 4));
  int32_t* inv = reinterpret_cast<int32_t*>(take((size_t)E * 4));
  int32_t* pos_s = reinterpret_cast<int32_t*>(take((size_t)E * 4));
  p.pos_s = pos_s;
  p.dd = reinterpret_cast<float*>(take((size_t)n * 4));
  p.ds = reinterpret_cast<float*>(take((size_t)n * 4));
  p.dh = reinterpret_cast<float*>(take((size_t)n * cot * 4));
  int npc;
  const int ctas = gl_param_ctas(n, &npc);
  p.partials = reinterpret_cast<float*>(take((size_t)ctas * (co * ci + 3 * co) * 4));
  switch (cot) {
    case 8: return gl_backward<8>(p, perm, perm_s, inv, pos_s, gW, gas, gad, gb, stream);
    case 16: return gl_backward<16>(p, perm, perm_s, inv, pos_s, gW, gas, gad, gb, stream);
    case 32: return gl_backward<32>(p, perm, perm_s, inv, pos_s, gW, gas, gad, gb, stream);
    default: return gl_backward<64>(p, perm, perm_s, inv, pos_s, gW, gas, gad, gb, stream);
  }
}

}  // namespace swarm
