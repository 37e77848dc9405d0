// stack_device.cuh -- the forward of a multi-layer GAT Q-network for one node of an env tile (thread = agent), shared by
// the evaluation kernel (stack_kernels.cu gatstack_kernel) and the DQN gradient kernel (stack_grad_kernels.cu), so that
// the gradient kernel's Q values are the bits swarm_gatstack_forward returns.
#ifndef SWARM_STACK_DEVICE_CUH
#define SWARM_STACK_DEVICE_CUH

#include "tile_device.cuh"

namespace swarm {

constexpr int kStackMaxLayers = 4;

// shared-memory weight block, everything padded to HP channels / 8 input features with zeros
template <int HP>
struct StackLayout {
  static constexpr int kIn0 = 8;                                        // padded input features
  static constexpr int kLayer0 = kIn0 * HP + 3 * HP;                    // WT[8][HP], att_s, att_d, bias
  static constexpr int kLayer = HP * HP + 3 * HP;                       // WT[HP][HP], att_s, att_d, bias
  static constexpr int kW2Cols = 12;
  __host__ __device__ static int layer_off(int l) { return l == 0 ? 0 : kLayer0 + (l - 1) * kLayer; }
  __host__ __device__ static int lin1_off(int L) { return layer_off(L); }
  __host__ __device__ static int lin2_off(int L) { return lin1_off(L) + HP * HP + HP; }
  __host__ __device__ static int total(int L) { return lin2_off(L) + HP * kW2Cols + kW2Cols; }
};

__host__ __device__ inline int stack_weight_count(const SwarmStackSpec& s) {
  const int H = s.hidden;
  int n = 0;
  for (int l = 0; l < s.n_layers; ++l) n += 3 * H + H * (l == 0 ? s.in_features : H);
  return n + H * H + H + 9 * H + 9;
}

// packed weights (state-dict order: per layer att_src, att_dst, bias, lin.weight[H][Cin]; lin1.weight[H][H], lin1.bias,
// lin2.weight[9][H], lin2.bias) -> padded k-major shared layout
template <int HP>
__device__ __forceinline__ void stack_stage_weights(const SwarmStackSpec& s, const float* __restrict__ g, float* __restrict__ sw,
                                                    int tid, int nthreads) {
  using SL = StackLayout<HP>;
  const int H = s.hidden, L = s.n_layers;
  for (int o = tid; o < SL::total(L); o += nthreads) sw[o] = 0.0f;
  __syncthreads();
  int goff = 0;
  for (int l = 0; l < L; ++l) {
    const int cin = l == 0 ? s.in_features : H;
    const int cinp = l == 0 ? SL::kIn0 : HP;
    float* base = sw + SL::layer_off(l);
    float* vec = base + cinp * HP;
    for (int o = tid; o < 3 * H; o += nthreads) vec[(o / H) * HP + (o % H)] = g[goff + o];
    goff += 3 * H;
    for (int o = tid; o < H * cin; o += nthreads) {
      const int c = o / cin, k = o - c * cin;
      base[k * HP + c] = g[goff + o];
    }
    goff += H * cin;
  }
  float* l1 = sw + SL::lin1_off(L);
  for (int o = tid; o < H * H; o += nthreads) {
    const int c = o / H, k = o - c * H;
    l1[k * HP + c] = g[goff + o];
  }
  goff += H * H;
  for (int o = tid; o < H; o += nthreads) l1[HP * HP + o] = g[goff + o];
  goff += H;
  float* l2 = sw + SL::lin2_off(L);
  for (int o = tid; o < 9 * H; o += nthreads) {
    const int a = o / H, k = o - a * H;
    l2[k * SL::kW2Cols + a] = g[goff + o];
  }
  goff += 9 * H;
  for (int o = tid; o < 9; o += nthreads) l2[HP * SL::kW2Cols + o] = g[goff + o];
}

// node features (train:95-99): [pos, vel, goal, agent id] or, with 5 input features, [pos, vel, agent id]
template <int HP>
__device__ __forceinline__ void stack_features(float (&x)[HP], const float4& s, const SwarmConfig& c, int in_features, int i) {
#pragma unroll
  for (int k = 0; k < HP; ++k) x[k] = 0.0f;
  x[0] = s.x; x[1] = s.y; x[2] = s.z; x[3] = s.w;
  if (in_features == 7) {
    x[4] = c.goal_x; x[5] = c.goal_y; x[6] = (float)i;
  } else {
    x[4] = (float)i;
  }
}

// h = x W^T of layer l (sequential-k FFMA chains; float4 weight loads + packed FFMA2: per element the same chain of IEEE
// fused multiply-adds)
template <int HP>
__device__ __forceinline__ void stack_project(const float* __restrict__ base, int l, const float (&x)[HP], float (&h)[HP]) {
  using SL = StackLayout<HP>;
#pragma unroll
  for (int cc = 0; cc < HP; ++cc) h[cc] = 0.0f;
  if (l == 0) {
#pragma unroll
    for (int k = 0; k < SL::kIn0; ++k) {
#pragma unroll
      for (int cc = 0; cc < HP; cc += 4)
        fma4_packed(x[k], *reinterpret_cast<const float4*>(base + k * HP + cc), h[cc], h[cc + 1], h[cc + 2], h[cc + 3]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < HP; ++k) {
#pragma unroll
      for (int cc = 0; cc < HP; cc += 4)
        fma4_packed(x[k], *reinterpret_cast<const float4*>(base + k * HP + cc), h[cc], h[cc + 1], h[cc + 2], h[cc + 3]);
    }
  }
}

// Per-node values of one layer that the backward pass needs besides the layer's input and output rows
struct StackLayerKeep {
  float asrc, adst, m, inv;   // <h, att_src>, <h, att_dst>, max logit, 1 / (softmax denominator + 1e-16)
};

// One GATConv layer + activation of this thread's node, in place on x (layer input on entry, output on return), as
// torch_geometric's GATConv: h = x W^T, alpha = <h, att>, LeakyReLU(0.2) logits, max-subtracted softmax with the 1e-16
// denominator, messages alpha * h_src summed in edge-list order, + bias.  sh = [T][HP + 4] projected rows, sas = [T]
// alpha_src, sin / swt = the in-edge list and per-thread edge scratch (column tid), rows of the env from envbase.
// Every thread of the CTA must call it (block barriers); `sync_first`: the previous layer's rows may still be read.
template <int HP>
__device__ __forceinline__ StackLayerKeep stack_layer(const float* __restrict__ sw, int l, bool relu, float (&x)[HP],
                                                      float* sh, float* sas, const uint8_t* sin, float* swt, int tid,
                                                      int envbase, int deg, bool sync_first) {
  using SL = StackLayout<HP>;
  constexpr int kRow = HP + 4;
  constexpr int T = kTileThreads;
  const float* base = sw + SL::layer_off(l);
  const int cinp = l == 0 ? SL::kIn0 : HP;
  const float* vec = base + cinp * HP;
  float h[HP];
  stack_project<HP>(base, l, x, h);
  float asrc = 0.0f, adst = 0.0f;
#pragma unroll
  for (int cc = 0; cc < HP; ++cc) {
    asrc = __fadd_rn(asrc, __fmul_rn(h[cc], vec[cc]));
    adst = __fadd_rn(adst, __fmul_rn(h[cc], vec[HP + cc]));
  }
  if (sync_first) __syncthreads();                   // the previous layer's rows are no longer read
#pragma unroll
  for (int cc = 0; cc < HP; cc += 4)
    *reinterpret_cast<float4*>(sh + tid * kRow + cc) = make_float4(h[cc], h[cc + 1], h[cc + 2], h[cc + 3]);
  sas[tid] = asrc;
  __syncthreads();
  // softmax over the in-edges (max, denominator, messages), sources read from the env's rows
  const float* rows = sh + envbase * kRow;
  const float* as_env = sas + envbase;
  float m = -INFINITY;
  for (int e = 0; e < deg; ++e) m = fmaxf(m, gat_logit(as_env[sin[e * T]], adst));
  // unnormalised weights once (kept in the per-thread scratch column), one reciprocal, messages as fused
  // multiply-adds in edge-list order
  float den = 0.0f;
  for (int e = 0; e < deg; ++e) {
    const float we = expf(__fsub_rn(gat_logit(as_env[sin[e * T]], adst), m));
    swt[e * T] = we;
    den = __fadd_rn(den, we);
  }
  const float inv = __fdiv_rn(1.0f, __fadd_rn(den, 1e-16f));
#pragma unroll
  for (int cc = 0; cc < HP; ++cc) x[cc] = 0.0f;
  for (int e = 0; e < deg; ++e) {
    const float a = __fmul_rn(swt[e * T], inv);
    const float* hj = rows + sin[e * T] * kRow;
#pragma unroll
    for (int cc = 0; cc < HP; cc += 4)
      fma4_packed(a, *reinterpret_cast<const float4*>(hj + cc), x[cc], x[cc + 1], x[cc + 2], x[cc + 3]);
  }
#pragma unroll
  for (int cc = 0; cc < HP; ++cc) {
    const float v = __fadd_rn(x[cc], vec[2 * HP + cc]);
    x[cc] = relu ? fmaxf(v, 0.0f) : tanhf(v);        // padded channels: weights and bias are 0, tanh(0) = relu(0) = 0
  }
  return StackLayerKeep{asrc, adst, m, inv};
}

// head: r = ReLU(lin1 x), q = lin2 r (9 actions + 3 zero-padded columns) WITHOUT lin2.bias: the caller adds
// stack_lin2_bias(sw, L)[a] to q[a] (the evaluation kernel inside its argmax loop)
template <int HP>
__device__ __forceinline__ void stack_head(const float* __restrict__ sw, int L, const float (&x)[HP], float (&r)[HP],
                                           float (&q)[StackLayout<HP>::kW2Cols]) {
  using SL = StackLayout<HP>;
  const float* l1 = sw + SL::lin1_off(L);
#pragma unroll
  for (int cc = 0; cc < HP; ++cc) r[cc] = 0.0f;
#pragma unroll
  for (int k = 0; k < HP; ++k) {
#pragma unroll
    for (int cc = 0; cc < HP; cc += 4)
      fma4_packed(x[k], *reinterpret_cast<const float4*>(l1 + k * HP + cc), r[cc], r[cc + 1], r[cc + 2], r[cc + 3]);
  }
#pragma unroll
  for (int cc = 0; cc < HP; ++cc) r[cc] = fmaxf(__fadd_rn(r[cc], l1[HP * HP + cc]), 0.0f);
  const float* l2 = sw + SL::lin2_off(L);
#pragma unroll
  for (int a = 0; a < SL::kW2Cols; ++a) q[a] = 0.0f;
#pragma unroll
  for (int k = 0; k < HP; ++k) {
#pragma unroll
    for (int a = 0; a < SL::kW2Cols; a += 4)
      fma4_packed(r[k], *reinterpret_cast<const float4*>(l2 + k * SL::kW2Cols + a), q[a], q[a + 1], q[a + 2], q[a + 3]);
  }
}

template <int HP>
__device__ __forceinline__ const float* stack_lin2_bias(const float* sw, int L) {
  using SL = StackLayout<HP>;
  return sw + SL::lin2_off(L) + HP * SL::kW2Cols;
}

}  // namespace swarm
#endif
