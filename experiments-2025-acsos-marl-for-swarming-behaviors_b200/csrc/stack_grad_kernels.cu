// stack_grad_kernels.cu -- DQN update of stacked GAT Q-networks (train_step_dqn, train_gcn_dqn.py:112-137, for the
// conv1 .. convL form of data/models/experiment_Flocking-seed_*.pth): TD target, loss and the hand-written backward pass
// through the layer stack, then clip_grad_norm_ + Adam over the stack's packed weights.
//
// stack_grad_kernel keeps the env-tile scheme of gatstack_kernel (thread = node, CTA = up to floor(128 / N) sampled
// transitions) and runs the forward through the same device code (stack_device.cuh), so its Q values are the bits of
// swarm_gatstack_forward.  Per CTA: target network on s' (only max_a Q is kept), online network on s keeping each layer's
// input / output rows and, per node and layer, alpha_src, alpha_dst, the max logit and 1 / (den + 1e-16); the backward
// recomputes the softmax weights from those instead of storing one per edge.  Terms that flow to a SOURCE node are
// gathers: the target node writes the sum of its edges' attention weights into a per-env dense [i][j] matrix (parallel
// kNN edges add into the same cell), then thread j walks its column in ascending i.  Weight gradients are contractions
// over the CTA's node rows in a fixed order, written as per-CTA partials (count gradients + the sum of squared TD
// errors); stack_reduce_kernel sums them in CTA order.  No atomics: two calls give the same bits.
#include <cstring>

#include "dqn_common.cuh"
#include "stack_device.cuh"
#include "launchers.h"

namespace swarm {

struct StackGradParams {
  SwarmConfig cfg;
  SwarmStackSpec spec;
  const float* w_online;
  const float* w_target;
  SwarmReplay batch;
  const int64_t* indices;
  int32_t n_graphs;
  float gamma;
  float loss_scale;
  float* partials;            // [n_ctas][stride]
  float* td;
  int32_t epb, maxdeg, stride, count;
  float qmax_r;
  // device-driven tick (stack_grad_ctl_kernel): slots are drawn here from the ring fill after this tick's push
  const SwarmTrainCtl* ctl;
  int64_t* indices_out;       // [n_graphs] the drawn slots (exported for tests / logging)
  unsigned long long sample_seed;
  int32_t pushed_envs;        // transitions pushed by this tick's rollout
};

struct StackGradSmem {
  int w, st, x0, x, h, d, keep, nodes, inl, wt, kv, total;
};

// x = the layers' output rows X[1..L] (X[L] feeds the head), h / d = projected rows / gradient rows of the layer being
// differentiated, keep = [L][4][T] StackLayerKeep, nodes = [6][T] per-node scalars, wt = the forward's edge scratch and,
// in the backward pass, the per-env [i][j] attention-weight matrices
template <int HP>
__host__ __device__ inline StackGradSmem stack_grad_smem(int L, int maxdeg, int graph_mode) {
  constexpr int T = kTileThreads;
  constexpr int kRowB = (HP + 4) * 4 * T;
  StackGradSmem s;
  int off = 0;
  s.w = off;     off = tile_align16(off + StackLayout<HP>::total(L) * 4);
  s.st = off;    off = tile_align16(off + T * 16);
  s.x0 = off;    off = tile_align16(off + T * 8 * 4);
  s.x = off;     off = tile_align16(off + L * kRowB);
  s.h = off;     off = tile_align16(off + kRowB);
  s.d = off;     off = tile_align16(off + kRowB);
  s.keep = off;  off = tile_align16(off + L * 4 * T * 4);
  s.nodes = off; off = tile_align16(off + 6 * T * 4);
  s.inl = off;   off = tile_align16(off + maxdeg * T);
  s.wt = off;    off = tile_align16(off + maxdeg * T * 4);      // >= epb * N * N floats: maxdeg >= N, T >= epb * N
  s.kv = off;    off = tile_align16(off + (graph_mode == SWARM_GRAPH_KNN ? T * 4 : 0));
  s.total = off;
  return s;
}

// out[o] = sum over rows n (ascending) of a[n * lda] * b[n * ldb]  (a == nullptr: ones)
__device__ __forceinline__ float stack_contract(const float* a, int lda, const float* b, int ldb, int rows) {
  float acc = 0.0f;
  if (a) {
#pragma unroll 4
    for (int n = 0; n < rows; ++n) acc = __fmaf_rn(a[n * lda], b[n * ldb], acc);
  } else {
#pragma unroll 4
    for (int n = 0; n < rows; ++n) acc = __fadd_rn(acc, b[n * ldb]);
  }
  return acc;
}

template <int HP>
__device__ __forceinline__ void load_row(const float* tile, int row, float (&v)[HP]) {
  const float4* r = reinterpret_cast<const float4*>(tile + row * (HP + 4));
#pragma unroll
  for (int c4 = 0; c4 < HP / 4; ++c4) {
    const float4 q = r[c4];
    v[4 * c4] = q.x; v[4 * c4 + 1] = q.y; v[4 * c4 + 2] = q.z; v[4 * c4 + 3] = q.w;
  }
}
template <int HP>
__device__ __forceinline__ void store_row(float* tile, int row, const float (&v)[HP]) {
  float4* r = reinterpret_cast<float4*>(tile + row * (HP + 4));
#pragma unroll
  for (int c4 = 0; c4 < HP / 4; ++c4) r[c4] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
}
template <int HP>
__device__ __forceinline__ float dot_row(const float (&v)[HP], const float* row) {
  float acc = 0.0f;
#pragma unroll
  for (int c = 0; c < HP; ++c) acc = __fmaf_rn(v[c], row[c], acc);
  return acc;
}

// CTL: the gradient phase of swarm_train_tick_stack -- every CTA exits while the ring holds fewer than n_graphs slots,
// otherwise graph g takes a slot drawn from the ring fill (the draw of dqn_grad_tc_kernel).  A separate template value
// so that the stand-alone gradient kernel keeps its code instruction for instruction (the parameter block is taken by
// value for the same reason: through a reference the inlined body compiled to different code).
template <int HP, bool CTL>
__device__ __forceinline__ void stack_grad_body(const StackGradParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  using SL = StackLayout<HP>;
  constexpr int T = kTileThreads;
  constexpr int kRow = HP + 4;
  const SwarmConfig& c = p.cfg;
  const SwarmStackSpec& sp = p.spec;
  const int N = c.n_agents, K = c.knn_k, L = sp.n_layers, H = sp.hidden;
  const TileThread t = tile_thread(N, p.epb, p.n_graphs);
  const int tid = t.tid;
  if (CTL && train_ring_size(p.ctl, p.pushed_envs, p.batch.capacity) < p.n_graphs) return;   // not filled yet (train:113-115)
  const StackGradSmem S = stack_grad_smem<HP>(L, p.maxdeg, c.graph_mode);
  float* sw = reinterpret_cast<float*>(smem + S.w);
  float4* sst = reinterpret_cast<float4*>(smem + S.st);
  float* sx0 = reinterpret_cast<float*>(smem + S.x0);
  float* sx = reinterpret_cast<float*>(smem + S.x);
  float* sh = reinterpret_cast<float*>(smem + S.h);
  float* sd = reinterpret_cast<float*>(smem + S.d);
  StackLayerKeep* skeep = reinterpret_cast<StackLayerKeep*>(smem + S.keep);     // [L][T]
  float* snode = reinterpret_cast<float*>(smem + S.nodes);
  float* sas = snode;                  // alpha_src of the layer in flight (forward)
  float* sdot = snode + T;             // sum_e alpha_e d alpha_e of target node i
  float* sdt = snode + 2 * T;          // d alpha_dst
  float* sds = snode + 3 * T;          // d alpha_src
  float* sdq = snode + 4 * T;          // d Q(s, a) (one-hot over the actions)
  float* sred = snode + 5 * T;         // squared TD error
  float* smat = reinterpret_cast<float*>(smem + S.wt);
  TileGraphSmem g = {};
  g.sas = sas;
  g.sin = smem + S.inl;
  g.skv = reinterpret_cast<float*>(smem + S.kv);
  const uint8_t* sin = g.sin + tid;
  float* swt = smat + tid;
  const long long g0 = (long long)blockIdx.x * p.epb;
  const int rows = (int)((p.n_graphs - g0 < p.epb ? p.n_graphs - g0 : p.epb) * N);     // node rows of this CTA

  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s;
  int act = 0;
  float rew = 0.0f;
  if (t.active) {
    long long slot = t.env;
    if (CTL) {
      const uint64_t rnd = rng_draw(p.sample_seed, (uint64_t)t.env, (uint64_t)(p.ctl->tick + 1), 0x5A17u);
      slot = (long long)__umul64hi(rnd, (uint64_t)train_ring_size(p.ctl, p.pushed_envs, p.batch.capacity));
      if (p.indices_out && t.i == 0) p.indices_out[t.env] = slot;
    } else if (p.indices) {
      slot = p.indices[t.env];                            // caller-supplied: clamped into the ring, never out of bounds
      slot = slot < 0 ? 0 : (slot >= p.batch.capacity ? p.batch.capacity - 1 : slot);
    }
    const long long ri = slot * N + t.i;
    s = reinterpret_cast<const float4*>(p.batch.state)[ri];
    s2 = reinterpret_cast<const float4*>(p.batch.next_state)[ri];
    act = sanitize_action(p.batch.actions[ri]);
    rew = p.batch.rewards[ri];
  }

  // ---- target network on s' -> y = r + gamma * max_a Q_target(s')  (train:120-121) ------------------------------------
  // then the online network on s with the activations kept (train:119); the two passes share the weight block
  float y = 0.0f, delta = 0.0f;
  float rr[HP];                          // ReLU(lin1 x) of the online pass
  int deg = 0;                           // in-degree of the node in the online pass's graph (the list stays in smem)
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    const bool online = pass == 1;
    const float4 sp4 = online ? s : s2;
    if (online) __syncthreads();                          // the target pass no longer reads the weights / rows
    stack_stage_weights<HP>(sp, online ? p.w_online : p.w_target, sw, tid, T);
    sst[tid] = sp4;
    __syncthreads();
    deg = 0;
    if (c.graph_mode == SWARM_GRAPH_KNN) {
      uint64_t cache_rank = ~0ull, cache_nbr = 0;
      const uint64_t nbr = tile_knn_small(t, sst, sp4, N, K, cache_rank, cache_nbr);
      deg = tile_in_edges_knn_small(g, t, N, K, nbr, reinterpret_cast<uint32_t*>(g.skv));
    } else if (c.graph_mode == SWARM_GRAPH_RADIUS) {
      if (t.active) deg = tile_in_edges_radius(g, t, sst, sp4, N, p.qmax_r);
    } else if (t.active) {
      deg = tile_in_edges_complete(g, t, N);
    }
    float x[HP];
    stack_features<HP>(x, sp4, c, sp.in_features, t.i);
    if (online) {
      *reinterpret_cast<float4*>(sx0 + tid * 8) = make_float4(x[0], x[1], x[2], x[3]);
      *reinterpret_cast<float4*>(sx0 + tid * 8 + 4) = make_float4(x[4], x[5], x[6], x[7]);
    }
    for (int l = 0; l < L; ++l) {
      const StackLayerKeep k = stack_layer<HP>(sw, l, sp.activation[l] == 1, x, sh, sas, sin, swt, tid, t.envbase, deg, l > 0);
      if (online) {
        skeep[l * T + tid] = k;
        store_row<HP>(sx + l * kRow * T, tid, x);
      }
    }
    float q[SL::kW2Cols];
    stack_head<HP>(sw, L, x, rr, q);
    const float* b2 = stack_lin2_bias<HP>(sw, L);
#pragma unroll
    for (int a = 0; a < 9; ++a) q[a] = __fadd_rn(q[a], b2[a]);
    if (!online) {
      float qmax = q[0];
#pragma unroll
      for (int a = 1; a < 9; ++a) qmax = fmaxf(qmax, q[a]);
      y = __fadd_rn(rew, __fmul_rn(p.gamma, qmax));
    } else {
      float v = q[0];
#pragma unroll
      for (int a = 1; a < 9; ++a) v = (act == a) ? q[a] : v;        // values = Q(s).gather(1, a)  (train:119)
      delta = v;
    }
  }

  // ---- TD error, d loss / d Q(s, a) = 2 loss_scale (values - targets)  (nn.MSELoss with loss_scale = 1 / (G N)) --------
  float dq = 0.0f;
  if (t.active) {
    delta = __fsub_rn(delta, y);
    dq = __fmul_rn(__fmul_rn(2.0f, p.loss_scale), delta);
    if (p.td) p.td[t.gidx] = delta;
  } else {
    delta = 0.0f;
  }
  sred[tid] = __fmul_rn(delta, delta);

  // ---- head backward: lin2 -> ReLU -> lin1 ------------------------------------------------------------------------
  float dy[HP];                           // d loss / d (output of the layer being differentiated)
  {
    const float* l1 = sw + SL::lin1_off(L);
    const float* l2 = sw + SL::lin2_off(L);
    float dp[HP];
#pragma unroll
    for (int k = 0; k < HP; ++k) dp[k] = rr[k] > 0.0f ? __fmul_rn(l2[k * SL::kW2Cols + act], dq) : 0.0f;
#pragma unroll
    for (int k = 0; k < HP; ++k) dy[k] = dot_row<HP>(dp, l1 + k * HP);     // W1^T dp
    __syncthreads();                      // the online pass no longer reads sh
    store_row<HP>(sh, tid, rr);
    store_row<HP>(sd, tid, dp);
    sdq[tid] = dq;
    reinterpret_cast<int*>(sds)[tid] = act;
    __syncthreads();
    float* out = p.partials + (long long)blockIdx.x * p.stride;
    const float* xl = sx + (L - 1) * kRow * T;
    const int off = p.count - (H * H + H + 9 * H + 9);
    const int* sacts = reinterpret_cast<const int*>(sds);
    for (int o = tid; o < H * H + H + 9 * H + 9; o += T) {
      float v;
      if (o < H * H) {                                  // d lin1.weight[c][k] = sum_n dp_n[c] X_L[n][k]
        v = stack_contract(sd + o / H, kRow, xl + o % H, kRow, rows);
      } else if (o < H * H + H) {                       // d lin1.bias[c] = sum_n dp_n[c]
        v = stack_contract(nullptr, 0, sd + (o - H * H), kRow, rows);
      } else if (o < H * H + H + 9 * H) {               // d lin2.weight[a][k] = sum_n [a_n = a] dq_n r_n[k]
        const int a = (o - H * H - H) / H, k = (o - H * H - H) % H;
        float acc = 0.0f;
        for (int n = 0; n < rows; ++n) acc = __fmaf_rn(sacts[n] == a ? sdq[n] : 0.0f, sh[n * kRow + k], acc);
        v = acc;
      } else {                                          // d lin2.bias[a] = sum_n [a_n = a] dq_n
        const int a = o - H * H - H - 9 * H;
        float acc = 0.0f;
        for (int n = 0; n < rows; ++n) acc = __fadd_rn(acc, sacts[n] == a ? sdq[n] : 0.0f);
        v = acc;
      }
      out[off + o] = v;
    }
  }

  // ---- layers, top to bottom: activation', bias, attention, projection -------------------------------------------------
  float* out = p.partials + (long long)blockIdx.x * p.stride;
  int loff[kStackMaxLayers];
  {
    int goff = 0;
    for (int l = 0; l < L; ++l) {
      loff[l] = goff;
      goff += 3 * H + H * (l == 0 ? sp.in_features : H);
    }
  }
  for (int l = L - 1; l >= 0; --l) {
    const float* base = sw + SL::layer_off(l);
    const float* vec = base + (l == 0 ? SL::kIn0 : HP) * HP;
    const bool relu = sp.activation[l] == 1;
    const int cin = l == 0 ? sp.in_features : H;
    const StackLayerKeep kp = skeep[l * T + tid];
    const StackLayerKeep* kenv = skeep + l * T + t.envbase;
    float dout[HP], h[HP];
    {
      float yv[HP], xin[HP];
      load_row<HP>(sx + l * kRow * T, tid, yv);
#pragma unroll
      for (int cc = 0; cc < HP; ++cc)     // tanh' = 1 - y^2, relu' = [y > 0] (torch's tanh_backward / threshold_backward)
        dout[cc] = relu ? (yv[cc] > 0.0f ? dy[cc] : 0.0f) : __fmul_rn(dy[cc], __fsub_rn(1.0f, __fmul_rn(yv[cc], yv[cc])));
#pragma unroll
      for (int kk = 0; kk < HP; ++kk) xin[kk] = 0.0f;
      if (l == 0) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) xin[kk] = sx0[tid * 8 + kk];
      } else {
        load_row<HP>(sx + (l - 1) * kRow * T, tid, xin);
      }
      stack_project<HP>(base, l, xin, h);              // the forward's h, bit for bit
    }
    __syncthreads();                                     // previous readers of sh / sd / the matrices are done
    store_row<HP>(sh, tid, h);
    store_row<HP>(sd, tid, dout);
    __syncthreads();
    // d bias[c] = sum_n dout_n[c]
    for (int cc = tid; cc < H; cc += T) out[loff[l] + 2 * H + cc] = stack_contract(nullptr, 0, sd + cc, kRow, rows);
    // target role (node i): alpha_e recomputed as the forward formed it, d alpha_e = <dout_i, h_j>, softmax backward
    // d z_e = alpha_e (d alpha_e - sum_e' alpha_e' d alpha_e'), LeakyReLU backward -> d alpha_dst_i; the edge's attention
    // weight is added into A[i][j]
    if (t.active) {
      float* arow = smat + (t.el * N + t.i) * N;
      for (int j = 0; j < N; ++j) arow[j] = 0.0f;
      const float* hrows = sh + t.envbase * kRow;
      float dot = 0.0f;
      for (int e = 0; e < deg; ++e) {
        const int j = sin[e * T];
        const float a = __fmul_rn(expf(__fsub_rn(gat_logit(kenv[j].asrc, kp.adst), kp.m)), kp.inv);
        dot = __fmaf_rn(a, dot_row<HP>(dout, hrows + j * kRow), dot);
        arow[j] = __fadd_rn(arow[j], a);
      }
      float dt_i = 0.0f;
      for (int e = 0; e < deg; ++e) {
        const int j = sin[e * T];
        const float z = __fadd_rn(kenv[j].asrc, kp.adst);
        const float a = __fmul_rn(expf(__fsub_rn(z > 0.0f ? z : __fmul_rn(z, 0.2f), kp.m)), kp.inv);
        const float dz = __fmul_rn(a, __fsub_rn(dot_row<HP>(dout, hrows + j * kRow), dot));
        dt_i = __fadd_rn(dt_i, z > 0.0f ? dz : __fmul_rn(dz, 0.2f));
      }
      sdot[tid] = dot;
      sdt[tid] = dt_i;
    } else {
      sdot[tid] = 0.0f;
      sdt[tid] = 0.0f;
    }
    __syncthreads();
    // source role (node j): d h_j = sum_i A[i][j] dout_i + ds_j att_src + dt_j att_dst, with
    // ds_j = sum_i A[i][j] (<dout_i, h_j> - dot_i) LeakyReLU'(z_ij), column j in ascending i
    float dh[HP];
#pragma unroll
    for (int cc = 0; cc < HP; ++cc) dh[cc] = 0.0f;
    float ds_j = 0.0f;
    if (t.active) {
      const float* acol = smat + t.el * N * N + t.i;
      for (int ii = 0; ii < N; ++ii) {
        const float a = acol[ii * N];
        if (a == 0.0f) continue;
        const float* di = sd + (t.envbase + ii) * kRow;
        const float z = __fadd_rn(kp.asrc, kenv[ii].adst);
        const float dz = __fmul_rn(a, __fsub_rn(dot_row<HP>(h, di), sdot[t.envbase + ii]));
        ds_j = __fadd_rn(ds_j, z > 0.0f ? dz : __fmul_rn(dz, 0.2f));
#pragma unroll
        for (int cc = 0; cc < HP; ++cc) dh[cc] = __fmaf_rn(a, di[cc], dh[cc]);
      }
      const float dt_j = sdt[tid];
#pragma unroll
      for (int cc = 0; cc < HP; ++cc) dh[cc] = __fmaf_rn(ds_j, vec[cc], __fmaf_rn(dt_j, vec[HP + cc], dh[cc]));
    }
    __syncthreads();                                     // dout rows no longer read
    store_row<HP>(sd, tid, dh);
    sds[tid] = ds_j;
    __syncthreads();
    // d att_src[c] = sum_n ds_n h_n[c], d att_dst[c] = sum_n dt_n h_n[c], d lin.weight[c][k] = sum_n dh_n[c] x_n[k]
    const float* xl = l == 0 ? sx0 : sx + (l - 1) * kRow * T;
    const int ldx = l == 0 ? 8 : kRow;
    for (int o = tid; o < 2 * H + H * cin; o += T) {
      float v;
      if (o < H) v = stack_contract(sds, 1, sh + o, kRow, rows);
      else if (o < 2 * H) v = stack_contract(sdt, 1, sh + (o - H), kRow, rows);
      else {
        const int cc = (o - 2 * H) / cin, kk = (o - 2 * H) % cin;
        v = stack_contract(sd + cc, kRow, xl + kk, ldx, rows);
      }
      out[loff[l] + (o < 2 * H ? o : o + H)] = v;
    }
    // d x = W^T d h for the layer below
    if (l > 0) {
#pragma unroll
      for (int kk = 0; kk < HP; ++kk) dy[kk] = dot_row<HP>(dh, base + kk * HP);
    }
  }
  if (tid == 0) {
    float sse = 0.0f;
    for (int n = 0; n < rows; ++n) sse = __fadd_rn(sse, sred[n]);
    out[p.count] = sse;
  }
}

template <int HP>
__global__ void __launch_bounds__(kTileThreads) stack_grad_kernel(const __grid_constant__ StackGradParams p) {
  stack_grad_body<HP, false>(p);
}

// width 8: a 96-register budget (five CTAs per SM, more than the Flocking shape's shared memory allows) -- with ptxas's
// own choice of 72 the sampling prologue spilled 24 bytes
template <int HP>
__global__ void __launch_bounds__(kTileThreads, HP == 8 ? 5 : 0) stack_grad_ctl_kernel(const __grid_constant__ StackGradParams p) {
  stack_grad_body<HP, true>(p);
}

// sum over CTAs (in CTA order) of partials[cta][o]
__device__ __forceinline__ float stack_partial_sum(const float* __restrict__ partials, int n_ctas, int stride, int o) {
  float acc = 0.0f;
  for (int b = 0; b < n_ctas; ++b) acc = __fadd_rn(acc, partials[(long long)b * stride + o]);
  return acc;
}

// grad[o] = the CTA-order sum of the partials; loss = loss_scale * sum of squared TD errors
__device__ __forceinline__ void stack_reduce_element(const float* __restrict__ partials, int n_ctas, int stride, int count,
                                                     float loss_scale, float* __restrict__ grad, float* __restrict__ loss,
                                                     int o) {
  if (o > count) return;
  const float acc = stack_partial_sum(partials, n_ctas, stride, o);
  if (o < count) grad[o] = acc;
  else loss[0] = __fmul_rn(acc, loss_scale);
}

__global__ void __launch_bounds__(256) stack_reduce_kernel(const float* __restrict__ partials, int n_ctas, int stride,
                                                           int count, float loss_scale, float* __restrict__ grad,
                                                           float* __restrict__ loss) {
  stack_reduce_element(partials, n_ctas, stride, count, loss_scale, grad, loss, blockIdx.x * blockDim.x + threadIdx.x);
}

// device-driven tick: publishes whether this tick updates (read by the clip + Adam kernel) and leaves grad / loss
// untouched when it does not (as dqn_reduce_kernel).
// PEERS: the data-parallel tick -- the one-shot PUSH all-reduce of reduce_clip_adam_kernel<true> (dqn_kernels.cu) over
// NVLink peer memory, one gradient element per thread after the CTA-order sum: the thread writes its word
// (epoch = tick + 1 << 32 | float bits) into slot [parity of the epoch][own rank][o] of every rank's buffer, own buffer
// first, then in ring order; polls its own buffer's [parity][r][o] for every rank r; and sums the ranks in rank order,
// so every rank holds the same bits.  Every rank agrees on `upd` (equal shards, same ring fill), so either all ranks
// exchange this tick or none does.  A separate template value so that the one-GPU kernel keeps its code.
template <bool PEERS>
__device__ __forceinline__ void stack_reduce_ctl_body(const float* __restrict__ partials, int n_ctas, int stride, int count,
                                                      float loss_scale, float* __restrict__ grad, float* __restrict__ loss,
                                                      SwarmTrainCtl* __restrict__ ctl, int pushed_envs, long long capacity,
                                                      int n_graphs, const SwarmPeerExchange* peers) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  const bool upd = train_ring_size(ctl, pushed_envs, capacity) >= n_graphs;
  if (o == 0) ctl->updating = upd ? 1 : 0;
  if (!upd) return;
  if (!PEERS) {
    stack_reduce_element(partials, n_ctas, stride, count, loss_scale, grad, loss, o);
    return;
  }
  if (o > count) return;
  float g = stack_partial_sum(partials, n_ctas, stride, o);
  if (o == count) g = __fmul_rn(g, loss_scale);
  const uint32_t epoch = (uint32_t)(ctl->tick + 1);
  const int W = peers->world_size, rank = peers->rank;
  const size_t par_base = (size_t)(epoch & 1u) * W * SWARM_XCHG_STACK_STRIDE;
  const uint64_t word = ((uint64_t)epoch << 32) | (uint64_t)__float_as_uint(g);
  for (int q = 0; q < W; ++q) {
    const int peer = (rank + q) % W;                      // own buffer first, then ring order: spreads the links
    st_relaxed_sys_u64(peers->data[peer] + par_base + (size_t)rank * SWARM_XCHG_STACK_STRIDE + o, word);
  }
  const uint64_t* mine = peers->data[rank] + par_base + o;
  uint64_t got[SWARM_MAX_PEERS];
  bool ok = false;
  for (long long it = 0; it < (1ll << 26) && !ok; ++it) {      // bounded: a lost peer traps instead of hanging
    ok = true;
#pragma unroll
    for (int r = 0; r < SWARM_MAX_PEERS; ++r)
      got[r] = (r < W) ? ld_relaxed_sys_u64(mine + (size_t)r * SWARM_XCHG_STACK_STRIDE) : ((uint64_t)epoch << 32);
#pragma unroll
    for (int r = 0; r < SWARM_MAX_PEERS; ++r) ok = ok && ((uint32_t)(got[r] >> 32) == epoch);
  }
  if (!ok) __trap();
  g = 0.0f;
#pragma unroll
  for (int r = 0; r < SWARM_MAX_PEERS; ++r)
    if (r < W) g = __fadd_rn(g, __uint_as_float((uint32_t)got[r]));     // rank order
  if (o < count) grad[o] = g;
  else loss[0] = g;
}

__global__ void __launch_bounds__(256) stack_reduce_ctl_kernel(const float* __restrict__ partials, int n_ctas, int stride,
                                                               int count, float loss_scale, float* __restrict__ grad,
                                                               float* __restrict__ loss, SwarmTrainCtl* __restrict__ ctl,
                                                               int pushed_envs, long long capacity, int n_graphs) {
  stack_reduce_ctl_body<false>(partials, n_ctas, stride, count, loss_scale, grad, loss, ctl, pushed_envs, capacity,
                               n_graphs, nullptr);
}

__global__ void __launch_bounds__(256) stack_reduce_peers_kernel(const float* __restrict__ partials, int n_ctas, int stride,
                                                                 int count, float loss_scale, float* __restrict__ grad,
                                                                 float* __restrict__ loss, SwarmTrainCtl* __restrict__ ctl,
                                                                 int pushed_envs, long long capacity, int n_graphs,
                                                                 const __grid_constant__ SwarmPeerExchange peers) {
  stack_reduce_ctl_body<true>(partials, n_ctas, stride, count, loss_scale, grad, loss, ctl, pushed_envs, capacity,
                              n_graphs, &peers);
}

// ---- launchers -------------------------------------------------------------------------------------------------------
static int stack_hp(const SwarmStackSpec& s) { return s.hidden <= 8 ? 8 : (s.hidden <= 16 ? 16 : 32); }

int stack_grad_maxdeg(const SwarmConfig& c) {
  return c.graph_mode == SWARM_GRAPH_KNN ? (c.n_agents + c.knn_k + 1) : c.n_agents;
}

int stack_grad_smem_bytes(const SwarmConfig& c, const SwarmStackSpec& s) {
  const int maxdeg = stack_grad_maxdeg(c);
  switch (stack_hp(s)) {
    case 8: return stack_grad_smem<8>(s.n_layers, maxdeg, c.graph_mode).total;
    case 16: return stack_grad_smem<16>(s.n_layers, maxdeg, c.graph_mode).total;
    default: return stack_grad_smem<32>(s.n_layers, maxdeg, c.graph_mode).total;
  }
}

// graphs per CTA: up to floor(128 / N), fewer for small batches so that the update spreads over the SMs (as dqn_epb)
static int stack_grad_epb(const SwarmConfig& c, int n_graphs) {
  const int full = kTileThreads / c.n_agents;
  int epb = (n_graphs + 147) / 148;
  if (epb < 1) epb = 1;
  return epb < full ? epb : full;
}

static int stack_grad_stride(const SwarmStackSpec& s) { return (stack_weight_count(s) + 1 + 3) & ~3; }

long long stack_grad_workspace_bytes(const SwarmConfig& c, const SwarmStackSpec& s, int n_graphs) {
  const int epb = stack_grad_epb(c, n_graphs);
  const long long ctas = (n_graphs + epb - 1) / epb;
  return ctas * stack_grad_stride(s) * 4 + 256;
}

template <int HP>
static cudaError_t launch_stack_grad_hp(const StackGradParams& p, int ctas, cudaStream_t stream) {
  const int smem = stack_grad_smem<HP>(p.spec.n_layers, p.maxdeg, p.cfg.graph_mode).total;
  auto* kernel = p.ctl ? stack_grad_ctl_kernel<HP> : stack_grad_kernel<HP>;
  cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (err != cudaSuccess) return err;
  kernel<<<ctas, kTileThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_stack_grad(const SwarmConfig& c, const SwarmStackSpec& spec, const float* w_online, const float* w_target,
                              const SwarmReplay& batch, const int64_t* indices, int n_graphs, float gamma, float loss_scale,
                              float* grad, float* loss, float* td, void* workspace, cudaStream_t stream,
                              SwarmTrainCtl* ctl, int64_t* indices_out, unsigned long long sample_seed, int pushed_envs,
                              const SwarmPeerExchange* peers) {
  StackGradParams p;
  std::memset(&p, 0, sizeof(p));
  p.ctl = ctl;
  p.indices_out = indices_out;
  p.sample_seed = sample_seed;
  p.pushed_envs = pushed_envs;
  p.cfg = c;
  p.spec = spec;
  p.w_online = w_online;
  p.w_target = w_target;
  p.batch = batch;
  p.indices = indices;
  p.n_graphs = n_graphs;
  p.gamma = gamma;
  p.loss_scale = loss_scale;
  p.partials = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  p.td = td;
  p.epb = stack_grad_epb(c, n_graphs);
  p.maxdeg = stack_grad_maxdeg(c);
  p.stride = stack_grad_stride(spec);
  p.count = stack_weight_count(spec);
  p.qmax_r = c.graph_mode == SWARM_GRAPH_RADIUS ? sq_threshold(c.graph_radius) : 0.0f;
  const int ctas = (n_graphs + p.epb - 1) / p.epb;
  cudaError_t err;
  switch (stack_hp(spec)) {
    case 8: err = launch_stack_grad_hp<8>(p, ctas, stream); break;
    case 16: err = launch_stack_grad_hp<16>(p, ctas, stream); break;
    default: err = launch_stack_grad_hp<32>(p, ctas, stream); break;
  }
  if (err != cudaSuccess) return err;
  const int blocks = (p.count + 1 + 255) / 256;
  if (ctl && peers)
    stack_reduce_peers_kernel<<<blocks, 256, 0, stream>>>(p.partials, ctas, p.stride, p.count, loss_scale, grad, loss, ctl,
                                                          pushed_envs, batch.capacity, n_graphs, *peers);
  else if (ctl)
    stack_reduce_ctl_kernel<<<blocks, 256, 0, stream>>>(p.partials, ctas, p.stride, p.count, loss_scale, grad, loss, ctl,
                                                        pushed_envs, batch.capacity, n_graphs);
  else
    stack_reduce_kernel<<<blocks, 256, 0, stream>>>(p.partials, ctas, p.stride, p.count, loss_scale, grad, loss);
  return cudaGetLastError();
}

// ---- clip_grad_norm_ + Adam over a stack's packed weights, one CTA -------------------------------------------------------
// The per-tensor norms are taken over the state-dict tensors in packed order (StackedGCN.parameters() order), with the
// sums of adam_clip_kernel: per tensor a double sum of squares (per warp, then the eight warps in order), its float norm,
// then the double sum of the squared norms in tensor order; Adam op for op as torch.optim.Adam (adam_element).
constexpr int kStackAdamPer = 20;                        // 256 x 20 >= 5 033, the largest stack (L = 4, H = 32, 7 inputs)
constexpr int kStackMaxTensors = 4 * kStackMaxLayers + 4;

struct StackAdamParams {
  float* w;
  const float* grad;
  float* m;
  float* v;
  float* target;
  float* grad_norm;
  int32_t count, n_tensors;
  int32_t seg[kStackMaxTensors + 1];
  AdamScalars sc;
  float max_norm;
  // device-driven tick (stack_adam_clip_ctl_kernel): the step-dependent scalars come from *ctl on the device and the
  // cursor is advanced at the end
  SwarmTrainCtl* ctl;
  double lr, beta1, beta2;
  long long ring_capacity;
  int32_t num_envs;
  int32_t update_target_every;
};

// CTL: the last launch of swarm_train_tick_stack, as adam_clip_kernel<false> with a cursor (dqn_kernels.cu): bias
// corrections from ctl->opt_step + 1, target sync when (ctl->tick + 1) % update_target_every == 0, no update while
// ctl->updating == 0, then the cursor advances.  A separate template value so that the stand-alone kernel keeps its code
// instruction for instruction (tid is read in the kernel, where the compiler knows it is below 256).
template <bool CTL>
__device__ __forceinline__ void stack_adam_clip_body(const StackAdamParams p, const int tid) {
  __shared__ double swarp[kStackMaxTensors][8];
  __shared__ float s_coef;
  __shared__ float s_neg_step, s_bc2_sqrt;
  __shared__ int s_update, s_sync;
  const int lane = tid & 31, warp = tid >> 5;
  float g_[kStackAdamPer];
#pragma unroll
  for (int i = 0; i < kStackAdamPer; ++i) {
    const int o = tid + 256 * i;
    g_[i] = o < p.count ? p.grad[o] : 0.0f;
  }
  if (CTL && tid == 255) {
    // step-dependent scalars from the device cursor (after this warp's loads went out: the two pow chains run under
    // their latency)
    const long long step = p.ctl->opt_step + 1;
    const double bc1 = 1.0 - pow(p.beta1, (double)step);
    const double bc2 = 1.0 - pow(p.beta2, (double)step);
    s_neg_step = (float)(-(p.lr / bc1));
    s_bc2_sqrt = (float)sqrt(bc2);
    s_update = p.ctl->updating;
    s_sync = ((p.ctl->tick + 1) % p.update_target_every) == 0;
  }
  for (int sgi = 0; sgi < p.n_tensors; ++sgi) {
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < kStackAdamPer; ++i) {
      const int o = tid + 256 * i;
      if (o >= p.seg[sgi] && o < p.seg[sgi + 1]) acc += (double)g_[i] * (double)g_[i];
    }
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, sh);
    if (lane == 0) swarp[sgi][warp] = acc;
  }
  __syncthreads();
  AdamScalars sc = p.sc;
  float* target = p.target;
  if (CTL) {
    if (!s_update) {
      if (tid == 0) train_ctl_advance(p.ctl, p.num_envs, p.ring_capacity, false);
      return;
    }
    sc.neg_step_size = s_neg_step;
    sc.bc2_sqrt = s_bc2_sqrt;
    if (!s_sync) target = nullptr;
  }
  if (tid == 0) {
    double tot = 0.0;
    for (int sgi = 0; sgi < p.n_tensors; ++sgi) {
      double ss = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) ss += swarp[sgi][w];
      const float nrm = (float)sqrt(ss);
      tot += (double)nrm * (double)nrm;
    }
    const float total_norm = (float)sqrt(tot);
    float coef = 1.0f;
    if (p.max_norm > 0.0f) {
      coef = p.max_norm / (total_norm + 1e-6f);
      coef = coef > 1.0f ? 1.0f : coef;
    }
    s_coef = coef;
    if (p.grad_norm) p.grad_norm[0] = total_norm;
  }
  __syncthreads();
  const float coef = s_coef;
#pragma unroll
  for (int i = 0; i < kStackAdamPer; ++i) {
    const int o = tid + 256 * i;
    if (o >= p.count) break;
    float m = p.m[o], v = p.v[o], w = p.w[o];
    adam_element(sc, g_[i], coef, m, v, w);
    p.m[o] = m;
    p.v[o] = v;
    p.w[o] = w;
    if (target) target[o] = w;
  }
  if (CTL && tid == 0) train_ctl_advance(p.ctl, p.num_envs, p.ring_capacity, true);
}

__global__ void __launch_bounds__(256) stack_adam_clip_kernel(const __grid_constant__ StackAdamParams p) {
  stack_adam_clip_body<false>(p, threadIdx.x);
}

__global__ void __launch_bounds__(256) stack_adam_clip_ctl_kernel(const __grid_constant__ StackAdamParams p) {
  stack_adam_clip_body<true>(p, threadIdx.x);
}

cudaError_t launch_stack_adam_clip(const SwarmStackSpec& spec, float* w, const float* grad, float* m, float* v,
                                   long long step, double lr, double beta1, double beta2, double eps, double max_norm,
                                   float* target, float* grad_norm, cudaStream_t stream, SwarmTrainCtl* ctl,
                                   int num_envs, long long ring_capacity, int update_target_every) {
  StackAdamParams p;
  std::memset(&p, 0, sizeof(p));
  p.ctl = ctl;
  p.lr = lr;
  p.beta1 = beta1;
  p.beta2 = beta2;
  p.ring_capacity = ring_capacity;
  p.num_envs = num_envs;
  p.update_target_every = update_target_every > 0 ? update_target_every : 1;
  p.w = w;
  p.grad = grad;
  p.m = m;
  p.v = v;
  p.target = target;
  p.grad_norm = grad_norm;
  p.count = stack_weight_count(spec);
  const int H = spec.hidden;
  int off = 0, n = 0;
  for (int l = 0; l < spec.n_layers; ++l) {
    const int sizes[4] = {H, H, H, H * (l == 0 ? spec.in_features : H)};     // att_src, att_dst, bias, lin.weight
    for (int k = 0; k < 4; ++k) { p.seg[n++] = off; off += sizes[k]; }
  }
  const int head[4] = {H * H, H, 9 * H, 9};                                    // lin1.weight, lin1.bias, lin2.weight, lin2.bias
  for (int k = 0; k < 4; ++k) { p.seg[n++] = off; off += head[k]; }
  p.seg[n] = off;
  p.n_tensors = n;
  // scalars exactly as torch.optim.Adam computes them (Python doubles, cast to float where they meet tensors)
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  p.sc.lerp_w = (float)(1.0 - beta1);
  p.sc.beta2 = (float)beta2;
  p.sc.one_minus_beta2 = (float)(1.0 - beta2);
  p.sc.neg_step_size = (float)(-(lr / bc1));
  p.sc.bc2_sqrt = (float)sqrt(bc2);
  p.sc.eps = (float)eps;
  p.max_norm = (float)max_norm;
  if (ctl) stack_adam_clip_ctl_kernel<<<1, 256, 0, stream>>>(p);
  else stack_adam_clip_kernel<<<1, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace swarm
