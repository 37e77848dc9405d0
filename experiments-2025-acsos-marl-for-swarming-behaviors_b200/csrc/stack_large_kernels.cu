// stack_large_kernels.cu -- multi-layer GAT Q-networks on large swarms (any N, built for 128 < N <= 4096): the whole
// stacked forward
//     node features -> per-env graph -> L x [GATConv -> activation] -> lin1 -> ReLU -> lin2 -> argmax
// in ONE launch with ONE CTA per env, for every SwarmStackSpec.  gatstack_kernel (stack_kernels.cu) keeps a whole env in
// a 128-thread tile; here an env no longer fits, so
//   * the attention runs in input space, per layer.  The projection has no bias, so with layer input rows x
//         sum_e alpha_e h_src(e) = W (sum_e alpha_e x_src(e))      and      <h_j, att> = <x_j, W^T att>:
//     per node two dot products with the pre-multiplied attention vectors, a softmax-weighted mean of its sources'
//     input rows (8 padded input features for conv1, HP for the others), then ONE projection (the mathematics of the
//     one-layer gatq_large_x_kernel / gatq_large_sorted_kernel, grid_kernels.cu, applied to every layer; float32-level
//     different rounding from torch_geometric's op order);
//   * the layer rows live in a caller workspace in global memory, double-buffered across layers ([2][B][N][HP] floats:
//     64 MB for the width-8 Flocking checkpoints at 1 024 envs x 1 024 agents, so they stay in the 126 MB L2);
//   * the graph is built once per forward and reused by every layer (positions do not change between layers):
//       radius    the uniform grid of grid_device.cuh (3 x 3 cell walk, exact squared-distance membership);
//       complete  the O(N log N) sorted-prefix factorisation of gatq_large_sorted_kernel, generalised from its six
//                 weighted quantities to 1 + (input width): per layer the sources are sorted by that layer's alpha_src;
//       kNN       the caller's torch.topk-exact table (swarm_graph_build), transposed once per forward into in-edge
//                 lists (workspace, sorted by row: deterministic sums) as gatq_knn_large_x_kernel does.
// The head (lin1 -> ReLU -> lin2) and the weight staging are stack_device.cuh's.
#include <cstring>

#include "grid_device.cuh"
#include "stack_device.cuh"
#include "launchers.h"

namespace swarm {

struct StackLargeParams {
  SwarmConfig cfg;
  SwarmStackSpec spec;
  const float* weights;
  const float4* state;
  const int32_t* nbr;        // kNN: [B][N][K]
  float* q_out;              // [B*N][9] or nullptr
  int32_t* act_out;          // [B*N] or nullptr
  float* rows;               // [2][B][N][HP] layer rows
  uint16_t* rev;             // kNN: [B][N*K] in-edge lists from other rows
  float qmax_r;
  int32_t sshift;            // complete graph: scans kept every (1 << sshift) sorted positions
};

// complete graph: scans kept every 2^s-th sorted position, s >= 2 chosen so that at most 258 positions are stored
__host__ __device__ inline int stack_large_sshift(int N) {
  int s = 2;
  while ((N >> s) > 256) ++s;
  return s;
}

struct StackLargeSmem {
  int w, v, as, ad, red, hold, pos, keys, cells, perm, sorted, pre, suf, roff, rcur, total;
};

template <int HP>
__host__ __device__ inline StackLargeSmem stack_large_smem(int L, int N, int graph_mode) {
  constexpr int Q = HP + 1;                          // weighted quantities of the complete graph: 1, x[0 .. HP)
  StackLargeSmem s = {};
  const int P = grid_pow2(N);
  int off = 0;
  s.w = off;     off = tile_align16(off + StackLayout<HP>::total(L) * 4);
  s.v = off;     off = tile_align16(off + 2 * HP * 4);
  s.as = off;    off = tile_align16(off + N * 4);
  s.ad = off;    off = tile_align16(off + N * 4);
  s.red = off;   off = tile_align16(off + 64 * 4);
  if (graph_mode == SWARM_GRAPH_RADIUS) {
    s.pos = off;   off = tile_align16(off + N * 8);
    s.keys = off;  off = tile_align16(off + P * 4);
    s.cells = off; off = tile_align16(off + kGridCells * 4);
  } else if (graph_mode == SWARM_GRAPH_KNN) {
    s.roff = off;  off = tile_align16(off + (N + 1) * 4);
    s.rcur = off;  off = tile_align16(off + (N + 1) * 4);
  } else {
    const int NC = (N >> stack_large_sshift(N)) + 2;
    s.hold = off;   off = tile_align16(off + Q * 4);
    s.keys = off;   off = tile_align16(off + P * 4);
    s.perm = off;   off = tile_align16(off + P * 2);
    s.sorted = off; off = tile_align16(off + N * 4);
    s.pre = off;    off = tile_align16(off + NC * Q * 4);
    s.suf = off;    off = tile_align16(off + NC * Q * 4);
  }
  s.total = off;
  return s;
}

// exclusive prefix sum of cnt[0 .. N) into off[0 .. N], every thread of the CTA calls it (gatq_knn_large_x_kernel's scan)
__device__ __forceinline__ void block_exclusive_scan(const int* cnt, int* off, int N, int* warp_tot) {
  const int tid = threadIdx.x;
  const int per = (N + kGridThreads - 1) / kGridThreads;
  const int b0 = tid * per;
  int local = 0;
  for (int k = 0; k < per; ++k) local += (b0 + k < N) ? cnt[b0 + k] : 0;
  int incl = local;
#pragma unroll
  for (int sft = 1; sft < 32; sft <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, sft);
    if ((tid & 31) >= sft) incl += v;
  }
  if ((tid & 31) == 31) warp_tot[tid >> 5] = incl;
  __syncthreads();
  int base = 0;
  for (int w = 0; w < (tid >> 5); ++w) base += warp_tot[w];
  int run = base + incl - local;
  for (int k = 0; k < per; ++k) {
    if (b0 + k < N) {
      const int c = cnt[b0 + k];
      off[b0 + k] = run;
      run += c;
    }
  }
  if (tid == kGridThreads - 1) off[N] = base + incl;
  __syncthreads();
}

// one row of CP floats (CP a multiple of 4) from global memory
template <int CP>
__device__ __forceinline__ void load_row(const float* __restrict__ r, float (&x)[CP]) {
#pragma unroll
  for (int c = 0; c < CP; c += 4) {
    const float4 v = *reinterpret_cast<const float4*>(r + c);
    x[c] = v.x; x[c + 1] = v.y; x[c + 2] = v.z; x[c + 3] = v.w;
  }
}

template <int CP>
__device__ __forceinline__ void acc_row(float w, const float* __restrict__ r, float (&acc)[CP]) {
#pragma unroll
  for (int c = 0; c < CP; c += 4) {
    const float4 v = *reinterpret_cast<const float4*>(r + c);
    fma4_packed(w, v, acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
  }
}

// One GATConv layer (+ activation) of every node of the env, CP = padded input width (8 for conv1, HP after); the last
// layer runs the head and writes Q / actions instead of a row.  Block barriers inside; ends with one.
template <int HP, int CP>
__device__ __forceinline__ void stack_large_layer(const StackLargeParams& p, unsigned char* smem, const StackLargeSmem& S,
                                                  int l, const CellGrid& grid, const float* __restrict__ xin,
                                                  float* __restrict__ xout) {
  using SL = StackLayout<HP>;
  constexpr int Q = CP + 1;
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, K = c.knn_k, L = p.spec.n_layers;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kGridThreads / 32;
  const long long env = blockIdx.x;
  const float* sw = reinterpret_cast<const float*>(smem + S.w);
  float* sv = reinterpret_cast<float*>(smem + S.v);        // v_s[CP], v_d[CP]
  float* sas = reinterpret_cast<float*>(smem + S.as);
  float* sad = reinterpret_cast<float*>(smem + S.ad);
  float* sred = reinterpret_cast<float*>(smem + S.red);
  const float* base = sw + SL::layer_off(l);
  const float* vec = base + CP * HP;                       // att_src[HP], att_dst[HP], bias[HP]
  const bool complete = c.graph_mode == SWARM_GRAPH_COMPLETE;

  // attention vectors pulled through the projection: v[k] = sum_c att[c] W[c][k]
  if (tid < 2 * CP) {
    const int k = tid % CP;
    const float* att = vec + (tid < CP ? 0 : HP);
    float v = 0.0f;
    for (int cc = 0; cc < HP; ++cc) v = fmaf(att[cc], base[k * HP + cc], v);
    sv[tid] = v;
  }
  __syncthreads();
  // alpha_src / alpha_dst of every node; complete graph: sort keys and the two largest alpha_src
  float t1 = -INFINITY, t2 = -INFINITY;
  int t1i = -1;
  uint32_t* keys = reinterpret_cast<uint32_t*>(smem + S.keys);
  uint16_t* perm = reinterpret_cast<uint16_t*>(smem + S.perm);
  const int P = grid_pow2(N);
  for (int j = tid; j < (complete ? P : N); j += kGridThreads) {
    uint32_t key = 0xFFFFFFFFu;
    if (j < N) {
      float x[CP];
      load_row<CP>(xin + (size_t)j * HP, x);
      float a = 0.0f, d = 0.0f;
#pragma unroll
      for (int k = 0; k < CP; ++k) { a = fmaf(x[k], sv[k], a); d = fmaf(x[k], sv[CP + k], d); }
      sas[j] = a;
      sad[j] = d;
      key = float_order_key(a);
      if (key == 0xFFFFFFFFu) key = 0xFFFFFFFEu;            // padding stays last
      if (a > t1) { t2 = t1; t1 = a; t1i = j; }
      else if (a > t2) t2 = a;
    }
    if (complete) {
      keys[j] = key;
      perm[j] = (uint16_t)(j < N ? j : 0);
    }
  }

  float* pre = reinterpret_cast<float*>(smem + S.pre);     // [NC][Q] pre[b] = sum over sorted positions <  b S, slope 0.2
  float* suf = reinterpret_cast<float*>(smem + S.suf);     // [NC][Q] suf[b] = sum over sorted positions >= b S, slope 1
  float* sa_sorted = reinterpret_cast<float*>(smem + S.sorted);
  float* shold = reinterpret_cast<float*>(smem + S.hold);
  const int sshift = p.sshift, SS = 1 << sshift;
  float A = 0.0f;
  if (complete) {
    auto merge = [&](float o1, int oi, float o2) {
      if (o1 > t1) { t2 = fmaxf(t1, o2); t1 = o1; t1i = oi; }
      else t2 = fmaxf(t2, o1);
    };
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) {
      const float o1 = __shfl_xor_sync(0xffffffffu, t1, sh), o2 = __shfl_xor_sync(0xffffffffu, t2, sh);
      const int oi = __shfl_xor_sync(0xffffffffu, t1i, sh);
      merge(o1, oi, o2);
    }
    if (lane == 0) {
      sred[warp * 3 + 0] = t1;
      sred[warp * 3 + 1] = __int_as_float(t1i);
      sred[warp * 3 + 2] = t2;
    }
    __syncthreads();
    t1 = -INFINITY; t2 = -INFINITY; t1i = -1;
    for (int w = 0; w < kWarps; ++w) merge(sred[w * 3 + 0], __float_as_int(sred[w * 3 + 1]), sred[w * 3 + 2]);
    A = t1;
    bitonic_sort_pairs(keys, perm, P);
    for (int pp = tid; pp < N; pp += kGridThreads) sa_sorted[pp] = sas[perm[pp]];
    // block sums of the NB = ceil(N / S) blocks of S sorted positions, one (block, quantity) pair per thread
    const int NB = (N + SS - 1) >> sshift;
    for (int it = tid; it < NB * Q; it += kGridThreads) {
      const int b = it / Q, q = it - b * Q;
      float sp = 0.0f, ss = 0.0f;
      const int e = min((b + 1) << sshift, N);
      for (int pp = b << sshift; pp < e; ++pp) {
        const int j = perm[pp];
        const float a = sas[j];
        const float v = q == 0 ? 1.0f : xin[(size_t)j * HP + q - 1];
        sp = fmaf(__expf(0.2f * (a - A)), v, sp);
        ss = fmaf(__expf(a - A), v, ss);
      }
      pre[(size_t)b * Q + q] = sp;
      suf[(size_t)b * Q + q] = ss;
    }
    __syncthreads();
    // exclusive prefix / inclusive-from-the-end suffix over the blocks, one warp per quantity, lanes over block chunks
    for (int q = warp; q < Q; q += kWarps) {
      const int per = (NB + 31) / 32, b0 = lane * per;
      float lp = 0.0f, ls = 0.0f;
      for (int k = 0; k < per; ++k)
        if (b0 + k < NB) { lp += pre[(size_t)(b0 + k) * Q + q]; ls += suf[(size_t)(b0 + k) * Q + q]; }
      float ip = lp, is = ls;
#pragma unroll
      for (int sh = 1; sh < 32; sh <<= 1) {
        const float up = __shfl_up_sync(0xffffffffu, ip, sh);
        const float dn = __shfl_down_sync(0xffffffffu, is, sh);
        if (lane >= sh) ip += up;
        if (lane + sh < 32) is += dn;
      }
      const float tot = __shfl_sync(0xffffffffu, ip, 31);
      // exclusive prefix at the chunk start / suffix just after the chunk end: the neighbour lane's inclusive value
      const float upx = __shfl_up_sync(0xffffffffu, ip, 1), dnx = __shfl_down_sync(0xffffffffu, is, 1);
      float runp = lane > 0 ? upx : 0.0f, runs = lane < 31 ? dnx : 0.0f;
      for (int k = 0; k < per; ++k) {
        if (b0 + k < NB) {
          const float vp = pre[(size_t)(b0 + k) * Q + q];
          pre[(size_t)(b0 + k) * Q + q] = runp;
          runp += vp;
        }
      }
      for (int k = per - 1; k >= 0; --k) {
        if (b0 + k < NB) {
          runs += suf[(size_t)(b0 + k) * Q + q];
          suf[(size_t)(b0 + k) * Q + q] = runs;
        }
      }
      if (lane == 0) {
        pre[(size_t)NB * Q + q] = tot;
        suf[(size_t)NB * Q + q] = 0.0f;
      }
    }
    if (warp == 0 && t1i > 0) {
      // the holder of the largest alpha_src: its row's largest logit comes from the second largest, so it sums its row
      // directly (32 lanes over the sources, fixed lane order: deterministic)
      const float adst = sad[t1i];
      const float m = gat_logit(t2, adst);
      float ds[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) ds[q] = 0.0f;
      for (int j = lane; j < N; j += 32) {
        if (j == t1i) continue;
        const float w = __expf(gat_logit(sas[j], adst) - m);
        ds[0] += w;
        float x[CP];
        load_row<CP>(xin + (size_t)j * HP, x);
#pragma unroll
        for (int q = 1; q < Q; ++q) ds[q] = fmaf(w, x[q - 1], ds[q]);
      }
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1)
#pragma unroll
        for (int q = 0; q < Q; ++q) ds[q] += __shfl_xor_sync(0xffffffffu, ds[q], sh);
      if (lane == 0)
#pragma unroll
        for (int q = 0; q < Q; ++q) shold[q] = ds[q];
    }
  }
  __syncthreads();

  const float2* spos = reinterpret_cast<const float2*>(smem + S.pos);
  const uint16_t* cbeg = reinterpret_cast<const uint16_t*>(smem + S.cells);
  const uint16_t* cend = cbeg + kGridCells;
  const int* roff = reinterpret_cast<const int*>(smem + S.roff);
  const uint16_t* rev = p.rev + env * N * K;
  const int32_t* nbr = p.nbr + env * N * K;
  for (int i = tid; i < N; i += kGridThreads) {
    const float adst = sad[i];
    float den = 0.0f;
    float acc[CP];
#pragma unroll
    for (int k = 0; k < CP; ++k) acc[k] = 0.0f;
    float m;
    auto add = [&](int j) {
      const float w = __expf(gat_logit(sas[j], adst) - m);
      den = __fadd_rn(den, w);
      acc_row<CP>(w, xin + (size_t)j * HP, acc);
    };
    if (c.graph_mode == SWARM_GRAPH_RADIUS) {
      // in-edges: agents j != i within the radius + the trailing (0,0) of node 0
      const float2 pi = spos[i];
      const float2 neg = make_float2(-pi.x, -pi.y);
      const int cx = grid.cx(pi.x), cy = grid.cy(pi.y);
      const int y0 = max(cy - 1, 0), y1 = min(cy + 1, grid.ny - 1), x0 = max(cx - 1, 0), x1 = min(cx + 1, grid.nx - 1);
      auto for_each_source = [&](auto&& fn) {
        for (int yy = y0; yy <= y1; ++yy)
          for (int xx = x0; xx <= x1; ++xx) {
            const int cc = yy * grid.nx + xx;
            for (int q = cbeg[cc], e = cend[cc]; q < e; ++q) {
              const int j = (int)(keys[q] & kIdxMask);
              if (j != i && grid_hit(spos[j], neg, p.qmax_r)) fn(j);
            }
          }
        if (i == 0) fn(0);
      };
      float amax = -INFINITY;
      for_each_source([&](int j) { amax = fmaxf(amax, sas[j]); });
      m = gat_logit(amax, adst);                           // LeakyReLU and the rounded add are monotone
      for_each_source(add);
    } else if (c.graph_mode == SWARM_GRAPH_KNN) {
      // in-edges in edge-list order (simulator.py:20-24): rows < i that list i, the own row (self twice), rows > i,
      // the trailing (0,0) of node 0
      const int b = roff[i], e = roff[i + 1];
      const int32_t* own = nbr + (size_t)i * K;
      int split = b;
      while (split < e && rev[split] < i) ++split;
      auto for_each_source = [&](auto&& fn) {
        for (int x = b; x < split; ++x) fn((int)rev[x]);
        for (int r = 0; r < K; ++r) {
          const int a = own[r];
          if (a == i) fn(i);
          fn(a);
        }
        for (int x = split; x < e; ++x) fn((int)rev[x]);
        if (i == 0) fn(0);
      };
      float amax = -INFINITY;
      for_each_source([&](int j) { amax = fmaxf(amax, sas[j]); });
      m = gat_logit(amax, adst);
      for_each_source(add);
    } else if (i == t1i && i != 0) {
      den = shold[0];
#pragma unroll
      for (int k = 0; k < CP; ++k) acc[k] = shold[k + 1];
    } else {
      // complete graph: sources split by the sign of a_j + d_i into a sorted prefix (slope 0.2) and suffix (slope 1),
      // each factorised against the env's largest a (see gatq_large_sorted_kernel); then the own term is removed
      const float zA = A + adst;
      m = zA > 0.0f ? zA : 0.2f * zA;                      // the row's largest logit (node 0 keeps its own source)
      int lo = 0, hi = N;
      const float thr = -adst;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sa_sorted[mid] <= thr) lo = mid + 1; else hi = mid;
      }
      const float c1 = __expf(zA - m), c2 = __expf(0.2f * zA - m);
      float ps[Q], ss[Q];
      const int cp = lo >> sshift, cs = (lo + SS - 1) >> sshift;
#pragma unroll
      for (int q = 0; q < Q; ++q) { ps[q] = pre[(size_t)cp * Q + q]; ss[q] = suf[(size_t)cs * Q + q]; }
      for (int pp = cp << sshift; pp < lo; ++pp) {
        const int j = perm[pp];
        const float e2 = __expf(0.2f * (sa_sorted[pp] - A));
        float x[CP];
        load_row<CP>(xin + (size_t)j * HP, x);
        ps[0] += e2;
#pragma unroll
        for (int q = 1; q < Q; ++q) ps[q] = fmaf(e2, x[q - 1], ps[q]);
      }
      const int top = min(cs << sshift, N);
      for (int pp = top - 1; pp >= lo; --pp) {
        const int j = perm[pp];
        const float e1 = __expf(sa_sorted[pp] - A);
        float x[CP];
        load_row<CP>(xin + (size_t)j * HP, x);
        ss[0] += e1;
#pragma unroll
        for (int q = 1; q < Q; ++q) ss[q] = fmaf(e1, x[q - 1], ss[q]);
      }
      den = fmaf(c1, ss[0], c2 * ps[0]);
#pragma unroll
      for (int k = 0; k < CP; ++k) acc[k] = fmaf(c1, ss[k + 1], c2 * ps[k + 1]);
      if (i != 0) {
        const float wown = __expf(gat_logit(sas[i], adst) - m);
        den -= wown;
        acc_row<CP>(-wown, xin + (size_t)i * HP, acc);
      }
    }
    // h = W (acc / (den + 1e-16)) + bias, activation
    const float inv = 1.0f / __fadd_rn(den, 1e-16f);
    float xm[HP];
#pragma unroll
    for (int k = 0; k < HP; ++k) xm[k] = k < CP ? acc[k < CP ? k : 0] * inv : 0.0f;
    float x[HP];
    stack_project<HP>(base, l, xm, x);
    const bool relu = p.spec.activation[l] == SWARM_ACT_RELU;
#pragma unroll
    for (int cc = 0; cc < HP; ++cc) {
      const float v = __fadd_rn(x[cc], vec[2 * HP + cc]);
      x[cc] = relu ? fmaxf(v, 0.0f) : tanhf(v);          // padded channels: weights and bias are 0
    }
    if (l + 1 < L) {
      float* r = xout + (size_t)i * HP;
#pragma unroll
      for (int cc = 0; cc < HP; cc += 4)
        *reinterpret_cast<float4*>(r + cc) = make_float4(x[cc], x[cc + 1], x[cc + 2], x[cc + 3]);
    } else {
      float rr[HP];
      float q[SL::kW2Cols];
      stack_head<HP>(sw, L, x, rr, q);
      const float* b2 = stack_lin2_bias<HP>(sw, L);
      float best = 0.0f;
      int action = 0;
#pragma unroll
      for (int a = 0; a < 9; ++a) {
        q[a] = __fadd_rn(q[a], b2[a]);
        if (a == 0 || q[a] > best) { best = q[a]; action = a; }
      }
      const long long g = env * N + i;
      if (p.q_out) {
#pragma unroll
        for (int a = 0; a < 9; ++a) p.q_out[g * 9 + a] = q[a];
      }
      if (p.act_out) p.act_out[g] = action;
    }
  }
  __syncthreads();
}

template <int HP>
__global__ void __launch_bounds__(kGridThreads) gatstack_large_kernel(const __grid_constant__ StackLargeParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, K = c.knn_k, L = p.spec.n_layers;
  const int tid = threadIdx.x;
  const long long env = blockIdx.x;
  const StackLargeSmem S = stack_large_smem<HP>(L, N, c.graph_mode);
  float* sw = reinterpret_cast<float*>(smem + S.w);
  float* rows0 = p.rows + env * N * HP;
  float* rows1 = p.rows + ((long long)c.num_envs + env) * N * HP;
  const float4* st = p.state + env * N;

  stack_stage_weights<HP>(p.spec, p.weights, sw, tid, kGridThreads);
  // conv1 input rows: the node features (train:95-99), 8 padded columns
  for (int i = tid; i < N; i += kGridThreads) {
    float x[HP];
    stack_features<HP>(x, st[i], c, p.spec.in_features, i);
    float4* r = reinterpret_cast<float4*>(rows0 + (size_t)i * HP);
    r[0] = make_float4(x[0], x[1], x[2], x[3]);
    r[1] = make_float4(x[4], x[5], x[6], x[7]);
  }
  CellGrid grid = {};
  if (c.graph_mode == SWARM_GRAPH_RADIUS) {
    float2* spos = reinterpret_cast<float2*>(smem + S.pos);
    for (int j = tid; j < N; j += kGridThreads) {
      const float4 s = st[j];
      spos[j] = make_float2(s.x, s.y);
    }
    __syncthreads();
    grid = grid_build([&](int j) { return spos[j]; }, N, grid_pow2(N), c.graph_radius,
                      reinterpret_cast<uint32_t*>(smem + S.keys), reinterpret_cast<uint16_t*>(smem + S.cells),
                      reinterpret_cast<uint16_t*>(smem + S.cells) + kGridCells, reinterpret_cast<float*>(smem + S.red));
  } else if (c.graph_mode == SWARM_GRAPH_KNN) {
    // transpose the topk table: rows ii != a that list a, per a, sorted by ii (the atomics' fill order is not
    // deterministic; the sums must be)
    int* roff = reinterpret_cast<int*>(smem + S.roff);
    int* rcur = reinterpret_cast<int*>(smem + S.rcur);
    __shared__ int warp_tot[kGridThreads / 32];
    const int32_t* nbr = p.nbr + env * N * K;
    uint16_t* rev = p.rev + env * N * K;
    for (int i = tid; i <= N; i += kGridThreads) rcur[i] = 0;
    __syncthreads();
    for (int e = tid; e < N * K; e += kGridThreads) {
      const int ii = e / K, a = nbr[e];
      if (a != ii) atomicAdd(&rcur[a], 1);
    }
    __syncthreads();
    block_exclusive_scan(rcur, roff, N, warp_tot);
    for (int i = tid; i < N; i += kGridThreads) rcur[i] = 0;
    __syncthreads();
    for (int e = tid; e < N * K; e += kGridThreads) {
      const int ii = e / K, a = nbr[e];
      if (a != ii) rev[roff[a] + atomicAdd(&rcur[a], 1)] = (uint16_t)ii;
    }
    __syncthreads();
    for (int i = tid; i < N; i += kGridThreads) {
      const int b = roff[i], e = roff[i + 1];
      for (int x = b + 1; x < e; ++x) {
        const uint16_t v = rev[x];
        int y = x - 1;
        while (y >= b && rev[y] > v) { rev[y + 1] = rev[y]; --y; }
        rev[y + 1] = v;
      }
    }
  }
  __syncthreads();
  for (int l = 0; l < L; ++l) {
    const float* xin = (l & 1) ? rows1 : rows0;
    float* xout = (l & 1) ? rows0 : rows1;
    if (l == 0) stack_large_layer<HP, 8>(p, smem, S, l, grid, xin, xout);
    else stack_large_layer<HP, HP>(p, smem, S, l, grid, xin, xout);
  }
}

template <int HP>
static int stack_large_smem_hp(const SwarmConfig& c, const SwarmStackSpec& s) {
  return stack_large_smem<HP>(s.n_layers, c.n_agents, c.graph_mode).total;
}

static int stack_large_hp(const SwarmStackSpec& s) { return s.hidden <= 8 ? 8 : (s.hidden <= 16 ? 16 : 32); }

int stack_large_smem_bytes(const SwarmConfig& c, const SwarmStackSpec& s) {
  const int hp = stack_large_hp(s);
  return hp == 8 ? stack_large_smem_hp<8>(c, s) : (hp == 16 ? stack_large_smem_hp<16>(c, s) : stack_large_smem_hp<32>(c, s));
}

// layer rows [2][B][N][HP] floats, then (kNN) the in-edge lists [B][N*K] uint16; 256-byte aligned pieces
long long stack_large_workspace_bytes(const SwarmConfig& c, int hp) {
  const long long bn = (long long)c.num_envs * c.n_agents;
  long long b = 256 + ((2 * bn * hp * 4 + 255) & ~255LL);
  if (c.graph_mode == SWARM_GRAPH_KNN) b += bn * c.knn_k * 2;
  return b;
}

long long stack_large_workspace_bytes(const SwarmConfig& c, const SwarmStackSpec& s) {
  return stack_large_workspace_bytes(c, stack_large_hp(s));
}

template <int HP>
static cudaError_t launch_stack_large_hp(const StackLargeParams& p, cudaStream_t stream) {
  const int smem = stack_large_smem_hp<HP>(p.cfg, p.spec);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  if (smem > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(gatstack_large_kernel<HP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
  }
  gatstack_large_kernel<HP><<<p.cfg.num_envs, kGridThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_gatstack_large(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, const float* state,
                                  const int32_t* nbr, float* q, int32_t* actions, void* workspace, cudaStream_t stream) {
  StackLargeParams p;
  std::memset(&p, 0, sizeof(p));
  p.cfg = c;
  p.spec = spec;
  p.weights = weights;
  p.state = reinterpret_cast<const float4*>(state);
  p.nbr = nbr;
  p.q_out = q;
  p.act_out = actions;
  const int hp = stack_large_hp(spec);
  const long long bn = (long long)c.num_envs * c.n_agents;
  const uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
  p.rows = reinterpret_cast<float*>(base);
  p.rev = reinterpret_cast<uint16_t*>(base + ((2 * bn * hp * 4 + 255) & ~255LL));
  p.qmax_r = c.graph_mode == SWARM_GRAPH_RADIUS ? sq_threshold(c.graph_radius) : 0.0f;
  p.sshift = stack_large_sshift(c.n_agents);
  if (hp == 8) return launch_stack_large_hp<8>(p, stream);
  if (hp == 16) return launch_stack_large_hp<16>(p, stream);
  return launch_stack_large_hp<32>(p, stream);
}

}  // namespace swarm
