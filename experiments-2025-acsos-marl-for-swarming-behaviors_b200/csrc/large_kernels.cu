// large_kernels.cu -- large swarms (128 < N <= 4096 agents per env; BASELINE config "1024 agents x 1024 envs").
//
// An env no longer fits a 128-thread tile, so the path is split into stand-alone kernels that keep one env's
// positions in shared memory (8 B per agent) and give every agent a thread:
//   sim_step_large_kernel   vmas Environment.step: O(N) branch-free contact sweep per agent against the env's
//                           positions in shared memory (same device code as the small-swarm kernels)
//   goto_reward_large_kernel GoTo's collective reward, summed sequentially in agent order like the reference
//   knn_large_kernel        simulator.py:9-26 for n >= 64 k, where torch.topk takes its std::partial_sort branch:
//                           heap_select + sort_heap (csrc/knn_select.h) over a *virtual* row -- the k-element heap
//                           lives in shared memory, the remaining candidates are streamed and their distances
//                           computed on the fly (a squared-distance test skips the sqrt for candidates that cannot
//                           beat the heap top), so no O(N^2) distance matrix is ever stored
//   complete_edges_kernel   train_gcn_dqn.py:94-110 edge list (closed form)
// The Q-network then runs through the generic CSR path (csr_kernels.cu).
#include "knn_select.h"
#include "knn_small.h"
#include "gatq_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kLargeThreads = 256;

// grid = envs: ONE CTA owns a whole env.  It stages every pre-step position of the env in shared memory before any
// thread writes a post-step state, so state_out may alias state_in (the in-place use of World.step / rollout_large);
// a (chunk, env) grid would let a later-scheduled chunk read partner positions that an earlier chunk already stepped.
__global__ void __launch_bounds__(kLargeThreads) sim_step_large_kernel(const __grid_constant__ SimStepArgs p) {
  extern __shared__ float2 spos[];
  __shared__ int s_hits;
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents;
  const long long env = blockIdx.x;
  const float4* env_state = p.state_in + env * N;
  if (threadIdx.x == 0) s_hits = 0;
  int my_hits = 0;
  for (int j = threadIdx.x; j < N; j += kLargeThreads) {
    const float4 s = env_state[j];
    spos[j] = make_float2(s.x, s.y);
  }
  __syncthreads();
  const bool oa = c.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE;
  for (int i = threadIdx.x; i < N; i += kLargeThreads) {
    const long long gidx = env * N + i;
    float4 s = env_state[i];               // only this thread ever writes index i: no hazard with the in-place store below
    float2 u;
    decode_action(p.actions[gidx], u.x, u.y);
    uint8_t flags = 0;
    uint32_t cmask = 0;
    agent_step(s, u, spos, N, i, oa, c, p.world, flags, cmask);
    float dgoal, dobs;
    const float reward = post_step_reward(s, oa, c, dgoal, dobs, flags);
    if (oa) {
      if (p.rewards) p.rewards[gidx] = reward;
      if (p.returns) p.returns[gidx] = __fadd_rn(p.returns[gidx], reward);
      my_hits += (flags & SWARM_FLAG_HIT) ? 1 : 0;
    }
    p.state_out[gidx] = s;
    store_step_outputs(p, gidx, s, dgoal, dobs, flags, 0u);     // no contact masks above 32 agents
  }
  if (p.hits) {
    if (my_hits) atomicAdd(&s_hits, my_hits);          // integer: order-independent
    __syncthreads();
    if (threadIdx.x == 0) p.hits[env] += s_hits;
  }
}

// GoTo (go_to:108-115): reward = 0 + (-d_0) + (-d_1) + ... summed in agent order, the same value for every agent.
__global__ void __launch_bounds__(kLargeThreads) goto_reward_large_kernel(SwarmConfig c, const float4* __restrict__ state,
                                                                          float* __restrict__ rewards,
                                                                          float* __restrict__ returns) {
  extern __shared__ float sdg[];
  __shared__ float total;
  const int N = c.n_agents;
  const long long env = blockIdx.x;
  for (int j = threadIdx.x; j < N; j += kLargeThreads) {
    const float4 s = state[env * N + j];
    sdg[j] = goal_distance(s.x, s.y, c);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float r = 0.0f;
    for (int a = 0; a < N; ++a) r = __fadd_rn(r, -sdg[a]);
    total = r;
  }
  __syncthreads();
  const float r = total;
  for (int j = threadIdx.x; j < N; j += kLargeThreads) {
    if (rewards) rewards[env * N + j] = r;
    if (returns) returns[env * N + j] = __fadd_rn(returns[env * N + j], r);
  }
}

// ---- kNN, partial_sort branch ------------------------------------------------------------------
// The K-entry heap of std::partial_sort lives in shared memory as ONE 8-byte word per entry: (key, index) with
// key = the distance's bit pattern (monotone for the non-negative 2-norm; every NaN maps to one key above +inf, like
// torch's comparator -- knn_small.h), so a heap access is a single 64-bit load / store and a comparison a single integer
// compare.  The algorithms are the generic ones of knn_select.h (make_heap, __adjust_heap for the replace-top of
// heap_select, sort_heap); only indices leave the kernel.
struct KnnKeyPair {
  uint32_t v;
  int i;
};
__device__ __forceinline__ bool knn_less(const KnnKeyPair& a, const KnnKeyPair& b) { return a.v < b.v; }

struct HeapRow {
  uint2* h;             // [K][threads]
  __device__ __forceinline__ KnnKeyPair get(int j) const {
    const uint2 w = h[j * kLargeThreads];
    KnnKeyPair p;
    p.v = w.x;
    p.i = (int)w.y;
    return p;
  }
  __device__ __forceinline__ void set(int j, const KnnKeyPair& p) { h[j * kLargeThreads] = make_uint2(p.v, (uint32_t)p.i); }
};

struct LargeKnnParams {
  SwarmConfig cfg;
  const float4* state;
  int32_t* edges;        // [B][2][E] or nullptr
  int32_t* nbr;          // [B][N][K] or nullptr
  int32_t edges_per_env;
};

// grid = (envs, chunks of 256 agents); dynamic smem: positions float2[N], heap uint2[K][256]
__global__ void __launch_bounds__(kLargeThreads) knn_large_kernel(const __grid_constant__ LargeKnnParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, K = c.knn_k;
  float2* spos = reinterpret_cast<float2*>(smem_raw);
  uint2* hw = reinterpret_cast<uint2*>(spos + N);
  float4* sbox = reinterpret_cast<float4*>(                                       // [chunks] (xmin, xmax, ymin, ymax)
      (reinterpret_cast<uintptr_t>(hw + (size_t)K * kLargeThreads) + 15) & ~(uintptr_t)15);
  const long long env = blockIdx.x;          // envs on grid.x (no 65 535 cap), agent chunks on grid.y
  for (int j = threadIdx.x; j < N; j += kLargeThreads) {
    const float4 s = p.state[env * N + j];
    spos[j] = make_float2(s.x, s.y);
  }
  __syncthreads();
  // bounding box of every candidate chunk (K + 32 c .. K + 32 c + 31): a chunk whose box lies beyond the heap top holds
  // no candidate and is skipped without looking at its members
  {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nchunks = (N - K + 31) / 32;
    for (int ch = warp; ch < nchunks; ch += kLargeThreads / 32) {
      const int j = K + ch * 32 + lane;
      const bool in = j < N;
      const float2 q = in ? spos[j] : make_float2(0.f, 0.f);
      float xmin = in ? q.x : INFINITY, xmax = in ? q.x : -INFINITY, ymin = in ? q.y : INFINITY, ymax = in ? q.y : -INFINITY;
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) {
        xmin = fminf(xmin, __shfl_xor_sync(0xffffffffu, xmin, sh));
        xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, sh));
        ymin = fminf(ymin, __shfl_xor_sync(0xffffffffu, ymin, sh));
        ymax = fmaxf(ymax, __shfl_xor_sync(0xffffffffu, ymax, sh));
      }
      if (lane == 0) sbox[ch] = make_float4(xmin, xmax, ymin, ymax);
    }
  }
  __syncthreads();
  const int i = blockIdx.y * kLargeThreads + threadIdx.x;
  if (i >= N) return;
  const float sx = spos[i].x, sy = spos[i].y;
  HeapRow heap{hw + threadIdx.x};
  for (int j = 0; j < K; ++j) {
    const float2 o = spos[j];
    KnnKeyPair pr;
    pr.v = knn_key_nonneg(norm2(__fsub_rn(o.x, sx), __fsub_rn(o.y, sy)));
    pr.i = j;
    heap.set(j, pr);
  }
  // std::partial_sort(b, b + k, e) = __heap_select + __sort_heap; the select loop is open-coded to skip the sqrt of
  // candidates whose squared distance already rules them out (q_j >= q_top  =>  d_j >= d_top  =>  !comp)
  knn_make_heap(heap, 0, K);
  // The candidates K .. N-1 are visited in index order, kChunk at a time.  A branch-free sweep (packed subtract, one
  // compare per candidate) marks those whose squared distance is below the heap top's at the START of the chunk --
  // the top only ever decreases, so this is a superset of the candidates heap_select would accept -- and only the
  // marked ones go through the (divergent) replace-top path, re-tested against the current top.
  // A warp therefore pays for max-over-lanes(inserts per chunk) heap updates instead of one per candidate at which
  // ANY of its 32 lanes inserts.  (Measured on C4: 16 per chunk 3.8 ms, 32: 2.9 ms, 64: 3.5 ms, unchunked: 5.7 ms.)
  constexpr int kChunk = 32;
  const float2 neg = make_float2(-sx, -sy);
  // squared-distance threshold for "could be below the top" (conservative: never drops a candidate with d_j < top);
  // a NaN top is above every real distance
  auto threshold = [](uint32_t top_key) {
    const float top = __uint_as_float(top_key);
    return (top != top) ? INFINITY : __fmul_rn(top, top) * 1.0000005f + 1e-37f;
  };
  for (int base = K; base < N; base += kChunk) {
    const int cnt = (N - base < kChunk) ? (N - base) : kChunk;
    const float thr0 = threshold(hw[threadIdx.x].x);
    {
      // squared distance to the chunk's bounding box, with a margin for its own rounding: beyond the threshold, no
      // member can be (a NaN threshold or box compares false and the chunk is swept)
      const float4 bb = sbox[(base - K) / kChunk];
      const float ex = fmaxf(fmaxf(bb.x - sx, sx - bb.y), 0.0f), ey = fmaxf(fmaxf(bb.z - sy, sy - bb.w), 0.0f);
      if (fmaf(ey, ey, ex * ex) * 0.999999f >= thr0) continue;
    }
    uint32_t m = 0;
#pragma unroll 8
    for (int u = 0; u < cnt; ++u) {
      const float2 d = __fadd2_rn(spos[base + u], neg);
      const float q = __fmaf_rn(d.y, d.y, __fmul_rn(d.x, d.x));
      m |= (q < thr0 || q != q) ? (1u << u) : 0u;
    }
    while (m) {
      const int j = base + __ffs(m) - 1;
      m &= m - 1;
      const float2 o = spos[j];
      const float dx = __fsub_rn(o.x, sx), dy = __fsub_rn(o.y, sy);
      const float q = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));
      const uint32_t top_key = hw[threadIdx.x].x;
      if (q < threshold(top_key) || q != q) {
        KnnKeyPair cand;
        cand.v = knn_key_nonneg(__fsqrt_rn(q));
        cand.i = j;
        if (cand.v < top_key) knn_adjust_heap(heap, 0, 0, K, cand);       // __pop_heap(first, middle, j)
      }
    }
  }
  knn_sort_heap(heap, 0, K);
  if (p.nbr)
    for (int r = 0; r < K; ++r) p.nbr[(env * N + i) * K + r] = (int)hw[r * kLargeThreads + threadIdx.x].y;
  if (p.edges) {
    const int E = p.edges_per_env;
    int32_t* r0 = p.edges + env * 2 * E;
    int32_t* r1 = r0 + E;
    for (int r = 0; r < K; ++r) {
      const int a = (int)hw[r * kLargeThreads + threadIdx.x].y;
      const int e = (i * K + r) * 2;
      r0[e] = i; r1[e] = a;
      r0[e + 1] = a; r1[e + 1] = i;
    }
    if (i == 0) { r0[E - 1] = 0; r1[E - 1] = 0; }
  }
}

// complete graph, closed form: pair (i, j), i < j at edges 2p, 2p+1 with p = i N - i(i+1)/2 + (j - i - 1)
__global__ void __launch_bounds__(kLargeThreads) complete_edges_kernel(int N, int E, int32_t* __restrict__ edges) {
  const long long env = blockIdx.x;
  int32_t* r0 = edges + env * 2 * E;
  int32_t* r1 = r0 + E;
  const int i = blockIdx.y;
  const long long base = (long long)i * N - ((long long)i * (i + 1)) / 2;
  for (int j = i + 1 + threadIdx.x; j < N; j += kLargeThreads) {
    const long long e = 2 * (base + (j - i - 1));
    r0[e] = i; r1[e] = j;
    r0[e + 1] = j; r1[e + 1] = i;
  }
  if (i == 0 && threadIdx.x == 0) { r0[E - 1] = 0; r1[E - 1] = 0; }
}

// ---- fused Q forward for large kNN swarms ---------------------------------------------------------------------
// GCN.forward (train_gcn_dqn.py:59-70) on the symmetrised kNN graph of simulator.py:9-26 straight from the topk table,
// one CTA per env, everything of the env in shared memory: the projected features (N x 32 floats), the table and its
// TRANSPOSE.  The in-edges of node i in edge-list order are: rows ii < i that list i (at most one edge each, topk rows
// hold distinct indices), then i's own row (per slot (i -> i) if a == i, then (a -> i)), then rows ii > i, and the
// trailing (0,0) for node 0.  "Rows that list i" is the transposed table: counted and filled with shared-memory
// atomics, then each (short) list is sorted by row index, which makes the order -- and therefore every sum --
// deterministic and equal to the generic path's (edge list -> stable sort by target -> CSR kernels), whose per-tick
// edge export (164 KB per env), int64 glue and radix sort this kernel replaces.
constexpr int kQLThreads = 512;

struct LargeQParams {
  SwarmConfig cfg;
  const float4* state;
  const int32_t* nbr;        // [B][N][K]
  const float* weights;
  float* q_out;              // [B*N][9] or nullptr
  int32_t* act_out;          // [B*N] or nullptr
};

__host__ __device__ inline size_t large_q_smem_bytes(int N, int K) {
  size_t b = (size_t)((TW_COUNT + 3) & ~3) * 4;      // weights
  b += (size_t)N * 32 * 4;                           // h rows
  b += (size_t)N * 2 * 4;                            // alpha_src, alpha_dst
  b += (size_t)(N + 1) * 4 * 2;                      // list offsets, fill cursors
  b += (size_t)N * K * 2 * 2;                        // table and transposed lists (uint16)
  return b + 64;
}

__global__ void __launch_bounds__(kQLThreads, 1) gatq_knn_large_kernel(const __grid_constant__ LargeQParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, K = c.knn_k;
  const int tid = threadIdx.x;
  const long long env = blockIdx.x;
  float* sw = reinterpret_cast<float*>(smem_raw);
  float* sh = sw + ((TW_COUNT + 3) & ~3);
  float* sas = sh + (size_t)N * 32;
  float* sad = sas + N;
  int* roff = reinterpret_cast<int*>(sad + N);           // [N + 1]
  int* rcur = roff + (N + 1);                            // [N + 1]
  uint16_t* tab = reinterpret_cast<uint16_t*>(rcur + (N + 1));
  uint16_t* rev = tab + (size_t)N * K;
  __shared__ int warp_tot[kQLThreads / 32];

  stage_weights(p.weights, sw, tid, kQLThreads);
  const int32_t* nbr = p.nbr + env * N * K;
  for (int e = tid; e < N * K; e += kQLThreads) tab[e] = (uint16_t)nbr[e];
  for (int i = tid; i <= N; i += kQLThreads) rcur[i] = 0;
  __syncthreads();
  // in-degree from other rows
  for (int e = tid; e < N * K; e += kQLThreads) {
    const int ii = e / K, a = tab[e];
    if (a != ii) atomicAdd(&rcur[a], 1);
  }
  __syncthreads();
  // exclusive scan of rcur[0..N) -> roff (every thread owns a contiguous chunk)
  {
    const int per = (N + kQLThreads - 1) / kQLThreads;
    const int b0 = tid * per;
    int local = 0;
    for (int k = 0; k < per; ++k) local += (b0 + k < N) ? rcur[b0 + k] : 0;
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
        const int cnt = rcur[b0 + k];
        roff[b0 + k] = run;
        run += cnt;
      }
    }
    if (tid == kQLThreads - 1) roff[N] = base + incl;
  }
  __syncthreads();
  for (int i = tid; i < N; i += kQLThreads) rcur[i] = 0;
  __syncthreads();
  for (int e = tid; e < N * K; e += kQLThreads) {
    const int ii = e / K, a = tab[e];
    if (a != ii) rev[roff[a] + atomicAdd(&rcur[a], 1)] = (uint16_t)ii;
  }
  __syncthreads();
  // sort every list by row index (insertion sort; the lists hold ~K entries) and project the node features
  for (int i = tid; i < N; i += kQLThreads) {
    const int b = roff[i], e = roff[i + 1];
    for (int x = b + 1; x < e; ++x) {
      const uint16_t v = rev[x];
      int y = x - 1;
      while (y >= b && rev[y] > v) { rev[y + 1] = rev[y]; --y; }
      rev[y + 1] = v;
    }
    const float4 st = p.state[env * N + i];
    const float xi[7] = {st.x, st.y, st.z, st.w, c.goal_x, c.goal_y, (float)i};
    float h[32], asrc, adst;
    gat_project(xi, sw, h, asrc, adst);
    float4* r = reinterpret_cast<float4*>(sh + (size_t)i * 32);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) r[c4] = make_float4(h[4 * c4], h[4 * c4 + 1], h[4 * c4 + 2], h[4 * c4 + 3]);
    sas[i] = asrc;
    sad[i] = adst;
  }
  __syncthreads();
  for (int i = tid; i < N; i += kQLThreads) {
    const float adst = sad[i];
    const int b = roff[i], e = roff[i + 1];
    const uint16_t* own = tab + (size_t)i * K;
    int split = b;                                    // first list entry with row index > i
    while (split < e && rev[split] < i) ++split;
    // the same three sweeps as csr_aggregate_kernel, over the in-edges in edge-list order
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
    float m = -INFINITY;
    for_each_source([&](int j) { m = fmaxf(m, gat_logit(sas[j], adst)); });
    float den = 0.0f;
    for_each_source([&](int j) { den = __fadd_rn(den, expf(__fsub_rn(gat_logit(sas[j], adst), m))); });
    den = __fadd_rn(den, 1e-16f);
    float a1[32];
#pragma unroll
    for (int cc = 0; cc < 32; ++cc) a1[cc] = 0.0f;
    for_each_source([&](int j) {
      const float w = expf(__fsub_rn(gat_logit(sas[j], adst), m));
      gat_accumulate(a1, __fdiv_rn(w, den), reinterpret_cast<const float4*>(sh + (size_t)j * 32));
    });
    float q[9];
    const int action = gat_head(a1, sw, q);
    const long long g = env * N + i;
    if (p.q_out) {
#pragma unroll
      for (int a = 0; a < 9; ++a) p.q_out[g * 9 + a] = q[a];
    }
    if (p.act_out) p.act_out[g] = action;
  }
}

// ---- the same forward with the attention in input space (tile_tc_device.cuh) -------------------------------------
// sum_e alpha_e h_src(e) = W0 (sum_e alpha_e x_src(e)) and <h_j, att> = <x_j, W0^T att>: no tile of projected features
// (N x 128 B -- what limited the kernel above to one CTA per SM and ~1 200 agents), the gather per in-edge is one 16-byte
// state instead of a 128-byte feature row, and the topk table is read from global memory.  Shared memory: 20 B per
// agent + 2 K B of reversed lists + 8 B of list offsets -> 76 KB at N = 1 024, k = 10 (two to three CTAs per SM), 202 KB
// at N = 4 096.  Same mathematics, float32-level different rounding than the bit-faithful kernel above; used where only
// the greedy actions are consumed (swarm_rollout_large), SWARM_TC=0 keeps the bit-faithful one.
__host__ __device__ inline size_t large_qx_smem_bytes(int N, int K) {
  size_t b = (size_t)((TW_COUNT + 3) & ~3) * 4 + 64;  // weights, v_s / v_d
  b += (size_t)N * 16;                                // states
  b += (size_t)N * 4;                                 // alpha_src
  b += (size_t)(N + 1) * 4 * 2;                       // list offsets, fill cursors
  b += (size_t)N * K * 2;                             // reversed lists (uint16)
  return b + 64;
}

__global__ void __launch_bounds__(kQLThreads, 2) gatq_knn_large_x_kernel(const __grid_constant__ LargeQParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, K = c.knn_k;
  const int tid = threadIdx.x;
  const long long env = blockIdx.x;
  float* sw = reinterpret_cast<float*>(smem_raw);
  float* sv = sw + ((TW_COUNT + 3) & ~3);                 // v_s[8], v_d[8]
  float4* sst = reinterpret_cast<float4*>(sv + 16);
  float* sas = reinterpret_cast<float*>(sst + N);
  int* roff = reinterpret_cast<int*>(sas + N);           // [N + 1]
  int* rcur = roff + (N + 1);                            // [N + 1]
  uint16_t* rev = reinterpret_cast<uint16_t*>(rcur + (N + 1));
  __shared__ int warp_tot[kQLThreads / 32];

  stage_weights(p.weights, sw, tid, kQLThreads);
  const int32_t* nbr = p.nbr + env * N * K;
  for (int i = tid; i < N; i += kQLThreads) sst[i] = p.state[env * N + i];
  for (int i = tid; i <= N; i += kQLThreads) rcur[i] = 0;
  __syncthreads();
  if (tid < 16) {
    // attention vectors pulled through the projection: v[k] = sum_c att[c] W0[c][k]
    const int k = tid & 7;
    const float* att = sw + (tid < 8 ? TW_ATT_S : TW_ATT_D);
    float v = 0.0f;
    if (k < 7)
      for (int cc = 0; cc < 32; ++cc) v = fmaf(att[cc], sw[TW_W0T + k * 32 + cc], v);
    sv[tid] = v;
  }
  // in-degree from other rows
  for (int e = tid; e < N * K; e += kQLThreads) {
    const int ii = e / K, a = nbr[e];
    if (a != ii) atomicAdd(&rcur[a], 1);
  }
  __syncthreads();
  // exclusive scan of rcur[0..N) -> roff (every thread owns a contiguous chunk)
  {
    const int per = (N + kQLThreads - 1) / kQLThreads;
    const int b0 = tid * per;
    int local = 0;
    for (int k = 0; k < per; ++k) local += (b0 + k < N) ? rcur[b0 + k] : 0;
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
        const int cnt = rcur[b0 + k];
        roff[b0 + k] = run;
        run += cnt;
      }
    }
    if (tid == kQLThreads - 1) roff[N] = base + incl;
  }
  __syncthreads();
  for (int i = tid; i < N; i += kQLThreads) rcur[i] = 0;
  __syncthreads();
  for (int e = tid; e < N * K; e += kQLThreads) {
    const int ii = e / K, a = nbr[e];
    if (a != ii) rev[roff[a] + atomicAdd(&rcur[a], 1)] = (uint16_t)ii;
  }
  __syncthreads();
  // sort every list by row index (the fill order of the atomics is not deterministic; sums must be) and publish the
  // alpha_src term of every node
  for (int i = tid; i < N; i += kQLThreads) {
    const int b = roff[i], e = roff[i + 1];
    for (int x = b + 1; x < e; ++x) {
      const uint16_t v = rev[x];
      int y = x - 1;
      while (y >= b && rev[y] > v) { rev[y + 1] = rev[y]; --y; }
      rev[y + 1] = v;
    }
    const float4 st = sst[i];
    sas[i] = fmaf(st.x, sv[0], fmaf(st.y, sv[1], fmaf(st.z, sv[2], fmaf(st.w, sv[3],
             fmaf(c.goal_x, sv[4], fmaf(c.goal_y, sv[5], (float)i * sv[6]))))));
  }
  __syncthreads();
  for (int i = tid; i < N; i += kQLThreads) {
    const float4 st = sst[i];
    const float adst = fmaf(st.x, sv[8], fmaf(st.y, sv[9], fmaf(st.z, sv[10], fmaf(st.w, sv[11],
                       fmaf(c.goal_x, sv[12], fmaf(c.goal_y, sv[13], (float)i * sv[14]))))));
    const int b = roff[i], e = roff[i + 1];
    const int32_t* own = nbr + (size_t)i * K;
    int split = b;                                    // first list entry with row index > i
    while (split < e && rev[split] < i) ++split;
    // in-edges in edge-list order (simulator.py:20-24): rows < i that list i, the own row (self twice), rows > i,
    // the trailing (0,0) of node 0
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
    const float m = gat_logit(amax, adst);             // LeakyReLU and the rounded add are monotone
    float den = 0.0f, acc_id = 0.0f;
    float2 acc_p = make_float2(0.f, 0.f), acc_v = make_float2(0.f, 0.f);
    for_each_source([&](int j) {
      const float4 sj = sst[j];
      const float w = __expf(gat_logit(sas[j], adst) - m);
      den = __fadd_rn(den, w);
      acc_p = __ffma2_rn(make_float2(w, w), make_float2(sj.x, sj.y), acc_p);
      acc_v = __ffma2_rn(make_float2(w, w), make_float2(sj.z, sj.w), acc_v);
      acc_id = fmaf(w, (float)j, acc_id);
    });
    const float inv = 1.0f / __fadd_rn(den, 1e-16f);
    const float wsum = den * inv;
    const float xm[7] = {acc_p.x * inv, acc_p.y * inv, acc_v.x * inv, acc_v.y * inv, c.goal_x * wsum, c.goal_y * wsum,
                         acc_id * inv};
    // agg = W0 xm (the projection of gat_project without its attention terms), then the head
    float a1[32];
#pragma unroll
    for (int cc = 0; cc < 32; ++cc) a1[cc] = 0.0f;
    const float4* w0 = reinterpret_cast<const float4*>(sw + TW_W0T);
#pragma unroll
    for (int k = 0; k < 7; ++k) {
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        fma4_packed(xm[k], w0[k * 8 + c4], a1[4 * c4 + 0], a1[4 * c4 + 1], a1[4 * c4 + 2], a1[4 * c4 + 3]);
      }
    }
    float q[9];
    const int action = gat_head_fast(a1, sw, q);
    const long long g = env * N + i;
    if (p.q_out) {
#pragma unroll
      for (int a = 0; a < 9; ++a) p.q_out[g * 9 + a] = q[a];
    }
    if (p.act_out) p.act_out[g] = action;
  }
}

bool gatq_knn_large_x_fits(int N, int K) { return N <= 65535 && large_qx_smem_bytes(N, K) <= 227 * 1024; }

cudaError_t launch_gatq_knn_large_x(const SwarmConfig& c, const float* weights, const float* state, const int32_t* nbr,
                                    float* q, int32_t* actions, cudaStream_t stream) {
  LargeQParams p;
  p.cfg = c;
  p.state = reinterpret_cast<const float4*>(state);
  p.nbr = nbr;
  p.weights = weights;
  p.q_out = q;
  p.act_out = actions;
  const size_t smem = large_qx_smem_bytes(c.n_agents, c.knn_k);
  cudaError_t err = cudaFuncSetAttribute(gatq_knn_large_x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  gatq_knn_large_x_kernel<<<c.num_envs, kQLThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

bool gatq_knn_large_fits(int N, int K) { return N <= 65535 && large_q_smem_bytes(N, K) <= 227 * 1024; }

cudaError_t launch_gatq_knn_large(const SwarmConfig& c, const float* weights, const float* state, const int32_t* nbr,
                                  float* q, int32_t* actions, cudaStream_t stream) {
  LargeQParams p;
  p.cfg = c;
  p.state = reinterpret_cast<const float4*>(state);
  p.nbr = nbr;
  p.weights = weights;
  p.q_out = q;
  p.act_out = actions;
  const size_t smem = large_q_smem_bytes(c.n_agents, c.knn_k);
  cudaError_t err = cudaFuncSetAttribute(gatq_knn_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  gatq_knn_large_kernel<<<c.num_envs, kQLThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

// ---- launchers ------------------------------------------------------------------------------
cudaError_t launch_sim_step_large(const SimStepArgs& p, cudaStream_t stream) {
  const SwarmConfig& c = p.cfg;
  // contact partners from the uniform grid (grid_kernels.cu; same bits) unless SWARM_STEP_GRID=0 asks for the full sweep
  if (sim_step_grid_enabled(c.n_agents) && c.n_agents <= 4096) {
    if (cudaError_t e = launch_sim_step_grid(p, stream); e != cudaSuccess) return e;
  } else {
    sim_step_large_kernel<<<c.num_envs, kLargeThreads, c.n_agents * sizeof(float2), stream>>>(p);
  }
  if (c.scenario == SWARM_SCENARIO_GOTO && (p.rewards || p.returns))
    goto_reward_large_kernel<<<c.num_envs, kLargeThreads, c.n_agents * sizeof(float), stream>>>(
        c, p.state_out, p.rewards, p.returns);
  return cudaGetLastError();
}

cudaError_t launch_graph_large(const SwarmConfig& c, const float* state, int32_t* edges, int32_t* nbr, int edges_per_env,
                               cudaStream_t stream) {
  if (c.graph_mode == SWARM_GRAPH_KNN) {
    LargeKnnParams p;
    p.cfg = c;
    p.state = reinterpret_cast<const float4*>(state);
    p.edges = edges;
    p.nbr = nbr;
    p.edges_per_env = edges_per_env;
    const dim3 grid(c.num_envs, (c.n_agents + kLargeThreads - 1) / kLargeThreads);
    const size_t smem = c.n_agents * sizeof(float2) + (size_t)c.knn_k * kLargeThreads * 8 +
                        (size_t)((c.n_agents - c.knn_k + 31) / 32) * sizeof(float4) + 16;
    cudaError_t err = cudaFuncSetAttribute(knn_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    knn_large_kernel<<<grid, kLargeThreads, smem, stream>>>(p);
  } else if (edges) {
    const dim3 grid(c.num_envs, c.n_agents);
    complete_edges_kernel<<<grid, kLargeThreads, 0, stream>>>(c.n_agents, edges_per_env, edges);
  }
  return cudaGetLastError();
}

}  // namespace swarm
