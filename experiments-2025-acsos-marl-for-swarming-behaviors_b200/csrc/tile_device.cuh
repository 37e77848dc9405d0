// tile_device.cuh -- device functions of the env-tile scheme (thread = agent, CTA = floor(128/N) envs),
// shared by the rollout / forward / graph kernels (tile_kernels.cu) and the DQN gradient kernel
// (dqn_tc_kernels.cu).
#ifndef SWARM_TILE_DEVICE_CUH
#define SWARM_TILE_DEVICE_CUH

#include "gatq_device.cuh"
#include "knn_select.h"
#include "knn_small.h"

namespace swarm {

struct SmemPairs {
  float* v;
  uint8_t* x;
  int stride;
  __device__ __forceinline__ KnnPair get(int j) const {
    KnnPair p;
    p.v = v[j * stride];
    p.i = x[j * stride];
    return p;
  }
  __device__ __forceinline__ void set(int j, const KnnPair& p) {
    v[j * stride] = p.v;
    x[j * stride] = (uint8_t)p.i;
  }
};

// Position of this thread inside the tile
struct TileThread {
  int tid, el, i, envbase;
  long long env, gidx;
  bool active;
};

__device__ __forceinline__ TileThread tile_thread(int n_agents, int epb, long long num_envs, int bal_q = 0, int bal_r = 0) {
  TileThread t;
  t.tid = threadIdx.x;
  t.el = t.tid / n_agents;
  t.i = t.tid - t.el * n_agents;
  const int b = blockIdx.x;
  if (bal_q > 0) {
    t.env = (long long)b * bal_q + (b < bal_r ? b : bal_r) + t.el;
    epb = bal_q + (b < bal_r ? 1 : 0);
  } else {
    t.env = (long long)b * epb + t.el;
  }
  t.active = (t.el < epb) && (t.env < num_envs);
  t.envbase = t.el * n_agents;
  t.gidx = t.env * n_agents + t.i;
  return t;
}

// Shared-memory views used by the graph + GAT forward
struct TileGraphSmem {
  float* sh;        // [T][kHPad] projected features
  float* sas;       // [T] alpha_src
  float* swt;       // [maxdeg][T] per-thread edge scratch (logit -> exp -> alpha)
  uint8_t* sin;     // [maxdeg][T] in-edge sources (env-local ids), edge-list order
  float* skv;       // [N][T] kNN distance rows
  uint8_t* ski;     // [N][T] kNN index rows
  uint8_t* snbr;    // [K][T] topk result rows
};

// complete graph (train:101-108): sources into node d in edge-list order are 0..N-1 without d; node 0
// additionally receives the final (0,0) self loop.  Returns the in-degree.
__device__ __forceinline__ int tile_in_edges_complete(const TileGraphSmem& g, const TileThread& t, int N) {
  const int T = kTileThreads;
  int deg = 0;
  for (int j = 0; j < N; ++j)
    if (j != t.i) g.sin[(deg++) * T + t.tid] = (uint8_t)j;
  if (t.i == 0) g.sin[(deg++) * T + t.tid] = 0;
  return deg;
}

// radius graph (EXTENSION, include/swarm_b200.h SWARM_GRAPH_RADIUS): the complete builder filtered by distance, so
// the in-edges of node i in edge-list order are the sources j != i with ||p_j - p_i|| <= r in ascending j; node 0
// additionally receives the trailing (0,0).  `pos` is the env-tile state buffer.
__device__ __forceinline__ bool radius_hit(const float4* pos, int j, const float2& neg, float qmax_r) {
  const float2 d = __fadd2_rn(xy_of(pos[j]), neg);
  return __fmaf_rn(d.y, d.y, __fmul_rn(d.x, d.x)) <= qmax_r;
}

__device__ __forceinline__ int tile_in_edges_radius(const TileGraphSmem& g, const TileThread& t, const float4* pos,
                                                    const float4& s, int N, float qmax_r) {
  const int T = kTileThreads;
  const float2 neg = make_float2(-s.x, -s.y);
  const float4* env = pos + t.envbase;
  uint8_t* sin = g.sin + t.tid;
  int deg = 0;
#pragma unroll 4
  for (int j = 0; j < N; ++j) {
    const bool hit = radius_hit(env, j, neg, qmax_r) && (j != t.i);
    if (hit) sin[deg * T] = (uint8_t)j;
    deg += hit ? 1 : 0;
  }
  if (t.i == 0) sin[(deg++) * T] = 0;
  return deg;
}

// Radius edge list export, compacted per env: every agent counts its partners j > i in range, publishes the count,
// an exclusive prefix sum over the env's agents gives its first pair slot; columns past the env's edge count are -1.
// Contains one block barrier: every thread of the CTA must call it.  `scnt` = int[T] scratch.
__device__ __forceinline__ void tile_write_edges_radius(const TileThread& t, const float4* pos, const float4& s, int N,
                                                        float qmax_r, int E, int32_t* eout, int32_t* counts, int* scnt) {
  const float2 neg = make_float2(-s.x, -s.y);
  const float4* env = pos + t.envbase;
  int mine = 0;
  if (t.active)
    for (int j = t.i + 1; j < N; ++j) mine += radius_hit(env, j, neg, qmax_r) ? 1 : 0;
  scnt[t.tid] = mine;
  __syncthreads();
  if (!t.active) return;
  int base = 0, total = 0;
  for (int a = 0; a < N; ++a) {
    const int c = scnt[t.envbase + a];
    base += (a < t.i) ? c : 0;
    total += c;
  }
  int32_t* r0 = eout + t.env * 2 * E;
  int32_t* r1 = r0 + E;
  for (int e = 2 * total + 1 + t.i; e < E; e += N) { r0[e] = -1; r1[e] = -1; }
  int slot = base;
  for (int j = t.i + 1; j < N; ++j) {
    if (radius_hit(env, j, neg, qmax_r)) {
      r0[2 * slot] = t.i; r1[2 * slot] = j;
      r0[2 * slot + 1] = j; r1[2 * slot + 1] = t.i;
      ++slot;
    }
  }
  if (t.i == 0) {
    r0[2 * total] = 0; r1[2 * total] = 0;
    if (counts) counts[t.env] = 2 * total + 1;
  }
}

// kNN rows (simulator.py:17-19): distance_to_i = ||x[:, :2] - x[i, :2]||, topk(k, largest=False) with
// torch's CPU tie order.  `pos` is the env-tile state buffer (float4 per thread).  Ends with a block barrier.
__device__ __forceinline__ void tile_knn_rows(const TileGraphSmem& g, const TileThread& t, const float4* pos,
                                              const float4& s, int N, int K) {
  const int T = kTileThreads;
  if (t.active) {
    SmemPairs row{g.skv + t.tid, g.ski + t.tid, T};
    for (int j = 0; j < N; ++j) {
      const float4 o = pos[t.envbase + j];
      KnnPair pr;
      pr.v = norm2(__fsub_rn(o.x, s.x), __fsub_rn(o.y, s.y));
      pr.i = j;
      row.set(j, pr);
    }
    // Fast path: K branch-free rounds of "smallest value above the previous pick" give the K smallest DISTINCT values
    // in ascending order.  If exactly K entries are <= the K-th value (no exact distance tie among the K smallest nor
    // at the K-th / (K+1)-th boundary) the result of *any* correct top-k is this list, so it equals torch.topk's.
    // Any tie (the rule on the regular start grids) or NaN falls back to the step-for-step libstdc++ emulation, whose
    // tie order is what torch produces.
    const float* __restrict__ kv = g.skv + t.tid;
    float prev = -INFINITY;
    for (int r = 0; r < K; ++r) {
      float best = INFINITY;
      int bi = 0;
#pragma unroll 4
      for (int l = 0; l < N; ++l) {
        const float v = kv[l * T];
        const float c = (v > prev) ? v : INFINITY;
        const bool lt = c < best;
        best = lt ? c : best;
        bi = lt ? l : bi;
      }
      g.snbr[r * T + t.tid] = (uint8_t)bi;
      prev = best;
    }
    int below = 0, nans = 0;
#pragma unroll 4
    for (int l = 0; l < N; ++l) {
      const float v = kv[l * T];
      below += (v <= prev) ? 1 : 0;
      nans += (v != v) ? 1 : 0;
    }
    const bool unique = (below == K) && (nans == 0) && (prev < INFINITY);
    if (!unique) {
      knn_topk_smallest(row, N, K);
      for (int r = 0; r < K; ++r) g.snbr[r * T + t.tid] = g.ski[r * T + t.tid];
    }
  }
  __syncthreads();
}

// in-edges of node d = i in edge-list order (simulator.py:20-24): for each row ii, slot r with
// a = topk[ii][r]: edge (ii -> a) then edge (a -> ii); finally (0 -> 0).
// The entries of one topk row are distinct, so a row ii != i sends at most ONE edge to i (when i is among its
// neighbours) while row i itself contributes, per slot, (i -> i) if a == i and then (a -> i).  Membership of i in
// the other rows is read from per-row bit masks (4 x 32 bits, N <= 128) published to shared memory, which turns the
// N x K scan per thread into N bit tests.  Contains two block barriers: every thread of the CTA must call it.
__device__ __forceinline__ int tile_in_edges_knn(const TileGraphSmem& g, const TileThread& t, int N, int K,
                                                 uint32_t* __restrict__ smask) {
  const int T = kTileThreads;
  const int words = (N + 31) >> 5;
  if (t.active) {
    uint32_t m[4] = {0u, 0u, 0u, 0u};
    for (int r = 0; r < K; ++r) {
      const int a = g.snbr[r * T + t.tid];
      m[0] |= (a < 32) ? (1u << a) : 0u;
      if (words > 1) {
        m[1] |= (a >= 32 && a < 64) ? (1u << (a - 32)) : 0u;
        m[2] |= (a >= 64 && a < 96) ? (1u << (a - 64)) : 0u;
        m[3] |= (a >= 96) ? (1u << (a - 96)) : 0u;
      }
    }
    for (int w = 0; w < words; ++w) smask[w * T + t.tid] = m[w];
  }
  __syncthreads();
  int deg = 0;
  if (t.active) {
    // Uniform control flow for the whole warp (every lane's own row sits at a different ii, so branching on
    // ii == i would make the warp run the K-slot loop in almost every iteration): one predicated pass over the
    // other rows, whose entries after row i are shifted by the size of the own block, then the own block.
    const int wi = t.i >> 5;
    const uint32_t bit = 1u << (t.i & 31);
    const uint32_t* __restrict__ col = smask + wi * T + t.envbase;
    uint8_t* __restrict__ sin = g.sin + t.tid;
    const uint8_t* __restrict__ nbr = g.snbr + t.tid;
    int own = K;
    for (int r = 0; r < K; ++r) own += (nbr[r * T] == t.i) ? 1 : 0;     // (i -> i) precedes (a -> i) when a == i
    int cnt = 0, lo = 0;
#pragma unroll 4
    for (int ii = 0; ii < N; ++ii) {
      const bool has = (ii != t.i) && (col[ii] & bit);
      lo = (ii == t.i) ? cnt : lo;
      if (has) sin[(cnt + (ii > t.i ? own : 0)) * T] = (uint8_t)ii;
      cnt += has ? 1 : 0;
    }
    int pos = lo;
    for (int r = 0; r < K; ++r) {
      const int a = nbr[r * T];
      if (a == t.i) sin[(pos++) * T] = (uint8_t)t.i;
      sin[(pos++) * T] = (uint8_t)a;
    }
    deg = cnt + own;
    if (t.i == 0) sin[(deg++) * T] = 0;
  }
  __syncthreads();            // smask may alias a buffer that is rewritten right after
  return deg;
}

// ---- small swarms (N <= 16): the kNN row lives in registers (knn_small.h) ------------------------------------------
constexpr int kKnnSmallMax = 16;

__device__ __forceinline__ int knn_nib(uint64_t w, int r) { return (int)((w >> (4 * r)) & 15u); }

// Row of this agent -> nibble word of its K neighbours in torch.topk's output order.  No shared-memory writes, no
// barrier.  (cache_rank, cache_nbr): the order pattern and answer of this thread's previous tie row -- on the start
// lattices the same pattern comes back tick after tick while the swarm moves in formation.
template <int NP>
__device__ __forceinline__ uint64_t tile_knn_small_np(const TileThread& t, const float4* pos, const float4& s, int N, int K,
                                                     uint64_t& cache_rank, uint64_t& cache_nbr) {
  uint32_t u[NP];
  const float4* env = pos + t.envbase;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    uint32_t key = kKnnPadKey;
    if (j < N) {
      const float2 o = xy_of(env[j]);
      key = knn_key_nonneg(norm2(__fsub_rn(o.x, s.x), __fsub_rn(o.y, s.y)));
    }
    u[j] = key;
  }
  int r[NP];
  uint32_t present;
  const uint64_t rank = knn_small_ranks<NP>(u, r, present);
  if (knn_small_tie_free(present, N, K)) return knn_small_by_rank<NP>(r, K);
  if (rank != cache_rank) {
    cache_nbr = knn_small_topk_fast(rank, N, K);
    cache_rank = rank;
  }
  return cache_nbr;
}

__device__ __forceinline__ uint64_t tile_knn_small(const TileThread& t, const float4* pos, const float4& s, int N, int K,
                                                  uint64_t& cache_rank, uint64_t& cache_nbr) {
  if (!t.active) return 0;
  if (N <= 8) return tile_knn_small_np<8>(t, pos, s, N, K, cache_rank, cache_nbr);
  if (N <= 12) return tile_knn_small_np<12>(t, pos, s, N, K, cache_rank, cache_nbr);
  return tile_knn_small_np<16>(t, pos, s, N, K, cache_rank, cache_nbr);
}

// ---- the SET of the K neighbours -----------------------------------------------------------------------------------
// The tensor-core Q forward consumes the kNN graph as in-edge multiplicities (tile_knn_counts_small): it needs WHICH K
// agents torch.topk returns, not in which order.  The set is unique unless a tie straddles the K boundary:
// S = {j : rank_j < K} always contains the K smallest, so |S| = K decides it without running any algorithm (ties inside
// the top K or beyond it -- the four equidistant lattice neighbours of an interior agent -- no longer matter; on C2
// rollouts 4.5 % of the rows are left instead of 10 %).  The remaining rows go through
//   1. the thread's previous boundary-tie row (cache_rank / cache_set: formation flight repeats its pattern),
//   2. a memo table in global memory shared by every CTA and launch (optional, caller-owned, swarms of <= 12 agents:
//      one 64-bit word per entry = 48-bit order pattern | 16-bit set, so a racing reader sees an old or a new entry,
//      never a torn one; direct-mapped, lossy; 95 % of the boundary-tie rows of a C2 rollout carry a pattern some env
//      has met before), and only then
//   3. the libstdc++ emulation (knn_small_topk_fast), whose answer is published to the table.
// The table belongs to ONE (n_agents, knn_k) pair: the order pattern does not encode them.
struct KnnMemo {
  unsigned long long* table;     // nullptr: no table
  uint32_t mask;                 // entries - 1 (power of two)
};

template <int NP>
__device__ __forceinline__ uint32_t tile_knn_small_set_np(const TileThread& t, const float4* pos, const float4& s, int N, int K,
                                                         uint64_t& cache_rank, uint64_t& cache_set, const KnnMemo& memo) {
  uint32_t u[NP];
  const float4* env = pos + t.envbase;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    uint32_t key = kKnnPadKey;
    if (j < N) {
      const float2 o = xy_of(env[j]);
      key = knn_key_nonneg(norm2(__fsub_rn(o.x, s.x), __fsub_rn(o.y, s.y)));
    }
    u[j] = key;
  }
  int r[NP];
  uint32_t present;
  const uint64_t rank = knn_small_ranks<NP>(u, r, present);
  uint32_t lt = 0;
#pragma unroll
  for (int j = 0; j < NP; ++j) lt |= (r[j] < K ? 1u : 0u) << j;     // padding ranks N >= K
  if (__popc(lt) == K) return lt;
  if (rank == cache_rank) return (uint32_t)cache_set;
  uint32_t set = 0;
  bool found = false;
  const bool use_table = NP <= 12 && memo.table != nullptr;
  unsigned long long* slot = nullptr;
  if (use_table) {
    slot = memo.table + ((uint32_t)((rank * 0x9E3779B97F4A7C15ull) >> 40) & memo.mask);
    const unsigned long long e = __ldcg(slot);
    if ((e >> 16) == rank && __popc((uint32_t)(e & 0xFFFFu)) == K) {
      set = (uint32_t)(e & 0xFFFFu);
      found = true;
    }
  }
  if (!found) {
    const uint64_t nbr = knn_small_topk_fast(rank, N, K);
    for (int q = 0; q < K; ++q) set |= 1u << knn_nib(nbr, q);
    if (use_table) __stcg(slot, (unsigned long long)((rank << 16) | set));
  }
  cache_rank = rank;
  cache_set = set;
  return set;
}

__device__ __forceinline__ uint32_t tile_knn_small_set(const TileThread& t, const float4* pos, const float4& s, int N, int K,
                                                      uint64_t& cache_rank, uint64_t& cache_set, const KnnMemo& memo) {
  if (!t.active) return 0;
  if (K >= N) return (1u << N) - 1u;                  // k = n (simulator.py:19 with 5 agents and k = 5): everybody
  if (N <= 8) return tile_knn_small_set_np<8>(t, pos, s, N, K, cache_rank, cache_set, memo);
  if (N <= 12) return tile_knn_small_set_np<12>(t, pos, s, N, K, cache_rank, cache_set, memo);
  return tile_knn_small_set_np<16>(t, pos, s, N, K, cache_rank, cache_set, memo);
}

// in-edges of node i from the neighbour words (same list, same order as tile_in_edges_knn): every thread publishes the
// 16-bit set of its row, one barrier, then N bit tests.  `smask` = uint32[T]; it is rewritten only after the barriers
// of the Q forward that follows, so no trailing barrier is needed.  Every thread of the CTA must call it.
__device__ __forceinline__ int tile_in_edges_knn_small(const TileGraphSmem& g, const TileThread& t, int N, int K, uint64_t nbr,
                                                       uint32_t* __restrict__ smask) {
  const int T = kTileThreads;
  uint32_t mine = 0;
  if (t.active)
    for (int r = 0; r < K; ++r) mine |= 1u << knn_nib(nbr, r);
  smask[t.tid] = mine;
  __syncthreads();
  int deg = 0;
  if (t.active) {
    const uint32_t* __restrict__ col = smask + t.envbase;
    uint8_t* __restrict__ sin = g.sin + t.tid;
    const int own = K + (int)((mine >> t.i) & 1u);      // (i -> i) precedes (a -> i) when a == i
    int cnt = 0, lo = 0;
#pragma unroll 4
    for (int ii = 0; ii < N; ++ii) {
      const bool has = (ii != t.i) && ((col[ii] >> t.i) & 1u);
      lo = (ii == t.i) ? cnt : lo;
      if (has) sin[(cnt + (ii > t.i ? own : 0)) * T] = (uint8_t)ii;
      cnt += has ? 1 : 0;
    }
    int pos = lo;
    for (int r = 0; r < K; ++r) {
      const int a = knn_nib(nbr, r);
      if (a == t.i) sin[(pos++) * T] = (uint8_t)t.i;
      sin[(pos++) * T] = (uint8_t)a;
    }
    deg = cnt + own;
    if (t.i == 0) sin[(deg++) * T] = 0;
  }
  return deg;
}

// Multiplicities of the in-edges of node i in the symmetrised kNN list (simulator.py:20-24), 2 bits per source j:
//   j != i:  [i in topk(j)] + [j in topk(i)]          (edge (j -> i) of row j, edge (j -> i) mirrored from row i)
//   j == i:  2 [i in topk(i)]                         (row i lists itself: (i -> i) and its mirror)   + 1 for node 0
// Every thread publishes the 16-bit set of its row, one barrier, then N bit tests.  Every thread of the CTA must call
// it; `smask` is rewritten only after the barriers of the Q forward that follows.
__device__ __forceinline__ uint32_t spread_bits16(uint32_t x) {       // bit j -> bit 2 j
  x = (x | (x << 8)) & 0x00FF00FFu;
  x = (x | (x << 4)) & 0x0F0F0F0Fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}
// (`mine` = the 16-bit set of this thread's row)
__device__ __forceinline__ uint32_t tile_knn_counts_small_set(const TileThread& t, int N, uint32_t mine,
                                                             uint32_t* __restrict__ smask);
__device__ __forceinline__ uint32_t tile_knn_counts_small(const TileThread& t, int N, int K, uint64_t nbr,
                                                         uint32_t* __restrict__ smask) {
  uint32_t mine = 0;
  if (t.active)
    for (int r = 0; r < K; ++r) mine |= 1u << knn_nib(nbr, r);
  return tile_knn_counts_small_set(t, N, mine, smask);
}
__device__ __forceinline__ uint32_t tile_knn_counts_small_set(const TileThread& t, int N, uint32_t mine,
                                                             uint32_t* __restrict__ smask) {
  smask[t.tid] = mine;
  __syncthreads();
  if (!t.active) return 0;
  const uint32_t* __restrict__ col = smask + t.envbase;
  uint32_t in = 0;
#pragma unroll 4
  for (int ii = 0; ii < N; ++ii) in |= ((col[ii] >> t.i) & 1u) << ii;
  in &= ~(1u << t.i);
  const uint32_t self2 = ((mine >> t.i) & 1u) << (2 * t.i);
  return spread_bits16(in) + spread_bits16(mine) + self2 + (t.i == 0 ? 1u : 0u);
}

// edge list export (env-local ids) in the reference's order
// (small swarms: `nbr_word` holds the neighbours, `use_word` = true)
__device__ __forceinline__ void tile_write_edges(const TileGraphSmem& g, const TileThread& t, int N, int K, bool knn,
                                                 int E, int32_t* eout, long long env_index, bool use_word = false,
                                                 uint64_t nbr_word = 0) {
  const int T = kTileThreads;
  int32_t* r0 = eout + env_index * 2 * E;
  int32_t* r1 = r0 + E;
  const int i = t.i;
  if (knn) {
    for (int r = 0; r < K; ++r) {
      const int a = use_word ? knn_nib(nbr_word, r) : (int)g.snbr[r * T + t.tid];
      const int e = (i * K + r) * 2;
      r0[e] = i; r1[e] = a;
      r0[e + 1] = a; r1[e + 1] = i;
    }
  } else {
    for (int j = i + 1; j < N; ++j) {
      const int e = 2 * (i * N - (i * (i + 1)) / 2 + (j - i - 1));
      r0[e] = i; r1[e] = j;
      r0[e + 1] = j; r1[e + 1] = i;
    }
  }
  if (i == 0) { r0[E - 1] = 0; r1[E - 1] = 0; }
}

// Publishes this node's projected features h and alpha_src to the tile (read by its neighbours).
__device__ __forceinline__ void tile_gat_publish(const TileGraphSmem& g, const TileThread& t, const float (&h)[32],
                                                 float asrc) {
  float4* hrow = reinterpret_cast<float4*>(g.sh + t.tid * kHPad);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) hrow[c4] = make_float4(h[4 * c4], h[4 * c4 + 1], h[4 * c4 + 2], h[4 * c4 + 3]);
  g.sas[t.tid] = asrc;
}

// Edge softmax over the in-edge list of this node in edge-list order (torch_geometric.utils.softmax: max,
// exp(z - max), sum + 1e-16, divide) followed by the aggregation.  On return agg = sum_e alpha_e h_j (bias not yet
// added); the parity path (FUSED = false) also leaves the attention coefficients alpha_e in g.swt[e][tid], which no
// caller reads.
template <bool FUSED = false>
__device__ __forceinline__ void tile_gat_attend(const TileGraphSmem& g, const TileThread& t, int deg, float adst,
                                                float (&agg)[32]) {
  const int T = kTileThreads;
#pragma unroll
  for (int cc = 0; cc < 32; ++cc) agg[cc] = 0.0f;
  if (t.active) {
    const uint8_t* __restrict__ sin = g.sin + t.tid;
    float* __restrict__ swt = g.swt + t.tid;
    const float* __restrict__ sas = g.sas + t.envbase;
    const float* __restrict__ shb = g.sh + t.envbase * kHPad;
    float m = -INFINITY;
#pragma unroll 4
    for (int e = 0; e < deg; ++e) {
      const float z = gat_logit(sas[sin[e * T]], adst);
      swt[e * T] = z;
      m = fmaxf(m, z);
    }
    if (FUSED) {
      // tensor-core path (activations feed a 3xTF32 contraction anyway): ONE more sweep computes the unnormalised
      // weights exp(z - max), their sum and the aggregation; the division by the sum is applied once to the 32
      // channels at the end.  Two edges per iteration, all 16 row loads issued before the 32 packed FFMAs, so the
      // shared-memory latency of one edge hides behind the other's math.
      float den = 0.0f;
      int e = 0;
      for (; e + 2 <= deg; e += 2) {
        const float4* __restrict__ r0 = reinterpret_cast<const float4*>(shb + sin[e * T] * kHPad);
        const float4* __restrict__ r1 = reinterpret_cast<const float4*>(shb + sin[(e + 1) * T] * kHPad);
        const float w0 = __expf(swt[e * T] - m), w1 = __expf(swt[(e + 1) * T] - m);
        float4 v0[8], v1[8];
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) { v0[c4] = r0[c4]; v1[c4] = r1[c4]; }
        den = __fadd_rn(__fadd_rn(den, w0), w1);
        gat_accumulate_regs(agg, w0, v0);
        gat_accumulate_regs(agg, w1, v1);
      }
      if (e < deg) {
        const float w0 = __expf(swt[e * T] - m);
        den = __fadd_rn(den, w0);
        gat_accumulate<true>(agg, w0, reinterpret_cast<const float4*>(shb + sin[e * T] * kHPad));
      }
      const float inv = 1.0f / __fadd_rn(den, 1e-16f);
      const float2 i2 = make_float2(inv, inv);
#pragma unroll
      for (int c2 = 0; c2 < 16; ++c2) {
        const float2 r = __fmul2_rn(make_float2(agg[2 * c2], agg[2 * c2 + 1]), i2);
        agg[2 * c2] = r.x;
        agg[2 * c2 + 1] = r.y;
      }
    } else {
      float den = 0.0f;
#pragma unroll 4
      for (int e = 0; e < deg; ++e) {
        const float w = expf(__fsub_rn(swt[e * T], m));
        swt[e * T] = w;
        den = __fadd_rn(den, w);
      }
      den = __fadd_rn(den, 1e-16f);
      for (int e = 0; e < deg; ++e) {
        const int j = sin[e * T];
        const float alpha = __fdiv_rn(swt[e * T], den);
        swt[e * T] = alpha;
        gat_accumulate<false>(agg, alpha, reinterpret_cast<const float4*>(shb + j * kHPad));
      }
    }
  }
}

// GATConv forward for the node of this thread (CUDA-core projection): projects x, publishes (h, alpha_src),
// one block barrier, then attention + aggregation.  adst is this node's alpha_dst.
__device__ __forceinline__ void tile_gat_conv(const TileGraphSmem& g, const TileThread& t, const float* sw,
                                              const float (&x)[7], int deg, float (&agg)[32], float& adst) {
  adst = 0.0f;
  if (t.active) {
    float h[32];
    float asrc;
    gat_project(x, sw, h, asrc, adst);
    tile_gat_publish(g, t, h, asrc);
  }
  __syncthreads();
  tile_gat_attend(g, t, deg, adst, agg);
}

// counter-based RNG for device-side exploration (documented deviation from the reference's Python
// Mersenne stream, train:164-165; parity tests inject the action stream instead)
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ uint64_t rng_draw(uint64_t seed, uint64_t env, uint64_t tick, uint32_t lane) {
  return splitmix64(splitmix64(seed ^ (env * 0xD1342543DE82EF95ull)) ^ (tick * 0xA24BAED4963EE407ull) ^ lane);
}

}  // namespace swarm
#endif
