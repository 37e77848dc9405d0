// tile_kernels.cuh -- parameter block + shared-memory layout of the "env tile" kernel family
// (one thread per agent, floor(threads / N) whole envs per CTA, N <= 128).
#ifndef SWARM_TILE_KERNELS_CUH
#define SWARM_TILE_KERNELS_CUH

#include "swarm_device.cuh"

namespace swarm {

constexpr int kTileThreads = 128;
constexpr int kHPad = 36;        // padded row of the hidden tile (floats); keeps float4 alignment, spreads banks
constexpr int kW2Pad = 12;       // lin2 rows padded 9 -> 12 so a k-slice is three float4

// kernel-side weight layout in shared memory (k-major = transposed, so one float4 feeds 4 output channels)
enum {
  TW_W0T = 0,                      // [7][32]
  TW_ATT_S = TW_W0T + 7 * 32,      // [32]
  TW_ATT_D = TW_ATT_S + 32,        // [32]
  TW_B0 = TW_ATT_D + 32,           // [32]
  TW_W1T = TW_B0 + 32,             // [32][32]
  TW_B1 = TW_W1T + 32 * 32,        // [32]
  TW_W2T = TW_B1 + 32,             // [32][12]
  TW_B2 = TW_W2T + 32 * kW2Pad,    // [12]
  TW_COUNT = TW_B2 + kW2Pad
};

// global packed weights (state-dict order) -> shared, transposed to k-major.
// The packed array is read in its own order, four floats at a time (every tensor starts at a multiple of four floats),
// with all of a thread's loads issued before the first store: one coalesced round trip to L2 instead of fourteen
// dependent scalar ones (this prologue was the largest exposed latency of the small-batch DQN gradient kernel).
__device__ __forceinline__ void stage_weight_value(float* __restrict__ s, int o, float v) {
  if (o < SWARM_W_ATT_SRC) {                    // conv1.lin.weight[c][k] -> W0T[k][c]
    const int c = o / 7, k = o - c * 7;
    s[TW_W0T + k * 32 + c] = v;
  } else if (o < SWARM_W_LIN1) {                // att_src, att_dst, conv1.bias keep their order
    s[TW_ATT_S + (o - SWARM_W_ATT_SRC)] = v;
  } else if (o < SWARM_W_LIN1_BIAS) {           // lin1.weight[c][k] -> W1T[k][c]
    const int r = o - SWARM_W_LIN1, c = r >> 5, k = r & 31;
    s[TW_W1T + k * 32 + c] = v;
  } else if (o < SWARM_W_LIN2) {
    s[TW_B1 + (o - SWARM_W_LIN1_BIAS)] = v;
  } else if (o < SWARM_W_LIN2_BIAS) {           // lin2.weight[a][k] -> W2T[k][a], a padded to 12
    const int r = o - SWARM_W_LIN2, a = r >> 5, k = r & 31;
    s[TW_W2T + k * kW2Pad + a] = v;
  } else if (o < SWARM_W_COUNT) {
    s[TW_B2 + (o - SWARM_W_LIN2_BIAS)] = v;
  }
}

__device__ __forceinline__ void stage_weights(const float* __restrict__ g, float* __restrict__ s, int tid, int nthreads) {
  static_assert(TW_ATT_D == TW_ATT_S + 32 && TW_B0 == TW_ATT_D + 32, "attention vectors and conv bias are contiguous");
  constexpr int kChunks = SWARM_W_COUNT / 4;                 // 418 whole float4 chunks + one scalar tail
  if ((reinterpret_cast<uintptr_t>(g) & 15u) == 0 && nthreads >= 128) {
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int ch = tid + k * nthreads;
      v[k] = ch < kChunks ? reinterpret_cast<const float4*>(g)[ch] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float tail = (tid == 0) ? g[SWARM_W_COUNT - 1] : 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int ch = tid + k * nthreads;
      if (ch < kChunks) {
        stage_weight_value(s, 4 * ch + 0, v[k].x);
        stage_weight_value(s, 4 * ch + 1, v[k].y);
        stage_weight_value(s, 4 * ch + 2, v[k].z);
        stage_weight_value(s, 4 * ch + 3, v[k].w);
      }
    }
    if (tid == 0) stage_weight_value(s, SWARM_W_COUNT - 1, tail);
  } else {
    for (int o = tid; o < SWARM_W_COUNT; o += nthreads) stage_weight_value(s, o, g[o]);
  }
  // zero padding of the lin2 rows / bias (a = 9 .. 11)
  for (int idx = tid; idx < 32 * 3 + 3; idx += nthreads) {
    if (idx < 96) s[TW_W2T + (idx / 3) * kW2Pad + 9 + idx % 3] = 0.0f;
    else s[TW_B2 + 9 + (idx - 96)] = 0.0f;
  }
}

enum TileMode { MODE_ROLLOUT = 0, MODE_FORWARD = 1, MODE_GRAPH = 3 };

struct TileParams {
  SwarmConfig cfg;
  const float* weights;          // packed state-dict order (SWARM_W_*)
  const float* state_in;
  float* state_out;
  const int32_t* actions_in;     // MODE_ROLLOUT: optional forced actions [ticks][B*N]
  float* returns;                // MODE_ROLLOUT: [B*N] +=
  int32_t* hits;                 // MODE_ROLLOUT: [B] +=
  SwarmTrace trace;              // MODE_ROLLOUT, optional
  float* q_out;                  // MODE_FORWARD
  int32_t* act_out;              // MODE_FORWARD
  int32_t* edges_out;            // MODE_GRAPH
  int32_t* nbr_out;              // MODE_GRAPH
  SwarmReplay replay;            // MODE_ROLLOUT, optional (state == nullptr: no push)
  const SwarmTrainCtl* ctl;      // MODE_ROLLOUT, optional: tick number / ring cursor / epsilon come from device memory
  long long replay_cursor;
  long long env_offset;
  unsigned long long rng_seed;
  long long rng_tick0;
  float epsilon;
  int32_t use_tc;                // 1: dense contractions on the tensor cores (tcgen05, 3xTF32)
  int32_t ticks;
  int32_t epb;                   // envs per block (capacity of a CTA)
  int32_t bal_q, bal_r;          // balanced assignment (bal_q > 0): CTA b owns bal_q + (b < bal_r) envs from
                                 // b * bal_q + min(b, bal_r) on -- a single-wave grid spread evenly over every CTA slot
  int32_t maxdeg;                // max in-degree of the graph (rows of the per-thread edge scratch)
  int32_t edges_per_env;
  WorldConsts world;
  float qmax_r;                  // largest q with sqrt(q) <= graph_radius (radius graph)
  int32_t* counts_out;           // MODE_GRAPH, radius graph: edges per env
  // MODE_ROLLOUT, FLOCK variant: the Flocking reward (flocking_scenario.py:124-171) instead of GoTo's on the GoTo world
  SwarmRewardSpec flock;         // its constants
  float2* shaping;               // [B*N] (previous_distance_to_goal, previous_distance_to_agents), read at launch, written back
  int32_t use_flock;
  // kNN rows of small swarms on the tensor-core path (tile_device.cuh): optional memo table of boundary-tie patterns
  unsigned long long* knn_memo;
  uint32_t knn_memo_mask;        // entries - 1
  int32_t knn_ordered;           // 1: always run the ordered (torch.topk output order) row code (SWARM_KNN_ORDERED=1)
};

// byte offsets of the dynamic shared memory regions
struct TileLayout {
  int w, st, h, asrc, wt, inl, deg, kv, ki, nbr, red, tc_w0, tc_w1, tc_w2, tc_vec, tc_bar, stage, total;
};

__host__ __device__ inline int tile_align16(int x) { return (x + 15) & ~15; }
__host__ __device__ inline int tile_align128(int x) { return (x + 127) & ~127; }

__host__ __device__ inline TileLayout tile_layout(int mode, int threads, int n, int k, int maxdeg, int graph_mode,
                                                  bool tc = false) {
  TileLayout L;
  int off = 0;
  const bool q = (mode == MODE_ROLLOUT || mode == MODE_FORWARD);
  const bool knn = (graph_mode == SWARM_GRAPH_KNN) && (q || mode == MODE_GRAPH);
  tc = tc && q;
  // tensor-core B operand tiles (weights) first (128-byte aligned); the A operand lives in tensor memory
  L.tc_w0 = off;  off = tile_align128(off + (tc ? 2 * 32 * 8 * 4 : 0));
  L.tc_w1 = off;  off = tile_align128(off + (tc ? 2 * 32 * 32 * 4 : 0));
  L.tc_w2 = off;  off = tile_align128(off + (tc ? 2 * 16 * 32 * 4 : 0));
  L.tc_vec = off; off = tile_align16(off + (tc ? 96 * 4 : 0));
  L.tc_bar = off; off = tile_align16(off + (tc ? 16 : 0));
  L.w = off;    off = tile_align16(off + ((q && !tc) ? TW_COUNT * 4 : 0));
  L.st = off;   off = tile_align16(off + 2 * threads * 16);
  // the tensor-core path attends in input space (tile_tc_device.cuh): no tile of projected features, no per-edge
  // scratch, and no edge list for the complete graph
  // (nor for kNN swarms of n <= 16, whose in-edges are multiplicity words in registers)
  const bool tc_complete = tc && (graph_mode == SWARM_GRAPH_COMPLETE || (graph_mode == SWARM_GRAPH_KNN && n <= 16));
  L.h = off;    off = tile_align16(off + ((q && !tc) ? threads * kHPad * 4 : 0));
  L.asrc = off; off = tile_align16(off + (q ? threads * 4 : 0));
  L.wt = off;   off = tile_align16(off + ((q && !tc) ? maxdeg * threads * 4 : 0));
  L.inl = off;  off = tile_align16(off + ((q && !tc_complete) ? maxdeg * threads : 0));
  L.deg = off;  off = tile_align16(off + (q ? threads : 0));
  // kNN rows: swarms of n <= 16 keep them in registers (knn_small.h) and only publish one membership word per thread
  const bool knn_rows = knn && n > 16;
  L.kv = off;   off = tile_align16(off + (knn ? (knn_rows ? n : 1) * threads * 4 : 0));
  L.ki = off;   off = tile_align16(off + (knn_rows ? n * threads : 0));
  L.nbr = off;  off = tile_align16(off + (knn_rows ? k * threads : 0));
  L.red = off;  off = tile_align16(off + threads * 4);
  // MODE_GRAPH: the tile's edge lists are staged here and written out with coalesced stores (0 = does not fit)
  {
    const long long e = (graph_mode == SWARM_GRAPH_KNN) ? (2LL * k * n + 1) : ((long long)n * (n - 1) + 1);
    const long long bytes = (long long)(threads / n) * 2 * e * 4;
    const bool staged = (mode == MODE_GRAPH) && (off + bytes <= 160 * 1024);
    L.stage = staged ? off : 0;
    if (staged) off = tile_align16(off + (int)bytes);
  }
  L.total = off;
  return L;
}

}  // namespace swarm
#endif
