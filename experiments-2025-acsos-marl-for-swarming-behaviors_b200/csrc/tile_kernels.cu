// tile_kernels.cu -- the env-tile kernel family for swarms of N <= 128 agents.
//
// One thread owns one agent; a CTA of 128 threads owns floor(128 / N) whole envs, so everything an
// agent needs from its swarm (partner positions, projected features, attention terms, kNN rows) is
// exchanged through shared memory and no env ever straddles a CTA.  The same device code is
// instantiated in three modes:
//   MODE_ROLLOUT  T x [graph -> GAT-Q -> (eps-)greedy -> world step (-> replay push)], state resident in
//                 registers (simulator.py:59-93 / train_gcn_dqn.py:153-178 inner loops)
//   MODE_FORWARD  graph -> GAT-Q (-> argmax) once                         (train_gcn_dqn.py:59-70)
//   MODE_GRAPH    edge list / neighbour table export                      (train:94-110, simulator:9-26)
// so the stand-alone kernels and the fused rollout are consistent by construction.  The rollout's world step is the
// agent_step of swarm_device.cuh, which the stand-alone world-step kernels (step_kernels.cu) run as well.
#include "tile_tc_device.cuh"
#include "launchers.h"

namespace swarm {

// DENSE: register budget for four resident CTAs per SM (127 registers) instead of three (156).  The tensor-core modes
// are built both ways: with more CTAs than 3 x 148 the fourth CTA per SM pays (+13 % at 65 536 envs), below that the
// roomier allocation is the faster one (C2: 410 CTAs).
// FLOCK (MODE_ROLLOUT only): the world is GoTo's, the reward is FlockingScenario's collective reward, evaluated with the
// op sequence of reward_kernels.cu on the post-step positions; the two shaping terms of the agent live in registers
// across the ticks like its state.  A separate template value so that the GoTo / ObstacleAvoidance instantiations keep
// their code byte for byte.
// NT: swarm size as a compile-time constant (0 = the run-time value): index arithmetic, attention loops and the partner
// sweep of the shapes the reference's experiments use unroll completely (the streaming world step gained 25-40 % from
// the same specialisation).
// PLAIN (MODE_ROLLOUT, TC only): the greedy evaluation rollout -- complete graph, no trace, no replay push, no forced
// actions, no device-side control block, epsilon 0 (launch_tile_q checks all of it).  The kNN / radius paths, the
// other attention heads and every per-tick test of an optional pointer are compiled out, which leaves the tick a
// straight line of about a quarter of the generic kernel's code.  Same arithmetic, same bits.
template <int MODE, bool TC, bool DENSE, bool FLOCK = false, int NT = 0, bool PLAIN = false>
__global__ void __launch_bounds__(kTileThreads, MODE == MODE_GRAPH ? 8 : ((TC && !DENSE) ? 3 : 4))
tile_kernel(const __grid_constant__ TileParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr bool kQ = (MODE == MODE_ROLLOUT || MODE == MODE_FORWARD);
  constexpr bool kGraphOut = (MODE == MODE_GRAPH || MODE == MODE_ROLLOUT);

  const SwarmConfig& c = p.cfg;
  const int T = kTileThreads;
  const int N = NT > 0 ? NT : c.n_agents;
  static_assert(!PLAIN || (MODE == MODE_ROLLOUT && TC && !FLOCK), "PLAIN is the tensor-core greedy rollout");
  const int K = c.knn_k;
  const bool knn = !PLAIN && (c.graph_mode == SWARM_GRAPH_KNN) && (kQ || MODE == MODE_GRAPH);
  const bool radius = !PLAIN && (c.graph_mode == SWARM_GRAPH_RADIUS) && (kQ || MODE == MODE_GRAPH);
  const TileThread t = tile_thread(N, p.epb, c.num_envs, p.bal_q, p.bal_r);
  const int tid = t.tid;
  const long long BN = (long long)c.num_envs * N;

  const TileLayout L = tile_layout(MODE, T, N, K, p.maxdeg, c.graph_mode, TC);
  float* sw = reinterpret_cast<float*>(smem + L.w);
  float4* sst = reinterpret_cast<float4*>(smem + L.st);
  float* sred = reinterpret_cast<float*>(smem + L.red);
  TileGraphSmem g;
  g.sh = reinterpret_cast<float*>(smem + L.h);
  g.sas = reinterpret_cast<float*>(smem + L.asrc);
  g.swt = reinterpret_cast<float*>(smem + L.wt);
  g.sin = smem + L.inl;
  g.skv = reinterpret_cast<float*>(smem + L.kv);
  g.ski = smem + L.ki;
  g.snbr = smem + L.nbr;

  // this agent's state, running return and the tick-dependent scalars: global loads issued before the weights are
  // staged, so their latency overlaps the staging round trip (a single-tick launch is mostly prologue)
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  float ret0 = 0.0f;
  if (t.active) {
    s = reinterpret_cast<const float4*>(p.state_in)[t.gidx];
    if (MODE == MODE_ROLLOUT && p.returns) ret0 = p.returns[t.gidx];
  }
  float2 shp = make_float2(0.0f, 0.0f);      // FLOCK: (previous_distance_to_goal, previous_distance_to_agents)
  if (FLOCK && t.active) shp = p.shaping[t.gidx];
  float epsilon = p.epsilon;
  long long rng_tick0 = p.rng_tick0, replay_cursor = p.replay_cursor;
  if (MODE == MODE_ROLLOUT && !PLAIN && p.ctl) {
    epsilon = p.ctl->epsilon;
    rng_tick0 = p.ctl->tick + 1;
    replay_cursor = p.ctl->ring_cursor;
  }

  TileTcSmem ts;
  uint32_t tmem = 0, parity = 0;
  if (TC) {
    ts.w0 = smem + L.tc_w0;
    ts.w1 = smem + L.tc_w1;
    ts.w2 = smem + L.tc_w2;
    ts.vec = reinterpret_cast<float*>(smem + L.tc_vec);
    ts.bar = reinterpret_cast<uint64_t*>(smem + L.tc_bar);
    ts.tmem_slot = reinterpret_cast<uint32_t*>(smem + L.tc_bar + 8);
    stage_weights_tc(p.weights, ts, tid, T);
    if (tid == 0) tc::mbar_init(ts.bar, 1);
    if ((tid >> 5) == 0) tc::tmem_alloc(ts.tmem_slot, kTmemCols);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    tmem = *ts.tmem_slot;
  } else if (kQ) {
    stage_weights(p.weights, sw, tid, T);
  }


  int deg = 0;
  const bool complete = !knn && !radius;
  if (kQ && !TC && complete && t.active) deg = tile_in_edges_complete(g, t, N);   // the TC path needs no edge list for it
  const bool knn_small = knn && N <= kKnnSmallMax;          // register-resident rows (knn_small.h)
  uint64_t nbr_word = 0, knn_cache_rank = ~0ull, knn_cache_nbr = 0;
  // order-free kNN: nobody reads the neighbours' ORDER (no edge export) and the forward takes multiplicities
  const bool knn_set = knn_small && TC && kQ && !(MODE == MODE_ROLLOUT && p.trace.edges) && !p.knn_ordered;
  const KnnMemo knn_memo{p.knn_memo, p.knn_memo_mask};

  float ret = 0.0f;
  int myhits = 0;

  SWARM_PHASE_RESET();
  for (int tick = 0; tick < p.ticks; ++tick) {
    SWARM_PHASE_START();
    const float4* pos = sst + (tick & 1) * T;
    sst[(tick & 1) * T + tid] = s;
    float adst_tc = 0.0f;
    if (TC && kQ) {
      // attention terms straight from the input features (tile_tc_device.cuh): published with the state
      const float x[7] = {s.x, s.y, s.z, s.w, c.goal_x, c.goal_y, (float)t.i};
      float asrc;
      tc_alpha_terms(ts, x, asrc, adst_tc);
      g.sas[tid] = asrc;
    }
    __syncthreads();
    SWARM_PHASE(PH_PUBLISH);

    int action = 0;

    // ------------------------------------------------------------------ graph ----------------
    uint32_t knn_counts = 0;
    if (knn_small && knn_set) {
      // the tensor-core forward needs the SET of the K neighbours only (tile_device.cuh)
      const uint32_t mine = tile_knn_small_set(t, pos, s, N, K, knn_cache_rank, knn_cache_nbr, knn_memo);
      knn_counts = tile_knn_counts_small_set(t, N, mine, reinterpret_cast<uint32_t*>(g.skv));
    } else if (knn_small) {
      nbr_word = tile_knn_small(t, pos, s, N, K, knn_cache_rank, knn_cache_nbr);
      if (kQ && TC) knn_counts = tile_knn_counts_small(t, N, K, nbr_word, reinterpret_cast<uint32_t*>(g.skv));
      else if (kQ) deg = tile_in_edges_knn_small(g, t, N, K, nbr_word, reinterpret_cast<uint32_t*>(g.skv));
    } else if (knn) {
      tile_knn_rows(g, t, pos, s, N, K);
      if (kQ) deg = tile_in_edges_knn(g, t, N, K, reinterpret_cast<uint32_t*>(g.skv));   // distance rows are dead now
    }
    if (radius && kQ && t.active) deg = tile_in_edges_radius(g, t, pos, s, N, p.qmax_r);
    if (MODE == MODE_GRAPH && radius) {
      tile_write_edges_radius(t, pos, s, N, p.qmax_r, p.edges_per_env, p.edges_out, p.counts_out, reinterpret_cast<int*>(sred));
    } else if (kGraphOut && !PLAIN) {
      int32_t* eout = nullptr;
      if (MODE == MODE_GRAPH) eout = p.edges_out;
      else if (p.trace.edges) eout = p.trace.edges + (long long)tick * c.num_envs * 2 * p.edges_per_env;
      if (MODE == MODE_GRAPH && eout && L.stage) {
        // stage the tile's edge lists in shared memory, then stream the contiguous [envs][2][E] block out with
        // coalesced 8-byte stores (E is odd, so the block is only 8-byte aligned)
        int32_t* stage = reinterpret_cast<int32_t*>(smem + L.stage);
        if (t.active) tile_write_edges(g, t, N, K, knn, p.edges_per_env, stage, t.el, knn_small, nbr_word);
        __syncthreads();
        const long long env0 = (long long)blockIdx.x * p.epb;
        const long long envs_here = (c.num_envs - env0 < p.epb) ? (c.num_envs - env0) : p.epb;
        const long long words = envs_here * 2 * p.edges_per_env;
        int32_t* dst = eout + env0 * 2 * p.edges_per_env;
        const long long pairs = words >> 1;
        for (long long w = tid; w < pairs; w += T) reinterpret_cast<int2*>(dst)[w] = reinterpret_cast<const int2*>(stage)[w];
        if ((words & 1) && tid == 0) dst[words - 1] = stage[words - 1];
      } else if (eout && t.active) {
        tile_write_edges(g, t, N, K, knn, p.edges_per_env, eout, t.env, knn_small, nbr_word);
      }
      if (MODE == MODE_GRAPH && knn && p.nbr_out && t.active)
        for (int r = 0; r < K; ++r) p.nbr_out[t.gidx * K + r] = knn_small ? knn_nib(nbr_word, r) : (int)g.snbr[r * T + tid];
    }

    // ------------------------------------------------------------------ GAT-Q forward --------
    if (kQ) {
      // node features (train:95-99): [pos, vel, goal, agent id]
      float q[9];
      if (TC) {
        if (complete)
          action = tile_q_forward_tc<ATT_COMPLETE, NT>(g, ts, t, tmem, pos, N, deg, 0u, adst_tc, c.goal_x, c.goal_y, parity, q);
        else if (knn_small)
          action = tile_q_forward_tc<ATT_COUNTS>(g, ts, t, tmem, pos, N, deg, knn_counts, adst_tc, c.goal_x, c.goal_y, parity, q);
        else
          action = tile_q_forward_tc<ATT_LIST>(g, ts, t, tmem, pos, N, deg, 0u, adst_tc, c.goal_x, c.goal_y, parity, q);
      } else {
        const float x[7] = {s.x, s.y, s.z, s.w, c.goal_x, c.goal_y, (float)t.i};
        float a1[32];
        float adst;
        tile_gat_conv(g, t, sw, x, deg, a1, adst);
        if (t.active) action = gat_head(a1, sw, q);
      }
      if (t.active) {
        if (MODE == MODE_FORWARD) {
          if (p.q_out) {
#pragma unroll
            for (int a = 0; a < 9; ++a) p.q_out[t.gidx * 9 + a] = q[a];
          }
          if (p.act_out) p.act_out[t.gidx] = action;
        } else if (!PLAIN && p.trace.q) {
          float* tq = p.trace.q + ((long long)tick * BN + t.gidx) * 9;
#pragma unroll
          for (int a = 0; a < 9; ++a) tq[a] = q[a];
        }
      }
    }

    // ------------------------------------------------------------------ world step ------------
    if (MODE == MODE_ROLLOUT) {
      float reward = 0.0f;
      if (t.active) {
        if (!PLAIN) {
          if (epsilon > 0.0f) {
            // train:164-165: one coin per tick for the whole swarm, then one uniform action per agent
            const unsigned long long genv = (unsigned long long)(p.env_offset + t.env);
            const unsigned long long gt = (unsigned long long)(rng_tick0 + tick);
            const float coin = (float)(rng_draw(p.rng_seed, genv, gt, 0xFFFFu) >> 40) * (1.0f / 16777216.0f);
            if (coin < epsilon) action = (int)(((rng_draw(p.rng_seed, genv, gt, (uint32_t)t.i) >> 32) * 9ull) >> 32);
          }
          if (p.actions_in) {
            const int fa = p.actions_in[(long long)tick * BN + t.gidx];
            if (fa >= 0) action = fa;
          }
        }
        const float4 s_prev = s;
        const bool oa = c.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE;
        uint8_t flags = 0;
        uint32_t cmask = 0;
        float2 u;
        decode_action(action, u.x, u.y);
        agent_step(s, u, pos + t.envbase, N, t.i, oa, c, p.world, flags, cmask);

        float dgoal, dobs;
        reward = post_step_reward(s, oa, c, dgoal, dobs, flags);
        if (oa) myhits += (flags & SWARM_FLAG_HIT) ? 1 : 0;
        else if (!FLOCK) sred[tid] = dgoal;     // GoTo's collective reward needs every agent's distance: finished below
        if (!PLAIN) {
          const long long tb = (long long)tick * BN + t.gidx;
          if (p.trace.state) reinterpret_cast<float4*>(p.trace.state)[tb] = s;
          if (p.trace.actions) p.trace.actions[tb] = action;
          if (p.trace.flags) p.trace.flags[tb] = flags;
          if (p.trace.contact) p.trace.contact[tb] = cmask;
          if (p.trace.dist) reinterpret_cast<float2*>(p.trace.dist)[tb] = make_float2(dgoal, dobs);
          if (p.replay.state) {
            // GraphReplayBuffer.push (train:171-172), state-only transition
            const long long slot = (replay_cursor + (long long)tick * c.num_envs + t.env) % p.replay.capacity;
            const long long ri = slot * N + t.i;
            reinterpret_cast<float4*>(p.replay.state)[ri] = s_prev;
            reinterpret_cast<float4*>(p.replay.next_state)[ri] = s;
            p.replay.actions[ri] = (uint8_t)sanitize_action(action);
          }
        }
      }
      if (FLOCK) {
        // Flocking (flocking:124-171): every agent's term from the POST-step positions of its env, then the collective
        // sum in agent order.  The post-step states go into the state buffer the next tick will fill anyway.
        const SwarmRewardSpec& fs = p.flock;
        float4* post = sst + ((tick + 1) & 1) * T;
        post[tid] = s;
        __syncthreads();
        float term = 0.0f;
        if (t.active) {
          const float d_goal = norm2(__fsub_rn(s.x, fs.goal_x), __fsub_rn(s.y, fs.goal_y));
          const float shaped_goal = __fmul_rn(d_goal, fs.pos_shaping);
          const float4* others = post + t.envbase;
          float sum;
          int close;
          flocking_partner_sweep(s.x, s.y, t.i, N, [&](int j) { return xy_of(others[j]); }, fs.desired_distance,
                                 fs.agent_radius, fs.min_collision_distance, sum, close);
          const float spacing = __fmul_rn(__fdiv_rn(sum, (float)(N - 1)), fs.dist_shaping);
          const float pos_rew = __fsub_rn(shp.x, shaped_goal);
          float r = pos_rew;
          if (d_goal < fs.goal_radius) r = __fadd_rn(r, fs.on_goal_bonus);
          const float avoid = close ? __fmul_rn((float)close, fs.collision_reward) : 0.0f;
          const float dist_rew = __fsub_rn(shp.y, spacing);
          shp = make_float2(shaped_goal, spacing);
          term = __fadd_rn(__fadd_rn(r, avoid), dist_rew);
        }
        sred[tid] = term;
        __syncthreads();
        if (t.active)
          for (int a = 0; a < N; ++a) reward = __fadd_rn(reward, sred[t.envbase + a]);
      } else if (c.scenario == SWARM_SCENARIO_GOTO) {
        // collective reward (go_to:108-115): 0 + (-d_0) + (-d_1) + ... in agent order, same for all agents
        __syncthreads();
        if (t.active)
          for (int a = 0; a < N; ++a) reward = __fadd_rn(reward, -sred[t.envbase + a]);
      }
      if (t.active) {
        ret = __fadd_rn(ret, reward);
        if (!PLAIN) {
          if (p.trace.rewards) p.trace.rewards[(long long)tick * BN + t.gidx] = reward;
          if (p.replay.state) {
            const long long slot = (replay_cursor + (long long)tick * c.num_envs + t.env) % p.replay.capacity;
            p.replay.rewards[slot * N + t.i] = reward;
          }
        }
      }
    }
    SWARM_PHASE(PH_WORLD);
  }
  SWARM_PHASE_FLUSH();

  if (MODE == MODE_ROLLOUT) {
    if (t.active) {
      reinterpret_cast<float4*>(p.state_out)[t.gidx] = s;
      if (p.returns) p.returns[t.gidx] = __fadd_rn(ret0, ret);
      if (FLOCK) p.shaping[t.gidx] = shp;
    }
    if (p.hits) {
      __syncthreads();
      reinterpret_cast<int*>(sred)[tid] = myhits;
      __syncthreads();
      if (t.active && t.i == 0) {
        int tot = 0;
        for (int a = 0; a < N; ++a) tot += reinterpret_cast<int*>(sred)[t.envbase + a];
        p.hits[t.env] += tot;
      }
    }
  }
  if (TC) {
    tc::fence_before_sync();
    __syncthreads();
    if ((tid >> 5) == 0) tc::tmem_dealloc(tmem, kTmemCols);
  }
}

// ---- replay ring copies ---------------------------------------------------------------------
__global__ void __launch_bounds__(256) replay_push_kernel(SwarmReplay r, long long cursor, int B, int N,
                                                          const float4* __restrict__ state,
                                                          const int32_t* __restrict__ actions,
                                                          const float* __restrict__ rewards,
                                                          const float4* __restrict__ next_state) {
  const long long total = (long long)B * N;
  for (long long gI = (long long)blockIdx.x * blockDim.x + threadIdx.x; gI < total; gI += (long long)gridDim.x * blockDim.x) {
    const long long b = gI / N;
    const int i = (int)(gI - b * N);
    const long long ri = ((cursor + b) % r.capacity) * N + i;
    reinterpret_cast<float4*>(r.state)[ri] = state[gI];
    reinterpret_cast<float4*>(r.next_state)[ri] = next_state[gI];
    r.actions[ri] = (uint8_t)sanitize_action(actions[gI]);
    r.rewards[ri] = rewards[gI];
  }
}

__global__ void __launch_bounds__(256) replay_gather_kernel(SwarmReplay r, const int64_t* __restrict__ indices, int G,
                                                            int N, float4* __restrict__ state,
                                                            int32_t* __restrict__ actions, float* __restrict__ rewards,
                                                            float4* __restrict__ next_state) {
  const long long total = (long long)G * N;
  for (long long gI = (long long)blockIdx.x * blockDim.x + threadIdx.x; gI < total; gI += (long long)gridDim.x * blockDim.x) {
    const long long b = gI / N;
    const int i = (int)(gI - b * N);
    long long slot = indices[b];                          // caller-supplied: clamped into the ring, never out of bounds
    slot = slot < 0 ? 0 : (slot >= r.capacity ? r.capacity - 1 : slot);
    const long long ri = slot * N + i;
    state[gI] = reinterpret_cast<const float4*>(r.state)[ri];
    next_state[gI] = reinterpret_cast<const float4*>(r.next_state)[ri];
    actions[gI] = r.actions[ri];
    rewards[gI] = r.rewards[ri];
  }
}

static int copy_blocks(long long total) {
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  return blocks < 1 ? 1 : (int)blocks;
}

cudaError_t launch_replay_push(const SwarmReplay& r, long long cursor, int B, int N, const float* state,
                               const int32_t* actions, const float* rewards, const float* next_state,
                               cudaStream_t stream) {
  replay_push_kernel<<<copy_blocks((long long)B * N), 256, 0, stream>>>(
      r, cursor, B, N, reinterpret_cast<const float4*>(state), actions, rewards, reinterpret_cast<const float4*>(next_state));
  return cudaGetLastError();
}

cudaError_t launch_replay_gather(const SwarmReplay& r, const int64_t* indices, int G, int N, float* state,
                                 int32_t* actions, float* rewards, float* next_state, cudaStream_t stream) {
  replay_gather_kernel<<<copy_blocks((long long)G * N), 256, 0, stream>>>(
      r, indices, G, N, reinterpret_cast<float4*>(state), actions, rewards, reinterpret_cast<float4*>(next_state));
  return cudaGetLastError();
}

// explicit instantiations + launcher
template <int MODE, bool TC, bool DENSE, bool FLOCK = false, int NT = 0, bool PLAIN = false>
static cudaError_t launch_tile_impl(const TileParams& p, cudaStream_t stream) {
  const SwarmConfig& c = p.cfg;
  const TileLayout L = tile_layout(MODE, kTileThreads, c.n_agents, c.knn_k, p.maxdeg, c.graph_mode, TC);
  const int grid = p.bal_q > 0 ? (int)((c.num_envs - p.bal_r) / p.bal_q) : (c.num_envs + p.epb - 1) / p.epb;
  if (L.total > 48 * 1024) {
    cudaError_t err =
        cudaFuncSetAttribute(tile_kernel<MODE, TC, DENSE, FLOCK, NT, PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             L.total);
    if (err != cudaSuccess) return err;
  }
  tile_kernel<MODE, TC, DENSE, FLOCK, NT, PLAIN><<<grid, kTileThreads, L.total, stream>>>(p);
  return cudaGetLastError();
}

// Grid shape of the Q modes.  A batch that fits one wave of CTA slots is spread EVENLY over all of them (a tick of a
// CTA costs about the same for 7 envs as for 10 -- it is latency bound -- so what counts is that every SM carries the
// same number of resident CTAs: C2's 4 096 envs are 410 full CTAs on 444 slots, 34 SMs with one CTA less).
static bool tile_grid_plan(TileParams& p) {
  const long long B = p.cfg.num_envs;
  const long long uniform = (B + p.epb - 1) / p.epb;
  const bool dense = uniform > 3 * 148;
  const long long slots = (dense ? 4 : 3) * 148;
  p.bal_q = p.bal_r = 0;
  if (uniform <= slots && B > 0) {
    const long long G = B < slots ? B : slots;       // uniform <= G <= B
    p.bal_q = (int)(B / G);
    p.bal_r = (int)(B - (long long)p.bal_q * G);
  }
  return dense;
}

// The launch takes the PLAIN rollout (see tile_kernel) when it asks for nothing but the greedy episode on the complete
// graph: final states, returns and hit counts.
static bool plain_rollout(const TileParams& p) {
  const SwarmTrace& tr = p.trace;
  const bool traced = tr.state || tr.actions || tr.q || tr.rewards || tr.flags || tr.contact || tr.edges || tr.dist;
  const bool scenario = p.cfg.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE || p.cfg.scenario == SWARM_SCENARIO_GOTO;
  return p.cfg.graph_mode == SWARM_GRAPH_COMPLETE && !traced && !p.replay.state && !p.actions_in && !p.ctl &&
         p.epsilon == 0.0f && scenario;
}

template <int MODE>
static cudaError_t launch_tile_q(const TileParams& p0, cudaStream_t stream) {
  if (!p0.use_tc) return launch_tile_impl<MODE, false, true>(p0, stream);
  TileParams p = p0;
  const bool dense = tile_grid_plan(p);
  if constexpr (MODE == MODE_ROLLOUT) {
    if (p.cfg.n_agents == 12 && plain_rollout(p))
      return dense ? launch_tile_impl<MODE, true, true, false, 12, true>(p, stream)
                   : launch_tile_impl<MODE, true, false, false, 12, true>(p, stream);
  }
  if (MODE == MODE_ROLLOUT && p.cfg.n_agents == 12)       // the benchmark shape with the swarm size at compile time
    return dense ? launch_tile_impl<MODE, true, true, false, 12>(p, stream)
                 : launch_tile_impl<MODE, true, false, false, 12>(p, stream);
  return dense ? launch_tile_impl<MODE, true, true>(p, stream) : launch_tile_impl<MODE, true, false>(p, stream);
}

// the Flocking-reward rollout: same selection of the tensor-core / register-budget variants
static cudaError_t launch_tile_flock(const TileParams& p0, cudaStream_t stream) {
  if (!p0.use_tc) return launch_tile_impl<MODE_ROLLOUT, false, true, true>(p0, stream);
  TileParams p = p0;
  const bool dense = tile_grid_plan(p);
  if (p.cfg.n_agents == 12)
    return dense ? launch_tile_impl<MODE_ROLLOUT, true, true, true, 12>(p, stream)
                 : launch_tile_impl<MODE_ROLLOUT, true, false, true, 12>(p, stream);
  return dense ? launch_tile_impl<MODE_ROLLOUT, true, true, true>(p, stream)
               : launch_tile_impl<MODE_ROLLOUT, true, false, true>(p, stream);
}

cudaError_t launch_tile(int mode, const TileParams& p, cudaStream_t stream) {
  switch (mode) {
    case MODE_ROLLOUT: return p.use_flock ? launch_tile_flock(p, stream) : launch_tile_q<MODE_ROLLOUT>(p, stream);
    case MODE_FORWARD: return launch_tile_q<MODE_FORWARD>(p, stream);
    case MODE_GRAPH: return launch_tile_impl<MODE_GRAPH, false, true>(p, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace swarm

#ifdef SWARM_PHASE_CLOCKS
// per-warp phase cycles of the last tile-kernel launch, [warps][PH_COUNT] (scripts/time_rollout_phases.py)
extern "C" int swarm_phase_cycles(unsigned long long* dst, int warps) {
  if (warps > swarm::kPhaseWarps) warps = swarm::kPhaseWarps;
  const cudaError_t e = cudaMemcpyFromSymbol(dst, swarm::g_phase_cycles, sizeof(unsigned long long) * swarm::PH_COUNT * warps);
  return e == cudaSuccess ? warps : -1;
}
#endif
