// stack_kernels.cu -- multi-layer GAT Q-networks in ONE launch (SURVEY 8(f) rank 4).
//
// The reference's GCN class carries two more GATConv layers in comments (train_gcn_dqn.py:54-55, 64-67) and ships ten
// checkpoints of that three-layer form (data/models/experiment_Flocking-seed_*.pth: conv1 7 -> 8, conv2 / conv3 8 -> 8,
// lin1 8 -> 8, lin2 8 -> 9).  Stacking the generic layer kernels (gatlayer_kernels.cu) costs one launch set per layer
// plus the edge-list / CSR glue; here a whole forward
//     node features -> per-env graph -> L x [GATConv -> activation] -> lin1 -> ReLU -> lin2 (-> argmax)
// is one env-tile kernel (thread = agent, CTA = floor(128 / N) envs, tile_device.cuh): the in-edge lists are built once
// in shared memory and reused by every layer, the layer outputs never leave the chip.  The input features are the
// reference's [pos, vel, goal, agent id] (train:95-99) or [pos, vel, agent id] for scenarios whose observation() is
// cat[pos, vel] (cohesion_scenario.py:87-94).  Per layer the arithmetic follows torch_geometric's GATConv like the
// one-layer kernels: h = x W^T, alpha = <h, att>, LeakyReLU(0.2) logits, max-subtracted softmax with the 1e-16
// denominator, messages alpha * h_src summed in edge-list order, + bias (alpha = weight x reciprocal of the sum and fused
// multiply-adds: float32-level different rounding than torch's separately rounded ops, like the tensor-core path).
#include <cstring>

#include "stack_device.cuh"
#include "launchers.h"

namespace swarm {

struct StackParams {
  SwarmConfig cfg;
  SwarmStackSpec spec;
  const float* weights;
  const float4* state;
  float* q_out;              // [B*N][9] or nullptr
  int32_t* act_out;          // [B*N] or nullptr
  int32_t epb, maxdeg;
  float qmax_r;
  // fused rollout (gatstack_rollout_kernel): `ticks` x [forward -> argmax -> world step -> reward], state in registers
  WorldConsts step;          // constants of the world step
  float4* state_rw;          // [B*N] advanced in place
  float* returns;            // [B*N] += (optional)
  int32_t* hits;             // [B] += (optional)
  SwarmRewardSpec flock;     // use_flock 1: the Flocking collective reward, 2: Cohesion's per-agent reward, instead of the world's
  float2* shaping;           // [B*N] Flocking memory, read at launch, written back
  int32_t use_flock;
  int32_t ticks;
  // device-driven train tick (gatstack_train_kernel): one tick with epsilon-greedy exploration and the replay push;
  // epsilon, the RNG tick and the ring cursor come from *ctl
  const SwarmTrainCtl* ctl;
  SwarmReplay replay;
  unsigned long long rng_seed;
  long long env_offset;
};

struct StackSmem {
  int w, st, red, h, asrc, inl, wt, kv, total;
};
template <int HP>
__host__ __device__ inline StackSmem stack_smem(int L, int n, int k, int maxdeg, int graph_mode) {
  StackSmem s;
  int off = 0;
  s.w = off;    off = tile_align16(off + StackLayout<HP>::total(L) * 4);
  s.st = off;   off = tile_align16(off + 2 * kTileThreads * 16);
  s.red = off;  off = tile_align16(off + kTileThreads * 4);
  s.h = off;    off = tile_align16(off + kTileThreads * (HP + 4) * 4);
  s.asrc = off; off = tile_align16(off + kTileThreads * 4);
  s.inl = off;  off = tile_align16(off + maxdeg * kTileThreads);
  s.wt = off;   off = tile_align16(off + maxdeg * kTileThreads * 4);
  s.kv = off;   off = tile_align16(off + (graph_mode == SWARM_GRAPH_KNN ? kTileThreads * 4 : 0));
  s.total = off;
  return s;
}

// ROLLOUT = false: one forward (swarm_gatstack_forward).  ROLLOUT = true: the evaluation loop simulator.py:59-93 for a
// stacked network -- p.ticks x [forward -> argmax -> world step -> reward] with the agent's state, running return and
// Flocking memory in registers, exactly the tick of tile_kernels.cu's rollout (same world-step and reward device code,
// so it equals forward + swarm_sim_step + swarm_scenario_reward composed by hand bit for bit).
// TRAIN (with ROLLOUT, p.ticks = 1): the rollout tick of the device-driven train tick (train:160-172) -- the greedy
// action is replaced by the exploration draws of tile_kernels.cu's MODE_ROLLOUT with p.ctl, and the transition
// (s, a, r, s') is pushed at slot (ctl->ring_cursor + env) % capacity.  A separate template value so that the forward
// and the evaluation rollout keep their code instruction for instruction.
template <int HP, bool ROLLOUT, bool TRAIN>
__device__ __forceinline__ void gatstack_body(const StackParams& p) {
  static_assert(!TRAIN || ROLLOUT, "the train tick is a rollout tick");
  extern __shared__ __align__(16) unsigned char smem[];
  using SL = StackLayout<HP>;
  const SwarmConfig& c = p.cfg;
  const SwarmStackSpec& sp = p.spec;
  const int T = kTileThreads, N = c.n_agents, K = c.knn_k, L = sp.n_layers;
  const TileThread t = tile_thread(N, p.epb, c.num_envs);
  const int tid = t.tid;
  const StackSmem S = stack_smem<HP>(L, N, K, p.maxdeg, c.graph_mode);
  float* sw = reinterpret_cast<float*>(smem + S.w);
  float4* sst = reinterpret_cast<float4*>(smem + S.st);
  float* sh = reinterpret_cast<float*>(smem + S.h);
  TileGraphSmem g = {};
  g.sas = reinterpret_cast<float*>(smem + S.asrc);
  g.sin = smem + S.inl;
  g.skv = reinterpret_cast<float*>(smem + S.kv);

  float* sred = reinterpret_cast<float*>(smem + S.red);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  float ret0 = 0.0f, ret = 0.0f;
  float2 shp = make_float2(0.0f, 0.0f);
  int myhits = 0;
  if (t.active) {
    s = ROLLOUT ? p.state_rw[t.gidx] : p.state[t.gidx];
    if (ROLLOUT && p.returns) ret0 = p.returns[t.gidx];
    if (ROLLOUT && p.use_flock == 1) shp = p.shaping[t.gidx];
  }
  stack_stage_weights<HP>(sp, p.weights, sw, tid, T);
  uint64_t cache_rank = ~0ull, cache_nbr = 0;
  int deg = 0;
  const int n_ticks = ROLLOUT ? p.ticks : 1;
  for (int tick = 0; tick < n_ticks; ++tick) {
  const float4* pos = sst + (tick & 1) * T;
  sst[(tick & 1) * T + tid] = s;
  __syncthreads();

  // ---- graph: in-edge list of this node in edge-list order, once for all layers ------------------------------------
  if (c.graph_mode == SWARM_GRAPH_KNN) {
    const uint64_t nbr = tile_knn_small(t, pos, s, N, K, cache_rank, cache_nbr);
    deg = tile_in_edges_knn_small(g, t, N, K, nbr, reinterpret_cast<uint32_t*>(g.skv));
  } else if (c.graph_mode == SWARM_GRAPH_RADIUS) {
    if (t.active) deg = tile_in_edges_radius(g, t, pos, s, N, p.qmax_r);
  } else if (t.active && tick == 0) {
    deg = tile_in_edges_complete(g, t, N);
  }

  // ---- node features (train:95-99), L x [GATConv -> activation], head: lin1 -> ReLU -> lin2, argmax (first maximum wins)
  float x[HP];
  stack_features<HP>(x, s, c, sp.in_features, t.i);
  const uint8_t* sin = g.sin + tid;
  float* swt = reinterpret_cast<float*>(smem + S.wt) + tid;
  for (int l = 0; l < L; ++l)
    stack_layer<HP>(sw, l, sp.activation[l] == 1, x, sh, g.sas, sin, swt, tid, t.envbase, deg, l > 0);
  float r[HP];
  float q[SL::kW2Cols];                                  // 9 actions + 3 zero-padded columns
  stack_head<HP>(sw, L, x, r, q);
  const float* b2 = stack_lin2_bias<HP>(sw, L);
  float best = 0.0f;
  int action = 0;
#pragma unroll
  for (int a = 0; a < 9; ++a) {
    q[a] = __fadd_rn(q[a], b2[a]);
    if (a == 0 || q[a] > best) { best = q[a]; action = a; }
  }
  if (!ROLLOUT) {
    if (t.active) {
      if (p.q_out) {
#pragma unroll
        for (int a = 0; a < 9; ++a) p.q_out[t.gidx * 9 + a] = q[a];
      }
      if (p.act_out) p.act_out[t.gidx] = action;
    }
  } else {
    // ---- world step + reward: the tick of tile_kernels.cu ------------------------------------------------------------
    float reward = 0.0f;
    if (t.active) {
      const bool oa = c.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE;
      uint8_t flags = 0;
      uint32_t cmask = 0;
      // the cursor is read here, not in the prologue: live across the layers it would cost spills
      const float epsilon = TRAIN ? p.ctl->epsilon : 0.0f;
      if (TRAIN && epsilon > 0.0f) {
        // train:164-165: one coin per tick for the whole swarm, then one uniform action per agent (the stream of the
        // one-layer tick)
        const unsigned long long genv = (unsigned long long)(p.env_offset + t.env);
        const unsigned long long gt = (unsigned long long)(p.ctl->tick + 1);
        const float coin = (float)(rng_draw(p.rng_seed, genv, gt, 0xFFFFu) >> 40) * (1.0f / 16777216.0f);
        if (coin < epsilon) action = (int)(((rng_draw(p.rng_seed, genv, gt, (uint32_t)t.i) >> 32) * 9ull) >> 32);
      }
      const float4 s_prev = s;
      float2 u;
      decode_action(action, u.x, u.y);
      agent_step(s, u, pos + t.envbase, N, t.i, oa, c, p.step, flags, cmask);
      if (TRAIN) {
        // GraphReplayBuffer.push (train:171-172), state-only transition; the reward follows below
        const long long ri = ((p.ctl->ring_cursor + t.env) % p.replay.capacity) * N + t.i;
        reinterpret_cast<float4*>(p.replay.state)[ri] = s_prev;
        reinterpret_cast<float4*>(p.replay.next_state)[ri] = s;
        p.replay.actions[ri] = (uint8_t)sanitize_action(action);
      }
      float dgoal, dobs;
      reward = post_step_reward(s, oa, c, dgoal, dobs, flags);
      if (oa) myhits += (flags & SWARM_FLAG_HIT) ? 1 : 0;
      else if (!p.use_flock) sred[tid] = dgoal;     // GoTo's collective reward needs every agent's distance: finished below
    }
    if (p.use_flock == 2) {
      // Cohesion (cohesion:66-85): smallest / largest surface distance to the other agents at their POST-step positions;
      // the op sequence of reward_kernels.cu (extreme squared distances, two exact square roots)
      const SwarmRewardSpec& fs = p.flock;
      float4* post = sst + ((tick + 1) & 1) * T;
      post[tid] = s;
      __syncthreads();
      if (t.active) {
        const float4* others = post + t.envbase;
        float lo = INFINITY, hi = 0.0f;
#pragma unroll 4
        for (int j = 0; j < N; ++j) {
          const float2 q = xy_of(others[j]);
          const float dx = __fsub_rn(s.x, q.x), dy = __fsub_rn(s.y, q.y);
          const float d2 = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));
          lo = fminf(lo, j == t.i ? INFINITY : d2);
          hi = fmaxf(hi, d2);
        }
        const float mn = __fsub_rn(__fsub_rn(__fsqrt_rn(lo), fs.agent_radius), fs.agent_radius);
        const float mx = __fsub_rn(__fsub_rn(__fsqrt_rn(hi), fs.agent_radius), fs.agent_radius);
        const float collision = mn > fs.sigma ? 0.0f : expf(-__fdiv_rn(mn, fs.sigma));    // cohesion:79-80
        const float cohesion = mn < fs.sigma ? 0.0f : -__fsub_rn(mx, fs.sigma);           // cohesion:82-83
        reward = __fadd_rn(collision, cohesion);
      }
    } else if (p.use_flock) {
      // Flocking (flocking:124-171): every agent's term from the POST-step positions of its env, then the collective sum
      // in agent order (the op sequence of reward_kernels.cu / the FLOCK tile kernel)
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
    ret = __fadd_rn(ret, reward);
    if (TRAIN && t.active) p.replay.rewards[((p.ctl->ring_cursor + t.env) % p.replay.capacity) * N + t.i] = reward;
  }
  }   // tick loop

  if (ROLLOUT) {
    if (t.active) {
      p.state_rw[t.gidx] = s;
      if (p.returns) p.returns[t.gidx] = __fadd_rn(ret0, ret);
      if (p.use_flock == 1) p.shaping[t.gidx] = shp;
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
}

template <int HP, bool ROLLOUT>
__global__ void __launch_bounds__(kTileThreads) gatstack_kernel(const __grid_constant__ StackParams p) {
  gatstack_body<HP, ROLLOUT, false>(p);
}

template <int HP>
__global__ void __launch_bounds__(kTileThreads) gatstack_train_kernel(const __grid_constant__ StackParams p) {
  gatstack_body<HP, true, true>(p);
}

template <int HP>
static cudaError_t launch_stack_hp(const StackParams& p, cudaStream_t stream) {
  const SwarmConfig& c = p.cfg;
  const StackSmem S = stack_smem<HP>(p.spec.n_layers, c.n_agents, c.knn_k, p.maxdeg, c.graph_mode);
  if (S.total > 227 * 1024) return cudaErrorInvalidConfiguration;
  auto* kernel = p.ctl ? gatstack_train_kernel<HP> : (p.ticks > 0 ? gatstack_kernel<HP, true> : gatstack_kernel<HP, false>);
  if (S.total > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, S.total);
    if (err != cudaSuccess) return err;
  }
  const int grid = (c.num_envs + p.epb - 1) / p.epb;
  kernel<<<grid, kTileThreads, S.total, stream>>>(p);
  return cudaGetLastError();
}

int stack_weight_count_host(const SwarmStackSpec& s) { return stack_weight_count(s); }

static cudaError_t launch_stack(const StackParams& p, cudaStream_t stream) {
  if (p.spec.hidden <= 8) return launch_stack_hp<8>(p, stream);
  if (p.spec.hidden <= 16) return launch_stack_hp<16>(p, stream);
  return launch_stack_hp<32>(p, stream);
}

static void stack_fill(StackParams& p, const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights) {
  std::memset(&p, 0, sizeof(p));
  p.cfg = c;
  p.spec = spec;
  p.weights = weights;
  p.epb = kTileThreads / c.n_agents;
  p.maxdeg = c.graph_mode == SWARM_GRAPH_KNN ? (c.n_agents + c.knn_k + 1) : c.n_agents;
  p.qmax_r = c.graph_mode == SWARM_GRAPH_RADIUS ? sq_threshold(c.graph_radius) : 0.0f;
}

// the fused evaluation loop; flock == nullptr: world reward
cudaError_t launch_gatstack_rollout(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, float* state,
                                    int ticks, const WorldConsts& step, const SwarmRewardSpec* flock, float* shaping,
                                    float* returns, int32_t* hits, cudaStream_t stream) {
  if (ticks <= 0) return cudaSuccess;
  StackParams p;
  stack_fill(p, c, spec, weights);
  p.step = step;
  p.state_rw = reinterpret_cast<float4*>(state);
  p.returns = returns;
  p.hits = hits;
  p.ticks = ticks;
  if (flock) {
    p.flock = *flock;
    p.shaping = reinterpret_cast<float2*>(shaping);
    p.use_flock = flock->kind == SWARM_REWARD_COHESION ? 2 : 1;
  }
  return launch_stack(p, stream);
}

// the rollout tick of swarm_train_tick_stack: one tick of the loop above with exploration and the replay push
cudaError_t launch_gatstack_train_tick(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, float* state,
                                       const WorldConsts& step, const SwarmRewardSpec* flock, float* shaping,
                                       float* returns, int32_t* hits, const SwarmReplay& ring, const SwarmTrainCtl* ctl,
                                       unsigned long long rng_seed, long long env_offset, cudaStream_t stream) {
  StackParams p;
  stack_fill(p, c, spec, weights);
  p.step = step;
  p.state_rw = reinterpret_cast<float4*>(state);
  p.returns = returns;
  p.hits = hits;
  p.ticks = 1;
  if (flock) {
    p.flock = *flock;
    p.shaping = reinterpret_cast<float2*>(shaping);
    p.use_flock = flock->kind == SWARM_REWARD_COHESION ? 2 : 1;
  }
  p.ctl = ctl;
  p.replay = ring;
  p.rng_seed = rng_seed;
  p.env_offset = env_offset;
  return launch_stack(p, stream);
}

cudaError_t launch_gatstack_forward(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, const float* state,
                                    float* q, int32_t* actions, cudaStream_t stream) {
  StackParams p;
  std::memset(&p, 0, sizeof(p));
  p.cfg = c;
  p.spec = spec;
  p.weights = weights;
  p.state = reinterpret_cast<const float4*>(state);
  p.q_out = q;
  p.act_out = actions;
  p.epb = kTileThreads / c.n_agents;
  p.maxdeg = c.graph_mode == SWARM_GRAPH_KNN ? (c.n_agents + c.knn_k + 1) : c.n_agents;
  p.qmax_r = c.graph_mode == SWARM_GRAPH_RADIUS ? sq_threshold(c.graph_radius) : 0.0f;
  if (spec.hidden <= 8) return launch_stack_hp<8>(p, stream);
  if (spec.hidden <= 16) return launch_stack_hp<16>(p, stream);
  return launch_stack_hp<32>(p, stream);
}

}  // namespace swarm
