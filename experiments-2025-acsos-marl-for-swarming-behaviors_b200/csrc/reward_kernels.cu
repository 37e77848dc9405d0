// reward_kernels.cu -- the reward functions of the two remaining reference scenarios, evaluated on the state that
// swarm_sim_step leaves in HBM (their physics is the GoTo world: colliding sphere agents, no colliding landmark):
//   Flocking  flocking_scenario.py:93-176  collective reward = sum over agents of (shaped goal progress [+ 50 on the
//             goal] + (-1) per other agent closer than 0.005 surface to surface + shaped spacing progress); keeps the
//             two `previous_*` shaping terms per agent between ticks, initialised the way reset_world_at does
//   Cohesion  cohesion_scenario.py:66-85   per-agent reward from the smallest / largest surface distance to the others
// Thread = agent, a CTA owns floor(128 / N) whole envs: positions go through shared memory once, each thread sweeps its
// partners in agent order (the order the reference's list comprehensions visit them), and -- Flocking -- the first
// thread of every env adds the N per-agent terms in agent order, as the reference's `+=` loop does.
// The reference evaluates Python `if`s on tensors (flocking:141,169; cohesion:80,83) and therefore only runs with one
// env; here every env is treated as its own copy of that one-env computation.
#include <cstdint>

#include "swarm_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kRewardThreads = 128;

// Pipeline: the state (and shaping) rows of the NEXT tile are loaded into registers before the current tile is
// computed, and the shared-memory arrays are double-buffered, so an iteration costs one barrier (Cohesion) or two
// (Flocking) and no load latency sits on the critical path (the first version -- load, barrier, compute, load shaping,
// barrier, sum, barrier -- spent two thirds of its time waiting on those two loads, profiles/r1_ncu_scenario_reward.txt).
// The partner sweeps are branch-free.  Flocking's walks the OTHER agents (compressed index k -> partner k + (k >= i)) in
// the order torch's CPU row sum adds them (swarm_device.cuh torch_row_sum: eight lanes, so eight independent exact
// square roots are in flight); Cohesion's neutralises the own slot with selects.
// NT: swarm size as a compile-time constant (0 = run-time value) for the sizes of the reference's experiments: the
// partner sweeps and the index arithmetic unroll completely (the same specialisation as the streaming world step).
template <int KIND, int NT>
__global__ void __launch_bounds__(kRewardThreads, KIND == SWARM_REWARD_FLOCKING ? 12 : 16) scenario_reward_kernel(SwarmRewardSpec sp,
                                                                             const float4* __restrict__ state,
                                                                             float2* __restrict__ shaping,
                                                                             float* __restrict__ reward,
                                                                             float4* __restrict__ terms) {
  __shared__ float2 spos[2][kRewardThreads];
  __shared__ float sterm[2][kRewardThreads];
  const int N = NT > 0 ? NT : sp.n_agents;
  const int epb = kRewardThreads / N;
  const int tid = threadIdx.x;
  const int le = tid / N;                       // env within the CTA
  const int i = tid - le * N;                   // agent within the env
  const bool lane_used = le < epb;
  const bool step_flocking = KIND == SWARM_REWARD_FLOCKING && !sp.reset;
  // 32-bit indices: the entry point rejects num_envs * n_agents >= 2^31
  const int tiles = (sp.num_envs + epb - 1) / epb;
  const int env_index = (int)sp.env_index;

  auto row_of = [&](int tile) { return (tile * epb + le) * N + i; };
  auto live_at = [&](int tile) { return lane_used && tile < tiles && tile * epb + le < sp.num_envs; };

  int tile = blockIdx.x;
  float2 p_next = make_float2(0.0f, 0.0f), prev_next = make_float2(0.0f, 0.0f);
  if (live_at(tile)) {
    const float4 s = state[row_of(tile)];
    p_next = make_float2(s.x, s.y);
    if (step_flocking) prev_next = shaping[row_of(tile)];
  }
  int buf = 0;
  for (; tile < tiles; tile += gridDim.x, buf ^= 1) {
    const int env = tile * epb + le;
    const bool live = live_at(tile);
    const bool selected = live && (env_index < 0 || env == env_index);
    const float2 p = p_next, prev = prev_next;
    spos[buf][tid] = p;
    const int nxt = tile + gridDim.x;
    if (live_at(nxt)) {                                   // in flight while this tile is computed
      const float4 s = state[row_of(nxt)];
      p_next = make_float2(s.x, s.y);
      if (step_flocking) prev_next = shaping[row_of(nxt)];
    }
    __syncthreads();
    const float2* others = spos[buf] + le * N;
    const int g = env * N + i;
    float term = 0.0f;
    if (KIND == SWARM_REWARD_FLOCKING) {
      if (selected) {
        const float d_goal = norm2(__fsub_rn(p.x, sp.goal_x), __fsub_rn(p.y, sp.goal_y));
        const float shaped_goal = __fmul_rn(d_goal, sp.pos_shaping);
        // spacing term ((|p_i - p_j| - desired)^2 over j != i).mean() * dist_shaping (flocking:109-121,148-160); at a
        // reset the agents after i have not been placed yet and still sit at the origin world.reset put them at
        const int placed = sp.reset ? i : N;              // partners j > placed are still at the origin
        float sum;
        int close;
        flocking_partner_sweep(p.x, p.y, i, N,
                               [&](int j) { return j > placed ? make_float2(0.0f, 0.0f) : others[j]; },
                               sp.desired_distance, sp.agent_radius, sp.min_collision_distance, sum, close);
        const float spacing = __fmul_rn(__fdiv_rn(sum, (float)(N - 1)), sp.dist_shaping);
        shaping[g] = make_float2(shaped_goal, spacing);                         // flocking:101-121,138,159
        if (!sp.reset) {
          const float pos_rew = __fsub_rn(prev.x, shaped_goal);                 // flocking:136-137
          float r = pos_rew;
          if (d_goal < sp.goal_radius) r = __fadd_rn(r, sp.on_goal_bonus);      // flocking:141-142
          const float avoid = close ? __fmul_rn((float)close, sp.collision_reward) : 0.0f;   // flocking:163-168
          const float dist_rew = __fsub_rn(prev.y, spacing);                    // flocking:158
          term = __fadd_rn(__fadd_rn(r, avoid), dist_rew);                      // flocking:129
          if (terms) terms[g] = make_float4(pos_rew, avoid, dist_rew, d_goal);
        }
      }
      if (!sp.reset) {
        sterm[buf][tid] = term;
        __syncthreads();
        if (selected && i == 0) {
          const float* t = sterm[buf] + le * N;
          float c = 0.0f;                                 // self.collective_reward = 0; += per agent (flocking:125-129)
          for (int j = 0; j < N; ++j) c = __fadd_rn(c, t[j]);
          reward[env] = c;
        }
      }
    } else if (selected) {
      // cohesion:66-85: distances = get_distance(agent, other) for every other agent; min / max of them.  The surface
      // distance is a monotone function of the squared centre distance, so the sweep keeps the extreme squares and the
      // two exact square roots are taken once
      float lo = INFINITY, hi = 0.0f;
#pragma unroll 4
      for (int j = 0; j < N; ++j) {
        const float2 q = others[j];
        const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y);
        const float d2 = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));
        lo = fminf(lo, j == i ? INFINITY : d2);
        hi = fmaxf(hi, d2);                               // the own slot contributes 0, never above the others
      }
      const float mn = __fsub_rn(__fsub_rn(__fsqrt_rn(lo), sp.agent_radius), sp.agent_radius);
      const float mx = __fsub_rn(__fsub_rn(__fsqrt_rn(hi), sp.agent_radius), sp.agent_radius);
      const float collision = mn > sp.sigma ? 0.0f : expf(-__fdiv_rn(mn, sp.sigma));    // cohesion:79-80
      const float cohesion = mn < sp.sigma ? 0.0f : -__fsub_rn(mx, sp.sigma);           // cohesion:82-83
      reward[g] = __fadd_rn(collision, cohesion);
      if (terms) terms[g] = make_float4(collision, cohesion, mn, mx);
    }
  }
}

cudaError_t launch_scenario_reward(const SwarmRewardSpec& sp, const float* state, float* shaping, float* reward,
                                   float* terms, cudaStream_t stream) {
  const int epb = kRewardThreads / sp.n_agents;
  long long tiles = ((long long)sp.num_envs + epb - 1) / epb;
  if (tiles > 148 * 16) tiles = 148 * 16;
  const float4* s = reinterpret_cast<const float4*>(state);
  float2* sh = reinterpret_cast<float2*>(shaping);
  float4* t = reinterpret_cast<float4*>(terms);
#define SWARM_REWARD_LAUNCH(NT)                                                                                         \
  do {                                                                                                                  \
    if (sp.kind == SWARM_REWARD_FLOCKING)                                                                               \
      scenario_reward_kernel<SWARM_REWARD_FLOCKING, NT><<<(int)tiles, kRewardThreads, 0, stream>>>(sp, s, sh, reward, t); \
    else                                                                                                                \
      scenario_reward_kernel<SWARM_REWARD_COHESION, NT><<<(int)tiles, kRewardThreads, 0, stream>>>(sp, s, sh, reward, t); \
  } while (0)
  switch (sp.n_agents) {
    case 5: SWARM_REWARD_LAUNCH(5); break;
    case 8: SWARM_REWARD_LAUNCH(8); break;
    case 10: SWARM_REWARD_LAUNCH(10); break;
    case 12: SWARM_REWARD_LAUNCH(12); break;
    default: SWARM_REWARD_LAUNCH(0); break;
  }
#undef SWARM_REWARD_LAUNCH
  return cudaGetLastError();
}

}  // namespace swarm
