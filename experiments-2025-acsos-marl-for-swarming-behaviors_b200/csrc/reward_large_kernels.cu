// reward_large_kernels.cu -- the Flocking and Cohesion rewards of reward_kernels.cu for swarms of up to 4 096 agents
// (swarm_scenario_reward_large, and the reward of swarm_rollout_stack_large).  Same arithmetic, op for op, as
// scenario_reward_kernel; two things change with the swarm size:
//   * the spacing term's `.pow(2).mean(-1)` over the N - 1 partner distances goes through torch_row_sum_cascade, the
//     order torch's CPU row sum takes once a row holds 512 floats or more (swarm_device.cuh);
//   * the layout: an env's positions are staged once per CTA in shared memory as float2 (32 KB at 4 096 agents), a
//     thread owns one agent and sweeps all partners in that order -- the lanes of a warp read the same or the adjacent
//     partner at each step, so the shared-memory reads are broadcasts.  An env larger than one CTA is split over
//     ceil(N / 256) CTAs, each staging the whole env, so that 256 envs x 4 096 agents still fill the GPU.
// Flocking's collective reward is the strict left-to-right sum of the N per-agent terms in agent order (flocking:125-129):
// the sweep writes the terms to the caller's workspace and flocking_collect_kernel, one CTA per env, adds them in that
// order (no float atomics) and broadcasts the sum to the env's running returns when asked to.
#include <cstdint>

#include "swarm_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kRewardLargeThreads = 256;

template <int KIND>
__global__ void __launch_bounds__(kRewardLargeThreads, 2) scenario_reward_large_kernel(SwarmRewardSpec sp,
                                                                                       const float4* __restrict__ state,
                                                                                       float2* __restrict__ shaping,
                                                                                       float* __restrict__ reward,
                                                                                       float4* __restrict__ terms,
                                                                                       float* __restrict__ term_ws,
                                                                                       float* __restrict__ returns) {
  extern __shared__ float2 spos[];
  const int N = sp.n_agents;
  const int parts = (N + blockDim.x - 1) / blockDim.x;
  // 32-bit indices: the entry point rejects num_envs * n_agents >= 2^31
  const int env = sp.env_index >= 0 ? (int)sp.env_index : (int)(blockIdx.x / parts);
  const int i = (int)(blockIdx.x % parts) * blockDim.x + threadIdx.x;
  const float4* env_state = state + (long long)env * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float4 s = env_state[j];
    spos[j] = make_float2(s.x, s.y);
  }
  __syncthreads();
  if (i >= N) return;
  const int g = env * N + i;
  const float2 p = spos[i];
  if (KIND == SWARM_REWARD_FLOCKING) {
    const float d_goal = norm2(__fsub_rn(p.x, sp.goal_x), __fsub_rn(p.y, sp.goal_y));
    const float shaped_goal = __fmul_rn(d_goal, sp.pos_shaping);
    // at a reset the agents after i have not been placed yet and still sit at the origin world.reset put them at
    const int placed = sp.reset ? i : N;
    float sum;
    int close;
    flocking_partner_sweep<true>(p.x, p.y, i, N, [&](int j) { return j > placed ? make_float2(0.0f, 0.0f) : spos[j]; },
                                 sp.desired_distance, sp.agent_radius, sp.min_collision_distance, sum, close);
    const float spacing = __fmul_rn(__fdiv_rn(sum, (float)(N - 1)), sp.dist_shaping);
    if (sp.reset) {
      shaping[g] = make_float2(shaped_goal, spacing);                           // flocking:101-121
      return;
    }
    const float2 prev = shaping[g];
    shaping[g] = make_float2(shaped_goal, spacing);                             // flocking:138,159
    const float pos_rew = __fsub_rn(prev.x, shaped_goal);                       // flocking:136-137
    float r = pos_rew;
    if (d_goal < sp.goal_radius) r = __fadd_rn(r, sp.on_goal_bonus);            // flocking:141-142
    const float avoid = close ? __fmul_rn((float)close, sp.collision_reward) : 0.0f;   // flocking:163-168
    const float dist_rew = __fsub_rn(prev.y, spacing);                          // flocking:158
    term_ws[g] = __fadd_rn(__fadd_rn(r, avoid), dist_rew);                      // flocking:129
    if (terms) terms[g] = make_float4(pos_rew, avoid, dist_rew, d_goal);
  } else {
    // cohesion:66-85, the sweep of scenario_reward_kernel: extreme squared centre distances, two exact square roots
    float lo = INFINITY, hi = 0.0f;
#pragma unroll 4
    for (int j = 0; j < N; ++j) {
      const float2 q = spos[j];
      const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y);
      const float d2 = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));
      lo = fminf(lo, j == i ? INFINITY : d2);
      hi = fmaxf(hi, d2);                                 // the own slot contributes 0, never above the others
    }
    const float mn = __fsub_rn(__fsub_rn(__fsqrt_rn(lo), sp.agent_radius), sp.agent_radius);
    const float mx = __fsub_rn(__fsub_rn(__fsqrt_rn(hi), sp.agent_radius), sp.agent_radius);
    const float collision = mn > sp.sigma ? 0.0f : expf(-__fdiv_rn(mn, sp.sigma));    // cohesion:79-80
    const float cohesion = mn < sp.sigma ? 0.0f : -__fsub_rn(mx, sp.sigma);           // cohesion:82-83
    const float rw = __fadd_rn(collision, cohesion);
    if (reward) reward[g] = rw;
    if (returns) returns[g] = __fadd_rn(returns[g], rw);
    if (terms) terms[g] = make_float4(collision, cohesion, mn, mx);
  }
}

// Flocking's collective reward of one env per CTA: 0 + t_0 + t_1 + ... + t_{N-1} in agent order (flocking:125-129)
// -> reward[env]; returns[env][i] += that sum for every agent
__global__ void __launch_bounds__(kRewardLargeThreads) flocking_collect_kernel(int N, long long env_index,
                                                                               const float* __restrict__ term_ws,
                                                                               float* __restrict__ reward,
                                                                               float* __restrict__ returns) {
  extern __shared__ float st[];
  __shared__ float total;
  const long long env = env_index >= 0 ? env_index : blockIdx.x;
  const float* t = term_ws + env * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) st[j] = t[j];
  __syncthreads();
  if (threadIdx.x == 0) {
    float c = 0.0f;
#pragma unroll 16
    for (int j = 0; j < N; ++j) c = __fadd_rn(c, st[j]);
    total = c;
    if (reward) reward[env] = c;
  }
  if (!returns) return;
  __syncthreads();
  const float c = total;
  float* ret = returns + env * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) ret[j] = __fadd_rn(ret[j], c);
}

// workspace: float[num_envs][n_agents] of Flocking per-agent terms (the step call); Cohesion needs none
long long scenario_reward_large_workspace_bytes(const SwarmRewardSpec& sp) {
  return sp.kind == SWARM_REWARD_FLOCKING ? (long long)sp.num_envs * sp.n_agents * 4 : 0;
}

// returns (optional): += the reward of the call, per agent (Flocking: the env's collective reward)
cudaError_t launch_scenario_reward_large(const SwarmRewardSpec& sp, const float* state, float* shaping, float* reward,
                                         float* terms, float* returns, void* workspace, cudaStream_t stream) {
  const int N = sp.n_agents;
  const int threads = N < kRewardLargeThreads ? (N + 31) & ~31 : kRewardLargeThreads;
  const int parts = (N + threads - 1) / threads;
  const int envs = sp.env_index >= 0 ? 1 : sp.num_envs;
  const float4* s = reinterpret_cast<const float4*>(state);
  float2* sh = reinterpret_cast<float2*>(shaping);
  float4* t = reinterpret_cast<float4*>(terms);
  float* tw = reinterpret_cast<float*>(workspace);
  const size_t smem = (size_t)N * sizeof(float2);
  if (sp.kind == SWARM_REWARD_FLOCKING) {
    scenario_reward_large_kernel<SWARM_REWARD_FLOCKING><<<envs * parts, threads, smem, stream>>>(sp, s, sh, nullptr, t, tw,
                                                                                                 nullptr);
    if (!sp.reset && (reward || returns))
      flocking_collect_kernel<<<envs, threads, (size_t)N * sizeof(float), stream>>>(N, sp.env_index, tw, reward, returns);
  } else {
    scenario_reward_large_kernel<SWARM_REWARD_COHESION><<<envs * parts, threads, smem, stream>>>(sp, s, nullptr, reward, t,
                                                                                                 nullptr, returns);
  }
  return cudaGetLastError();
}

}  // namespace swarm
