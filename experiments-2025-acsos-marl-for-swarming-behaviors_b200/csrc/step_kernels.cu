// step_kernels.cu -- the stand-alone world step (vmas Environment.step, train_gcn_dqn.py:169 / simulator.py:68)
// as a lean HBM-streaming kernel: 40 algorithmic bytes per agent-step (float4 state in, int32 action in, float4
// state out, float reward out) plus optional observation / distance / flag / mask outputs.
//
// 256 threads per CTA, thread = agent, floor(256/N) whole envs per CTA (N = 12: 252 of 256 lanes busy).  Partner
// positions are staged once in shared memory as float2; the pair loop is branch-light (the self pair is tested
// too: it yields a zero force and its mask bit is cleared afterwards) and unrolled for memory-level parallelism.
// The agent's step is agent_step of swarm_device.cuh, the world step of every other kernel, so results are
// bit-identical to the fused rollouts' world step.
//
// Two kernels with identical arithmetic:
//   sim_step_kernel         one tile per CTA, plain loads / stores (small batches, ragged tail, unaligned buffers,
//                           swarms of more than 64 agents)
//   sim_step_stream_kernel  persistent CTAs; every tile of floor(256/N) envs is one contiguous block of the state /
//                           action arrays, so it is pulled into a 4-deep shared-memory ring by the TMA engine
//                           (cp.async.bulk + mbarrier complete_tx) and the new state / rewards leave through bulk
//                           stores from a 3-deep staging ring: the SM never waits on its own loads and HBM sees long
//                           16-byte-aligned bursts only.
#include "tile_kernels.cuh"
#include "tc_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kStepThreads = 256;

__global__ void __launch_bounds__(kStepThreads) sim_step_kernel(const __grid_constant__ SimStepArgs p) {
  __shared__ float2 spos[kStepThreads];
  __shared__ float sdg[kStepThreads];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents;
  const int tid = threadIdx.x;
  const int el = tid / N;
  const int i = tid - el * N;
  const long long env = (long long)blockIdx.x * p.epb + el;
  const bool active = (el < p.epb) && (env < c.num_envs);
  const int envbase = el * N;
  const long long gidx = env * N + i;

  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  int action = 0;
  if (active) {
    s = p.state_in[gidx];
    action = p.actions[gidx];
  }
  spos[tid] = make_float2(s.x, s.y);
  __syncthreads();

  float reward = 0.0f;
  if (active) {
    const bool oa = c.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE;
    float2 u;
    decode_action(action, u.x, u.y);
    uint8_t flags = 0;
    uint32_t cmask = 0;
    agent_step(s, u, spos + envbase, N, i, oa, c, p.world, flags, cmask);
    float dgoal, dobs;
    reward = post_step_reward(s, oa, c, dgoal, dobs, flags);
    if (!oa) sdg[tid] = dgoal;
    p.state_out[gidx] = s;
    store_step_outputs(p, gidx, s, dgoal, dobs, flags, cmask);
  }
  if (c.scenario == SWARM_SCENARIO_GOTO) {
    // collective reward (go_to:108-115): 0 + (-d_0) + (-d_1) + ... in agent order, same value for every agent
    __syncthreads();
    if (active)
      for (int a = 0; a < N; ++a) reward = __fadd_rn(reward, -sdg[envbase + a]);
  }
  if (active && p.rewards) p.rewards[gidx] = reward;
}

// ---- persistent TMA-pipelined variant --------------------------------------------------------------------------
constexpr int kStepStages = 4;     // input ring depth
constexpr int kStepOutBufs = 4;    // output staging ring depth (two tiles per loop iteration)

__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   tc::smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(tc::smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_store(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(tc::smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}

struct StepStreamSmem {
  float4 sin[kStepStages][kStepThreads];
  float4 sout[kStepOutBufs][kStepThreads];
  int32_t ain[kStepStages][kStepThreads];
  float rout[kStepOutBufs][kStepThreads];
  float sdg[2][kStepThreads];
  uint64_t full[kStepStages];
  float2 force_of_action[16];     // decode table: flat action -> (ux, uy); entries >= 9 are zero (invalid actions)
};

// `ntiles` full tiles of p.epb envs each (the ragged tail goes to sim_step_kernel); p.epb * N is a multiple of 4 so
// every bulk copy is a multiple of 16 bytes at a 16-byte aligned address.
// EXTRAS: any of the optional outputs (flags / contact masks / observations / distances) is requested; OA: scenario
// known at compile time.  The minimal variant is issue bound (ncu: 81 % issue utilisation), so the four null checks
// and the scenario branches per agent are worth a template.
// NT: swarm size known at compile time (0 = run-time value): the index arithmetic and the partner sweep of the
// benchmark shape (12 agents) unroll completely.
template <bool EXTRAS, bool OA, int NT>
__global__ void __launch_bounds__(kStepThreads, 4) sim_step_stream_kernel(const __grid_constant__ SimStepArgs p,
                                                                          const long long ntiles) {
  __shared__ __align__(128) StepStreamSmem sm;
  const SwarmConfig& c = p.cfg;
  const int N = NT > 0 ? NT : c.n_agents;
  const int tid = threadIdx.x;
  const int el = tid / N;
  const int i = tid - el * N;
  const bool active = el < p.epb;
  const int envbase = el * N;
  const int tile_agents = p.epb * N;
  const uint32_t sbytes = (uint32_t)tile_agents * 16u, abytes = (uint32_t)tile_agents * 4u;

  const long long first = blockIdx.x, stride = gridDim.x;
  const long long n_my = first < ntiles ? (ntiles - first + stride - 1) / stride : 0;

  if (tid < 16) {
    float ux = 0.0f, uy = 0.0f;
    if (tid < 9) decode_action(tid, ux, uy);
    sm.force_of_action[tid] = make_float2(ux, uy);
  }
  if (tid == 0) {
    for (int s = 0; s < kStepStages; ++s) tc::mbar_init(&sm.full[s], 1);
    tc::fence_async_smem();
    for (int s = 0; s < kStepStages && s < n_my; ++s) {
      const long long a0 = (first + s * stride) * tile_agents;
      mbar_expect_tx(&sm.full[s], sbytes + abytes);
      bulk_load(sm.sin[s], p.state_in + a0, sbytes, &sm.full[s]);
      bulk_load(sm.ain[s], p.actions + a0, abytes, &sm.full[s]);
    }
  }
  __syncthreads();

  // Two tiles per loop iteration: the mbarrier waits, the proxy fence, the block barrier and thread 0's copy
  // bookkeeping are paid once per PAIR of tiles (the kernel is issue bound at ~290 instructions per agent, ~25 of them
  // this per-tile overhead), and the two agents of a thread are independent instruction streams.
  auto step_agent = [&](int stage, int ob, long long gidx, int which) -> float {
    float4 s = sm.sin[stage][tid];
    const int action = sm.ain[stage][tid];
    const float2 u = sm.force_of_action[min((unsigned)action, 9u)];      // vmas _set_action (a // 3, a % 3) -> (0, -1, +1)
    uint8_t flags = 0;
    uint32_t cmask = 0;
    agent_step(s, u, &sm.sin[stage][envbase], N, i, OA, c, p.world, flags, cmask);
    float dgoal, dobs;
    const float reward = post_step_reward(s, OA, c, dgoal, dobs, flags);
    if (!OA) sm.sdg[which][tid] = dgoal;
    sm.sout[ob][tid] = s;
    if (EXTRAS) store_step_outputs(p, gidx, s, dgoal, dobs, flags, cmask);
    return reward;
  };

  int stage = 0, ob = 0;
  uint32_t parity = 0;
  long long a0 = first * tile_agents;
  const long long a_stride = stride * tile_agents;
  for (long long it = 0; it < n_my; it += 2, a0 += 2 * a_stride) {
    const bool two = it + 1 < n_my;
    float reward0 = 0.0f, reward1 = 0.0f;
    tc::mbar_wait(&sm.full[stage], parity);
    if (active) reward0 = step_agent(stage, ob, a0 + tid, 0);
    if (two) {
      tc::mbar_wait(&sm.full[stage + 1], parity);
      if (active) reward1 = step_agent(stage + 1, ob + 1, a0 + a_stride + tid, 1);
    }
    if (!OA) {
      // GoTo's collective reward (go_to:108-115): 0 + (-d_0) + (-d_1) + ... in agent order
      __syncthreads();
      if (active) {
        for (int a = 0; a < N; ++a) reward0 = __fadd_rn(reward0, -sm.sdg[0][envbase + a]);
        if (two)
          for (int a = 0; a < N; ++a) reward1 = __fadd_rn(reward1, -sm.sdg[1][envbase + a]);
      }
    }
    if (active) {
      sm.rout[ob][tid] = reward0;
      if (two) sm.rout[ob + 1][tid] = reward1;
    }

    tc::fence_async_smem();          // generic-proxy writes of sout / rout -> visible to the bulk-copy engine
    __syncthreads();                 // ... and every thread is done reading sin[stage], sin[stage + 1] (and sdg)
    if (tid == 0) {
      bulk_store(p.state_out + a0, sm.sout[ob], sbytes);
      if (p.rewards) bulk_store(p.rewards + a0, sm.rout[ob], abytes);
      if (two) {
        bulk_store(p.state_out + a0 + a_stride, sm.sout[ob + 1], sbytes);
        if (p.rewards) bulk_store(p.rewards + a0 + a_stride, sm.rout[ob + 1], abytes);
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      for (int q = 0; q < 2; ++q) {
        if (it + q + kStepStages < n_my) {
          const long long n0 = a0 + (kStepStages + q) * a_stride;
          mbar_expect_tx(&sm.full[stage + q], sbytes + abytes);
          bulk_load(sm.sin[stage + q], p.state_in + n0, sbytes, &sm.full[stage + q]);
          bulk_load(sm.ain[stage + q], p.actions + n0, abytes, &sm.full[stage + q]);
        }
      }
      // the staging buffers written in the next iteration were last read by the stores issued one iteration ago
      asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
    }
    stage += 2;
    if (stage == kStepStages) { stage = 0; parity ^= 1u; }
    ob += 2;
    if (ob == kStepOutBufs) ob = 0;
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

static bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; }

cudaError_t launch_sim_step(SimStepArgs p, cudaStream_t stream) {
  const int N = p.cfg.n_agents;
  const long long num_envs = p.cfg.num_envs;
  long long env0 = 0;

  // streaming path: at most 64 agents, full tiles whose agent count is a multiple of 4 (16-byte bulk copies), all
  // buffers 16-byte aligned, and at least one tile per SM -- everything else (and the ragged tail) runs through the
  // one-tile-per-CTA kernel.  Larger swarms are bound by the O(N) contact sweep, not by HBM: at 96 and 128 agents
  // (16 384 envs, B200) the persistent pipelined kernel took 2-11 % longer than one tile per CTA.
  int epb_s = N <= 64 ? kStepThreads / N : 0;
  while (epb_s > 0 && ((epb_s * N) & 3)) --epb_s;
  const long long ntiles = epb_s > 0 ? num_envs / epb_s : 0;
  if (ntiles >= 148 && aligned16(p.state_in) && aligned16(p.actions) && aligned16(p.state_out) &&
      (!p.rewards || aligned16(p.rewards))) {
    p.epb = epb_s;
    const long long grid = ntiles < 148 * 4 ? ntiles : 148 * 4;
    const bool extras = p.flags || p.contact || p.obs || p.dist;
    const bool oa = p.cfg.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE;
#define SWARM_STEP_LAUNCH(NT)                                                                                           \
  do {                                                                                                                  \
    if (extras && oa) sim_step_stream_kernel<true, true, NT><<<(unsigned)grid, kStepThreads, 0, stream>>>(p, ntiles);   \
    else if (extras) sim_step_stream_kernel<true, false, NT><<<(unsigned)grid, kStepThreads, 0, stream>>>(p, ntiles);   \
    else if (oa) sim_step_stream_kernel<false, true, NT><<<(unsigned)grid, kStepThreads, 0, stream>>>(p, ntiles);       \
    else sim_step_stream_kernel<false, false, NT><<<(unsigned)grid, kStepThreads, 0, stream>>>(p, ntiles);              \
  } while (0)
    // the swarm sizes of the reference's experiments (5 .. 12 agents, SURVEY.md 8d) with the size as a compile-time
    // constant; any other size through the run-time variant
    switch (N) {
      case 5: SWARM_STEP_LAUNCH(5); break;
      case 6: SWARM_STEP_LAUNCH(6); break;
      case 7: SWARM_STEP_LAUNCH(7); break;
      case 8: SWARM_STEP_LAUNCH(8); break;
      case 9: SWARM_STEP_LAUNCH(9); break;
      case 10: SWARM_STEP_LAUNCH(10); break;
      case 11: SWARM_STEP_LAUNCH(11); break;
      case 12: SWARM_STEP_LAUNCH(12); break;
      default: SWARM_STEP_LAUNCH(0); break;
    }
#undef SWARM_STEP_LAUNCH
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    env0 = ntiles * epb_s;
    if (env0 == num_envs) return cudaSuccess;
    const long long a0 = env0 * N;
    p.state_in += a0;
    p.actions += a0;
    p.state_out += a0;
    if (p.rewards) p.rewards += a0;
    if (p.flags) p.flags += a0;
    if (p.contact) p.contact += a0;
    if (p.obs) p.obs += a0 * 6;
    if (p.dist) p.dist += a0;
    p.cfg.num_envs = (int)(num_envs - env0);
  }
  p.epb = kStepThreads / N;
  const long long grid = ((long long)p.cfg.num_envs + p.epb - 1) / p.epb;
  sim_step_kernel<<<(unsigned)grid, kStepThreads, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace swarm
