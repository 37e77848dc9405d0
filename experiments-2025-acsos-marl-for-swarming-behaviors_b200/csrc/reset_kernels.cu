// reset_kernels.cu -- generate_grid + reset_world_at (go_to_position_scenario.py:52-106,
// obstacle_avoidance_scenario.py:63-133): one thread per agent, float4 state writes.
#include "tile_device.cuh"
#include "launchers.h"

namespace swarm {

// The grid offsets (Python doubles cast to float32, go_to:68-76) are the same for every env: each CTA computes the N
// float2 offsets once in shared memory, so the per-agent work is two float adds and one 16-byte store (the double
// arithmetic per agent made the first version FP64-bound at 55 % of the HBM peak).
constexpr int kResetMaxSmemAgents = 4096;

__device__ __forceinline__ void stage_grid_offsets(float2* soff, int n, int cols, int rows, double spacing) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int r = i / cols, q = i % cols;
    soff[i] = make_float2((float)(((double)q - (double)(cols - 1) / 2.0) * spacing),
                          (float)(((double)r - (double)(rows - 1) / 2.0) * spacing));
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256) reset_grid_kernel(SwarmConfig c, int cols, int rows,
                                                         const float2* __restrict__ centers,
                                                         float4* __restrict__ state) {
  extern __shared__ float2 soff[];
  stage_grid_offsets(soff, c.n_agents, cols, rows, c.grid_spacing);
  const long long total = (long long)c.num_envs * c.n_agents;
  const unsigned n = (unsigned)c.n_agents;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const long long env = g / n;
    const int i = (int)(g - env * n);
    const float2 ctr = centers[env];
    const float2 o = soff[i];
    state[g] = make_float4(__fadd_rn(ctr.x, o.x), __fadd_rn(ctr.y, o.y), 0.0f, 0.0f);
  }
}

cudaError_t launch_reset_grid(const SwarmConfig& c, int cols, int rows, const float* centers, float* state,
                              cudaStream_t stream) {
  const long long total = (long long)c.num_envs * c.n_agents;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  reset_grid_kernel<<<(int)blocks, 256, c.n_agents * sizeof(float2), stream>>>(
      c, cols, rows, reinterpret_cast<const float2*>(centers), reinterpret_cast<float4*>(state));
  return cudaGetLastError();
}

// ---- device-side episode boundary ---------------------------------------------------------------------------
// centre of env b for episode e: base + (mean + std * z), z ~ N(0,1)^2 by Box-Muller on two counter-RNG uniforms
__device__ __forceinline__ float2 draw_center(const SwarmResetSpec& sp, long long genv, long long episode) {
  const uint64_t r = rng_draw(sp.seed, (uint64_t)genv, (uint64_t)episode, 0xC3A7u);
  const float u1 = ((float)(r >> 40) + 1.0f) * (1.0f / 16777216.0f);          // (0, 1]
  const float u2 = (float)((r >> 16) & 0xFFFFFFull) * (1.0f / 16777216.0f);   // [0, 1)
  const float rad = sqrtf(-2.0f * logf(u1));
  float sn, cs;
  sincosf(6.28318530717958647692f * u2, &sn, &cs);
  return make_float2(__fadd_rn(sp.base_x, __fadd_rn(sp.mean_x, sp.std_x * (rad * cs))),
                     __fadd_rn(sp.base_y, __fadd_rn(sp.mean_y, sp.std_y * (rad * sn))));
}

__global__ void __launch_bounds__(256) reset_random_kernel(SwarmConfig c, SwarmResetSpec sp, int cols, int rows,
                                                           const SwarmTrainCtl* __restrict__ ctl, long long episode,
                                                           float2* __restrict__ centers_out, float4* __restrict__ state) {
  extern __shared__ float2 soff[];
  stage_grid_offsets(soff, c.n_agents, cols, rows, c.grid_spacing);
  if (ctl) episode = ctl->episode;
  const long long total = (long long)c.num_envs * c.n_agents;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const long long env = g / c.n_agents;
    const int i = (int)(g - env * c.n_agents);
    const float2 ctr = draw_center(sp, sp.shared_center ? 0 : sp.env_offset + env, episode);
    if (centers_out && i == 0) centers_out[env] = ctr;
    const float2 o = soff[i];
    state[g] = make_float4(__fadd_rn(ctr.x, o.x), __fadd_rn(ctr.y, o.y), 0.0f, 0.0f);
  }
}

__global__ void __launch_bounds__(256) episode_end_kernel(SwarmConfig c, SwarmTrainCtl* ctl, float* __restrict__ returns,
                                                          int32_t* __restrict__ hits, const float* __restrict__ loss,
                                                          float* __restrict__ stats, long long max_episodes,
                                                          double eps0, double decay, double min_eps) {
  __shared__ double sret[256];
  __shared__ long long shit[256];
  const int tid = threadIdx.x;
  const int B = c.num_envs, N = c.n_agents;
  double r = 0.0;
  long long h = 0;
  for (int b = tid; b < B; b += 256) {
    r += (double)returns[(long long)b * N];          // agent 0's return (train:178,183)
    if (hits) h += hits[b];
  }
  sret[tid] = r;
  shit[tid] = h;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (tid < s) { sret[tid] += sret[tid + s]; shit[tid] += shit[tid + s]; }
    __syncthreads();
  }
  const long long ep = ctl->episode;
  const float eps_used = ctl->epsilon;
  __syncthreads();
  // zero the accumulators for the next episode
  for (long long g = tid; g < (long long)B * N; g += 256) returns[g] = 0.0f;
  if (hits) for (int b = tid; b < B; b += 256) hits[b] = 0;
  if (tid == 0) {
    if (stats && ep < max_episodes) {
      float* row = stats + ep * 4;
      row[0] = (float)(sret[0] / (double)N / (double)B);
      row[1] = (float)((double)shit[0] / (double)B);
      row[2] = (loss && ctl->opt_step > 0) ? loss[0] : 0.0f;
      row[3] = eps_used;
    }
    const double e = eps0 * exp(-decay * (double)ep);          // train:180 with the finished episode's index
    ctl->epsilon = (float)(e > min_eps ? e : min_eps);
    ctl->episode = ep + 1;
  }
}

cudaError_t launch_reset_random(const SwarmConfig& c, const SwarmResetSpec& sp, int cols, int rows, const SwarmTrainCtl* ctl,
                                long long episode, float* centers_out, float* state, cudaStream_t stream) {
  const long long total = (long long)c.num_envs * c.n_agents;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  reset_random_kernel<<<(int)blocks, 256, c.n_agents * sizeof(float2), stream>>>(c, sp, cols, rows, ctl, episode,
                                                       reinterpret_cast<float2*>(centers_out),
                                                       reinterpret_cast<float4*>(state));
  return cudaGetLastError();
}

cudaError_t launch_episode_end(const SwarmConfig& c, SwarmTrainCtl* ctl, float* returns, int32_t* hits, const float* loss,
                               float* stats, long long max_episodes, double eps0, double decay, double min_eps,
                               cudaStream_t stream) {
  episode_end_kernel<<<1, 256, 0, stream>>>(c, ctl, returns, hits, loss, stats, max_episodes, eps0, decay, min_eps);
  return cudaGetLastError();
}

}  // namespace swarm
