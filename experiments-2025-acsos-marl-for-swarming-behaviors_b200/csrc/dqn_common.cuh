// dqn_common.cuh -- parameter block of the DQN gradient kernel (dqn_tc_kernels.cu, launched from dqn_kernels.cu) and
// what the device-driven tick and the clip + Adam kernels share.
#ifndef SWARM_DQN_COMMON_CUH
#define SWARM_DQN_COMMON_CUH

#include "tile_device.cuh"

namespace swarm {

constexpr int kPartialStride = 1680;   // 1673 gradients + [1673] = sum of squared TD errors, padded
constexpr int kXPad = 8;

struct DqnParams {
  SwarmConfig cfg;
  const float* w_online;
  const float* w_target;
  SwarmReplay batch;
  const int64_t* indices;
  int32_t n_graphs;
  float gamma;
  float loss_scale;
  float* partials;
  float* td;
  int32_t epb, maxdeg;
  float qmax_r;               // radius graph threshold (see TileParams)
  // device-driven tick (swarm_train_tick_grad): slots are drawn here from the ring fill after this tick's push
  const SwarmTrainCtl* ctl;
  int64_t* indices_out;       // [n_graphs] the drawn slots (exported for tests / logging)
  unsigned long long sample_seed;
  int32_t pushed_envs;        // transitions pushed by this tick's rollout
};

// ring fill after this tick's push, and whether it allows an update (train:113-115)
__device__ __forceinline__ long long train_ring_size(const SwarmTrainCtl* ctl, int pushed, long long capacity) {
  const long long size = ctl->ring_size + pushed;
  return size < capacity ? size : capacity;
}

// end of a device-driven tick: tick, ring cursor / fill and (after an update) the optimiser step advance; shared by the
// clip + Adam kernels of the one-layer network and of stacked networks
__device__ __forceinline__ void train_ctl_advance(SwarmTrainCtl* ctl, int num_envs, long long capacity, bool stepped) {
  ctl->tick += 1;
  ctl->ring_cursor = (ctl->ring_cursor + num_envs) % capacity;
  const long long sz = ctl->ring_size + num_envs;
  ctl->ring_size = sz < capacity ? sz : capacity;
  if (stepped) ctl->opt_step += 1;
}

// one Adam step of one element, op for op as torch.optim.Adam (single-tensor path); shared by the clip + Adam kernels
// of the one-layer network (dqn_kernels.cu) and of stacked networks (stack_grad_kernels.cu)
struct AdamScalars {
  float lerp_w, beta2, one_minus_beta2, neg_step_size, bc2_sqrt, eps;
};
__device__ __forceinline__ void adam_element(const AdamScalars& a, float g, float coef, float& m_io, float& v_io, float& w_io) {
  const float gval = __fmul_rn(g, coef);
  // exp_avg.lerp_(grad, 1 - beta1)
  const float m = __fadd_rn(m_io, __fmul_rn(a.lerp_w, __fsub_rn(gval, m_io)));
  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value = 1 - beta2)
  float v = __fmul_rn(v_io, a.beta2);
  v = __fadd_rn(v, __fmul_rn(__fmul_rn(a.one_minus_beta2, gval), gval));
  // denom = sqrt(v) / sqrt(bias_correction2) + eps ; param.addcdiv_(exp_avg, denom, value = -step_size)
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), a.bc2_sqrt), a.eps);
  w_io = __fadd_rn(w_io, __fdiv_rn(__fmul_rn(a.neg_step_size, m), denom));
  m_io = m;
  v_io = v;
}

// the peer-memory gradient exchange of the data-parallel ticks (adam_clip_kernel<true> / reduce_clip_adam_kernel<true>
// in dqn_kernels.cu, stack_reduce_peers_kernel in stack_grad_kernels.cu): one naturally aligned 64-bit word =
// (epoch << 32 | float bits) is single-copy atomic, so the word itself is the flag
__device__ __forceinline__ void st_relaxed_sys_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed_sys_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

}  // namespace swarm
#endif
