// dqn_kernels.cu -- the rest of the one-layer DQN update on the device (train_gcn_dqn.py:112-137) around the
// gradient kernel of dqn_tc_kernels.cu:
//   dqn_reduce_kernel        the per-CTA partial gradients summed in CTA order (no atomics: bit-reproducible)
//   adam_clip_kernel         clip_grad_norm_ + torch.optim.Adam (+ target copy) in one CTA
//   reduce_clip_adam_kernel  the two as one thread-block cluster (swarm_train_tick)
//   csr_bwd_*_kernel         the GCN backward on an arbitrary CSR graph (the nn.Module seam)
// and the launchers of the whole update.
#include <cooperative_groups.h>

#include "dqn_common.cuh"
#include "launchers.h"

namespace swarm {

__device__ __forceinline__ void store_row32(float* tile, int row, const float (&v)[32]) {
  float4* r = reinterpret_cast<float4*>(tile + row * kHPad);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) r[c4] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
}
__device__ __forceinline__ void load_row32(const float* tile, int row, float (&v)[32]) {
  const float4* r = reinterpret_cast<const float4*>(tile + row * kHPad);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) {
    const float4 q = r[c4];
    v[4 * c4] = q.x; v[4 * c4 + 1] = q.y; v[4 * c4 + 2] = q.z; v[4 * c4 + 3] = q.w;
  }
}
__device__ __forceinline__ float f4c(const float4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

// acc[0..3] += sum_{n < rows} A[n*lda + ac] * B[n*ldb + bc .. bc+3]   (A == nullptr: column of ones)
__device__ __forceinline__ float4 tile_gemm4(const float* A, int lda, int ac, const float* B, int ldb, int bc, int rows) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int n = 0; n < rows; ++n) {
    const float a = A ? A[n * lda + ac] : 1.0f;
    const float4 b = *reinterpret_cast<const float4*>(B + n * ldb + bc);
    acc.x = fmaf(a, b.x, acc.x);
    acc.y = fmaf(a, b.y, acc.y);
    acc.z = fmaf(a, b.z, acc.z);
    acc.w = fmaf(a, b.w, acc.w);
  }
  return acc;
}

// (aggregate + conv1.bias) -> tanh -> lin1 -> ReLU -> lin2 with the same arithmetic as gat_head_keep
// (gatq_device.cuh), but ROLLED: the k loops run four input channels per iteration and read the layer input back
// from the thread's own shared-memory row, so the body is ~160 instructions instead of ~1 300 fully unrolled.
// The kernel executes every instruction once per warp, i.e. it streams its own code: size is what it pays for.
// On return urow = u = tanh(agg + b0), rrow / r = relu(W1 u + b1).
__device__ __forceinline__ void dqn_head(const float (&agg)[32], float* __restrict__ urow, float* __restrict__ rrow,
                                         const float* __restrict__ sw, float (&r)[32], float (&q)[9]) {
  float4* u4 = reinterpret_cast<float4*>(urow);
  float4* r4 = reinterpret_cast<float4*>(rrow);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) u4[c4] = make_float4(agg[4 * c4], agg[4 * c4 + 1], agg[4 * c4 + 2], agg[4 * c4 + 3]);
  const float4* b0 = reinterpret_cast<const float4*>(sw + TW_B0);
#pragma unroll 1
  for (int c4 = 0; c4 < 8; ++c4) {
    float4 v = u4[c4];
    const float4 b = b0[c4];
    v.x = tanhf(__fadd_rn(v.x, b.x));
    v.y = tanhf(__fadd_rn(v.y, b.y));
    v.z = tanhf(__fadd_rn(v.z, b.z));
    v.w = tanhf(__fadd_rn(v.w, b.w));
    u4[c4] = v;
  }
#pragma unroll
  for (int cc = 0; cc < 32; ++cc) r[cc] = 0.0f;
  const float4* w1 = reinterpret_cast<const float4*>(sw + TW_W1T);
#pragma unroll 1
  for (int k4 = 0; k4 < 8; ++k4) {
    const float4 uk = u4[k4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float a = f4c(uk, kk);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 w = w1[(k4 * 4 + kk) * 8 + c4];
        r[4 * c4 + 0] = fmaf(a, w.x, r[4 * c4 + 0]);
        r[4 * c4 + 1] = fmaf(a, w.y, r[4 * c4 + 1]);
        r[4 * c4 + 2] = fmaf(a, w.z, r[4 * c4 + 2]);
        r[4 * c4 + 3] = fmaf(a, w.w, r[4 * c4 + 3]);
      }
    }
  }
  const float* b1 = sw + TW_B1;
#pragma unroll
  for (int cc = 0; cc < 32; ++cc) r[cc] = fmaxf(__fadd_rn(r[cc], b1[cc]), 0.0f);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) r4[c4] = make_float4(r[4 * c4], r[4 * c4 + 1], r[4 * c4 + 2], r[4 * c4 + 3]);

  float qq[kW2Pad];
#pragma unroll
  for (int a = 0; a < kW2Pad; ++a) qq[a] = 0.0f;
  const float4* w2 = reinterpret_cast<const float4*>(sw + TW_W2T);
#pragma unroll 1
  for (int k4 = 0; k4 < 8; ++k4) {
    const float4 rk = r4[k4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float a = f4c(rk, kk);
#pragma unroll
      for (int a4 = 0; a4 < 3; ++a4) {
        const float4 w = w2[(k4 * 4 + kk) * 3 + a4];
        qq[4 * a4 + 0] = fmaf(a, w.x, qq[4 * a4 + 0]);
        qq[4 * a4 + 1] = fmaf(a, w.y, qq[4 * a4 + 1]);
        qq[4 * a4 + 2] = fmaf(a, w.z, qq[4 * a4 + 2]);
        qq[4 * a4 + 3] = fmaf(a, w.w, qq[4 * a4 + 3]);
      }
    }
  }
  const float* b2 = sw + TW_B2;
#pragma unroll
  for (int a = 0; a < 9; ++a) q[a] = __fadd_rn(qq[a], b2[a]);
}

// grad[o] = sum over CTAs (in CTA order) of partials[cta][o]; loss = loss_scale * sum of squared TD errors
__global__ void __launch_bounds__(256) dqn_reduce_kernel(const float* __restrict__ partials, int n_ctas, float loss_scale,
                                                         float* __restrict__ grad, float* __restrict__ loss,
                                                         SwarmTrainCtl* __restrict__ ctl, int pushed_envs,
                                                         long long capacity, int n_graphs) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (ctl) {
    // device-driven tick: publish whether this tick updates (read by the clip + Adam kernel)
    const bool upd = train_ring_size(ctl, pushed_envs, capacity) >= n_graphs;
    if (o == 0) ctl->updating = upd ? 1 : 0;
    if (!upd) return;
  }
  if (o > SWARM_W_COUNT) return;
  float acc = 0.0f;
  for (int b = 0; b < n_ctas; ++b) acc += partials[(long long)b * kPartialStride + o];
  if (o < SWARM_W_COUNT) grad[o] = acc;
  else loss[0] = acc * loss_scale;
}

// ---- clip_grad_norm_ + Adam (+ optional target copy), one CTA ---------------------------------------
struct AdamParams {
  float* w;
  const float* grad;
  float* m;
  float* v;
  float* target;
  float* grad_norm;
  float lerp_w;          // 1 - beta1
  float beta2;
  float one_minus_beta2;
  float neg_step_size;   // -(lr / (1 - beta1^t))
  float bc2_sqrt;        // sqrt(1 - beta2^t)
  float eps;
  float max_norm;
  // device-driven variant (swarm_train_tick_apply): step-dependent scalars are derived from *ctl on the device and
  // the cursor is advanced at the end
  SwarmTrainCtl* ctl;
  double lr, beta1, beta2d;
  long long ring_capacity;
  int32_t num_envs;
  int32_t update_target_every;
  // fused one-shot all-reduce over peer memory (ctl mode only); world_size <= 1: off
  SwarmPeerExchange peers;
  float* grad_rw;          // same buffer as `grad` (gradient + loss), written back after the exchange
  // reduce_clip_adam_kernel only: the gradient kernel's per-CTA partials
  const float* partials;   // [n_ctas][kPartialStride]
  int32_t n_ctas;
  int32_t n_graphs;
  float loss_scale;
};

constexpr int kAdamPer = (SWARM_W_COUNT + 1 + 255) / 256;      // elements per thread; + 1: the loss rides along

// torch.nn.utils.clip_grad_norm_: norms = [||g_t||_2 for each parameter tensor]; total = ||norms||_2.  g_[i] is element
// tid + 256 i of the gradient (0 beyond it); returns the clip coefficient on every thread (one block barrier inside).
// Shared by the two clip + Adam kernels so that both form the sums in the same order.
__device__ __forceinline__ float clip_coefficient(const float (&g_)[kAdamPer], double (&swarp)[8][8], float& s_coef,
                                                  float max_norm, float* grad_norm_out, bool pre_synced = false) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int seg_off[9] = {SWARM_W_CONV_LIN, SWARM_W_ATT_SRC, SWARM_W_ATT_DST, SWARM_W_CONV_BIAS, SWARM_W_LIN1,
                          SWARM_W_LIN1_BIAS, SWARM_W_LIN2, SWARM_W_LIN2_BIAS, SWARM_W_COUNT};
#pragma unroll
  for (int sgi = 0; sgi < 8; ++sgi) {
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < kAdamPer; ++i) {
      const int o = tid + 256 * i;
      if (o >= seg_off[sgi] && o < seg_off[sgi + 1]) acc += (double)g_[i] * (double)g_[i];
    }
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, sh);
    if (lane == 0) swarp[sgi][warp] = acc;
  }
  __syncthreads();
  if (tid < 32) {
    // lane s < 8: the norm of parameter tensor s (its warps' partial sums in warp order); lane 0 then adds the eight
    // squares in tensor order -- the sums of the serial loop, with the eight tensors' chains side by side
    double sq = 0.0;
    if (tid < 8) {
      double ss = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) ss += swarp[tid][w];
      const float nrm = (float)sqrt(ss);
      sq = (double)nrm * (double)nrm;
    }
    double tot = 0.0;
#pragma unroll
    for (int sgi = 0; sgi < 8; ++sgi) tot += __shfl_sync(0xffffffffu, sq, sgi);
    if (tid == 0) {
    const float total_norm = (float)sqrt(tot);
    float coef = 1.0f;
    if (max_norm > 0.0f) {
      coef = max_norm / (total_norm + 1e-6f);
      coef = coef > 1.0f ? 1.0f : coef;
    }
    s_coef = coef;
    if (grad_norm_out) grad_norm_out[0] = total_norm;
    }
  }
  __syncthreads();
  return s_coef;
}

// PEERS: with the fused peer-memory all-reduce (its register arrays and system-scope loads would otherwise slow the
// single-GPU kernel from 5.4 to 7.6 us)
template <bool PEERS>
__global__ void __launch_bounds__(256) adam_clip_kernel(AdamParams p) {
  __shared__ double swarp[8][8];            // [segment][warp] partial sums of squares
  __shared__ float s_coef, s_neg_step, s_bc2_sqrt;
  __shared__ int s_update, s_sync;
  const int tid = threadIdx.x;
  // every thread owns the elements tid, tid + 256, ...: one round trip to memory for grad / m / v / w, everything
  // else from registers
  constexpr int kPer = kAdamPer;                             // + 1: the loss rides along in the exchange
  float g_[kPer], m_[kPer], v_[kPer], w_[kPer];
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int o = tid + 256 * i;
    const bool in = o < SWARM_W_COUNT;
    g_[i] = (in || (PEERS && o == SWARM_W_COUNT)) ? p.grad[o] : 0.0f;
    m_[i] = in ? p.m[o] : 0.0f;
    v_[i] = in ? p.v[o] : 0.0f;
    w_[i] = in ? p.w[o] : 0.0f;
  }
  if (p.ctl && tid == 255) {
    // step-dependent scalars from the device cursor (after this warp's loads went out: the two pow chains run
    // under their latency)
    const long long step = p.ctl->opt_step + 1;
    const double bc1 = 1.0 - pow(p.beta1, (double)step);
    const double bc2 = 1.0 - pow(p.beta2d, (double)step);
    s_neg_step = (float)(-(p.lr / bc1));
    s_bc2_sqrt = (float)sqrt(bc2);
    s_update = p.ctl->updating;
    s_sync = ((p.ctl->tick + 1) % p.update_target_every) == 0;
  }
  if (PEERS && p.ctl) {
    // ---- one-shot PUSH all-reduce over NVLink peer memory ("low-latency" protocol) ---------------------------
    // Every rank agrees on `updating` (the trainer checks that all shards have the same env count and ring fill), so
    // either all ranks exchange this tick or none does.  Each rank WRITES its partial gradient + loss into its own
    // slot of every peer's receive buffer; each 8-byte word carries the value and the epoch (tick + 1), so a word is
    // its own arrival flag: no fence, no separate flag, and the waits poll LOCAL memory.  The critical path is one
    // one-way NVLink store latency (the pull version paid a remote flag poll plus two remote read round trips).
    // Slots are double-buffered by epoch parity: a rank can only be one exchange ahead of a peer, because its next
    // push needs the peer's words of the current one.
    const uint32_t epoch = (uint32_t)(p.ctl->tick + 1);
    const int par = (int)(epoch & 1u);
    const int W = p.peers.world_size;
    const bool upd = p.ctl->updating != 0;
    if (upd) {
      uint64_t word[kPer];
#pragma unroll
      for (int i = 0; i < kPer; ++i) word[i] = ((uint64_t)epoch << 32) | (uint64_t)__float_as_uint(g_[i]);
      const size_t my_slot = ((size_t)par * W + p.peers.rank) * SWARM_XCHG_STRIDE;
      for (int q = 0; q < W; ++q) {
        const int peer = (p.peers.rank + q) % W;            // own buffer first, then ring order: spreads the links
        uint64_t* dst = p.peers.data[peer] + my_slot;
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
          const int o = tid + 256 * i;
          if (o <= SWARM_W_COUNT) st_relaxed_sys_u64(dst + o, word[i]);
        }
      }
      // rank order on every rank: bit-identical sums
#pragma unroll
      for (int i = 0; i < kPer; ++i) g_[i] = 0.0f;
      const uint64_t* mine = p.peers.data[p.peers.rank] + (size_t)par * W * SWARM_XCHG_STRIDE;
      // the slots of four ranks are polled together (28 loads in flight per thread): a poll is a round trip to memory, and
      // waiting rank by rank made the exchange cost grow with the world size (8 ranks: eight round trips)
      constexpr int kGroup = 4;
      for (int r0 = 0; r0 < W; r0 += kGroup) {
        uint64_t got[kGroup][kPer];
        bool ok = false;
        for (long long it = 0; it < (1ll << 26) && !ok; ++it) {     // bounded: a lost peer traps instead of hanging
          ok = true;
#pragma unroll
          for (int q = 0; q < kGroup; ++q) {
            const uint64_t* src = mine + (size_t)(r0 + q) * SWARM_XCHG_STRIDE;
            const bool live = r0 + q < W;
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
              const int o = tid + 256 * i;
              got[q][i] = (live && o <= SWARM_W_COUNT) ? ld_relaxed_sys_u64(src + o) : ((uint64_t)epoch << 32);
            }
          }
#pragma unroll
          for (int q = 0; q < kGroup; ++q)
#pragma unroll
            for (int i = 0; i < kPer; ++i) ok = ok && ((uint32_t)(got[q][i] >> 32) == epoch);
        }
        if (!ok) __trap();
#pragma unroll
        for (int q = 0; q < kGroup; ++q)
#pragma unroll
          for (int i = 0; i < kPer; ++i) g_[i] += __uint_as_float((uint32_t)got[q][i]);       // rank order; absent ranks add +0
      }
#pragma unroll
      for (int i = 0; i < kPer; ++i) {
        const int o = tid + 256 * i;
        if (o <= SWARM_W_COUNT) p.grad_rw[o] = g_[i];      // reduced gradient + loss for the host-side statistics
      }
    }
  }
  __syncthreads();
  if (p.ctl) {
    p.neg_step_size = s_neg_step;
    p.bc2_sqrt = s_bc2_sqrt;
    if (!s_sync) p.target = nullptr;
    if (!s_update) {
      if (tid == 0) train_ctl_advance(p.ctl, p.num_envs, p.ring_capacity, false);
      return;
    }
  }
  const float coef = clip_coefficient(g_, swarp, s_coef, p.max_norm, p.grad_norm);
  const AdamScalars sc{p.lerp_w, p.beta2, p.one_minus_beta2, p.neg_step_size, p.bc2_sqrt, p.eps};
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int o = tid + 256 * i;
    if (o >= SWARM_W_COUNT) break;
    adam_element(sc, g_[i], coef, m_[i], v_[i], w_[i]);
    p.m[o] = m_[i];
    p.v[o] = v_[i];
    p.w[o] = w_[i];
    if (p.target) p.target[o] = w_[i];
  }
  if (p.ctl && tid == 0) train_ctl_advance(p.ctl, p.num_envs, p.ring_capacity, true);
}

// ---- partial reduction (+ peer exchange) + clip + Adam as ONE launch (swarm_train_tick) ----------------------------
// The two small launches at the end of a tick (dqn_reduce_kernel on 7 CTAs, adam_clip_kernel on one) as a single
// thread-block cluster of 7 working CTAs x 256 threads (launched as the portable size 8; the spare CTA computes the
// step's Adam scalars), one gradient element per thread:
//   1. element o = 256 c + t: the sum of the gradient kernel's partials in CTA order (dqn_reduce_kernel's sum);
//   2. every CTA pushes its 256 sums into the shared memory of all seven (distributed shared memory), one cluster
//      barrier, and every CTA holds the whole gradient laid out as adam_clip_kernel's registers are ([i][tid]), so the
//      clip coefficient is formed by the same code in the same order on every CTA -- no second exchange;
//   3. Adam on the CTA's own 256 elements; CTA 0 advances the device cursor.
// Same bits as the two launches.  A single CTA cannot do step 1 at this speed: the 32 x 6.7 KB of partials through one
// SM's L2 port cost as much as the launch they would save (tried: 34.8 vs 34.6 us per tick).

// split cluster barrier: every CTA arrives when it starts and waits just before its first store into a peer CTA's shared
// memory -- a CTA must have started executing before its shared memory is written remotely
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

constexpr int kAdamCluster = 8;
static_assert(kAdamPer <= kAdamCluster, "one CTA per 256 gradient elements");
// PEERS: the one-shot PUSH all-reduce of adam_clip_kernel<true> (same slots, same words, same rank-order sums -- see
// there), with one element per thread: every thread pushes ONE word per peer and polls world_size local words, all in
// flight together, and the seven CTAs use seven SMs' worth of NVLink store and poll bandwidth.
template <bool PEERS>
__global__ void __cluster_dims__(kAdamCluster, 1, 1) __launch_bounds__(256) reduce_clip_adam_kernel(AdamParams p) {
  namespace cg = cooperative_groups;
  __shared__ float sg[kAdamPer][256];
  __shared__ double swarp[8][8];
  __shared__ float s_coef, s_neg_step, s_bc2_sqrt;
  __shared__ int s_sync;
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x, c = (int)cluster.block_rank();
  cluster_arrive_relaxed();
  if (c >= kAdamPer) {
    // the spare CTA of the cluster: the step-dependent scalars (two double-precision pow chains, about a microsecond on
    // one thread each) computed beside the other CTAs' loads and delivered into their shared memory
    float fv = 0.0f;
    int iv = 0;
    if (tid == 0 || tid == 32 || tid == 64) {
      const long long step = p.ctl->opt_step + 1;
      if (tid == 0) fv = (float)(-(p.lr / (1.0 - pow(p.beta1, (double)step))));
      else if (tid == 32) fv = (float)sqrt(1.0 - pow(p.beta2d, (double)step));
      else iv = ((p.ctl->tick + 1) % p.update_target_every) == 0;
    }
    __syncwarp();
    cluster_wait();
    if (tid == 0 || tid == 32 || tid == 64) {
      for (int r = 0; r < kAdamPer; ++r) {
        if (tid == 0) *cluster.map_shared_rank(&s_neg_step, r) = fv;
        else if (tid == 32) *cluster.map_shared_rank(&s_bc2_sqrt, r) = fv;
        else *cluster.map_shared_rank(&s_sync, r) = iv;
      }
    }
    cluster.sync();
    return;
  }
  const int o = 256 * c + tid;
  const bool upd = train_ring_size(p.ctl, p.num_envs, p.ring_capacity) >= p.n_graphs;
  const bool in = o < SWARM_W_COUNT;
  float m = in ? p.m[o] : 0.0f, v = in ? p.v[o] : 0.0f, w = in ? p.w[o] : 0.0f;
  float g = 0.0f;
  if (o <= SWARM_W_COUNT) {
    // not conditional on `upd`: the loads go out beside the cursor's (a tick that does not update reads stale partials
    // and drops them)
    const float* src = p.partials + o;
    constexpr int kBatch = 32;       // the reference's 32 graphs: one CTA each, all partials of an element in flight
    for (int b0 = 0; b0 < p.n_ctas; b0 += kBatch) {
      float part[kBatch];
#pragma unroll
      for (int b = 0; b < kBatch; ++b) part[b] = (b0 + b < p.n_ctas) ? __ldcg(src + (size_t)(b0 + b) * kPartialStride) : 0.0f;
#pragma unroll
      for (int b = 0; b < kBatch; ++b)
        if (b0 + b < p.n_ctas) g += part[b];
    }
  }
  if (!upd) g = 0.0f;
  if (upd && o <= SWARM_W_COUNT) {
    if (o == SWARM_W_COUNT) g *= p.loss_scale;      // the loss rides along (exchange, caller's statistics)
    if (PEERS) {
      const uint32_t epoch = (uint32_t)(p.ctl->tick + 1);
      const int W = p.peers.world_size;
      const size_t par_base = (size_t)(epoch & 1u) * W * SWARM_XCHG_STRIDE;
      const uint64_t word = ((uint64_t)epoch << 32) | (uint64_t)__float_as_uint(g);
      for (int q = 0; q < W; ++q) {
        const int peer = (p.peers.rank + q) % W;            // own buffer first, then ring order: spreads the links
        st_relaxed_sys_u64(p.peers.data[peer] + par_base + (size_t)p.peers.rank * SWARM_XCHG_STRIDE + o, word);
      }
      const uint64_t* mine = p.peers.data[p.peers.rank] + par_base + o;
      uint64_t got[SWARM_MAX_PEERS];
      bool ok = false;
      for (long long it = 0; it < (1ll << 26) && !ok; ++it) {       // bounded: a lost peer traps instead of hanging
        ok = true;
#pragma unroll
        for (int r = 0; r < SWARM_MAX_PEERS; ++r)
          got[r] = (r < W) ? ld_relaxed_sys_u64(mine + (size_t)r * SWARM_XCHG_STRIDE) : ((uint64_t)epoch << 32);
#pragma unroll
        for (int r = 0; r < SWARM_MAX_PEERS; ++r) ok = ok && ((uint32_t)(got[r] >> 32) == epoch);
      }
      if (!ok) __trap();
      g = 0.0f;
#pragma unroll
      for (int r = 0; r < SWARM_MAX_PEERS; ++r) g += __uint_as_float((uint32_t)got[r]);     // rank order; absent ranks add +0
    }
    p.grad_rw[o] = g;
    if (o == SWARM_W_COUNT) g = 0.0f;
  }
  __syncwarp();
  cluster_wait();
#pragma unroll
  for (int r = 0; r < kAdamPer; ++r) *cluster.map_shared_rank(&sg[c][tid], r) = g;
  cluster.sync();       // every read of *ctl above precedes CTA 0's writes below
  if (!upd) {
    if (c == 0 && tid == 0) {
      p.ctl->updating = 0;
      train_ctl_advance(p.ctl, p.num_envs, p.ring_capacity, false);
    }
    return;
  }
  float g_[kAdamPer];
#pragma unroll
  for (int i = 0; i < kAdamPer; ++i) g_[i] = sg[i][tid];
  const float coef = clip_coefficient(g_, swarp, s_coef, p.max_norm, c == 0 ? p.grad_norm : nullptr);
  if (in) {
    const AdamScalars sc{p.lerp_w, p.beta2, p.one_minus_beta2, s_neg_step, s_bc2_sqrt, p.eps};
    adam_element(sc, g, coef, m, v, w);
    p.m[o] = m;
    p.v[o] = v;
    p.w[o] = w;
    if (s_sync && p.target) p.target[o] = w;
  }
  if (c == 0 && tid == 0) {
    p.ctl->updating = 1;
    train_ctl_advance(p.ctl, p.num_envs, p.ring_capacity, true);
  }
}

// ---- GCN backward on an arbitrary graph ------------------------------------------------------------------------
// The nn.Module seam: loss.backward() through GCN.forward(data) for any Data / Batch graph (train_gcn_dqn.py:116-124
// when the reference's own train_step_dqn drives the module).  Two gather passes, no atomics:
//   csr_bwd_target_kernel  thread = target node: recomputes its forward (softmax over the in-edge group in edge-list
//                          order, head), back-propagates the head, and for every in-edge stores alpha_e and
//                          d(raw logit)_e in by-target order; per-CTA tile GEMMs give the head's weight gradients
//   csr_bwd_source_kernel  thread = source node: gathers its out-edges (CSR by source) to form d h_j, then the tile
//                          GEMMs for conv1.lin.weight / att_src / att_dst
// followed by the same fixed-order partial reduction as the DQN gradient (bit-reproducible).
constexpr int kRowB = 36;   // rows workspace of csr_kernels.cu: h[32], alpha_src, alpha_dst, pad

struct CsrBwdParams {
  int n;
  const float* weights;
  const float* x;
  const int32_t* row_ptr;      // CSR by target (edge-list order inside a group)
  const int32_t* src;
  const int32_t* row_ptr_s;    // CSR by source
  const int32_t* tgt_s;
  const int32_t* pos_s;        // position in the by-target order of out-edge q
  const float* grad_q;         // [n][9]; conv_only: d(conv output) [n][32]
  int conv_only;               // 1: the GATConv layer alone (no head): gradients of conv1.* only
  const float* rows;           // [n][36] projected features (csr_project_kernel)
  float* d_out;                // [n][32] d(conv output)
  float* dd;                   // [n] d(alpha_dst)
  float* alpha;                // [E] attention coefficients, by-target order
  float* draw;                 // [E] d(raw logit), by-target order
  float* partials;             // [ctas][kPartialStride]
};

__global__ void csr_edge_positions_kernel(long long E, const int32_t* __restrict__ perm_t,
                                          const int32_t* __restrict__ perm_s, int32_t* __restrict__ inv,
                                          int32_t* __restrict__ pos_s, int phase) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
    if (phase == 0) inv[perm_t[e]] = (int32_t)e;          // original edge id -> by-target position
    else pos_s[e] = inv[perm_s[e]];
  }
}

__global__ void __launch_bounds__(kTileThreads) csr_bwd_target_kernel(const __grid_constant__ CsrBwdParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int T = kTileThreads;
  float* sw = reinterpret_cast<float*>(smem);
  float* tU = sw + ((TW_COUNT + 3) & ~3);
  float* tR = tU + T * kHPad;
  float* tDP = tR + T * kHPad;
  float* tDO = tDP + T * kHPad;
  float* tDQ = tDO + T * kHPad;
  const int tid = threadIdx.x;
  const int i = blockIdx.x * T + tid;
  const bool active = i < p.n;
  stage_weights(p.weights, sw, tid, T);
  if (!active) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    float* tiles[4] = {tU, tR, tDP, tDO};
#pragma unroll 1
    for (int b = 0; b < 4; ++b) {
      float4* row = reinterpret_cast<float4*>(tiles[b] + tid * kHPad);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) row[c4] = z;
    }
#pragma unroll
    for (int a = 0; a < kW2Pad; ++a) tDQ[tid * kW2Pad + a] = 0.0f;
  }
  __syncthreads();
  if (active) {
    const int e0 = p.row_ptr[i], e1 = p.row_ptr[i + 1];
    const float adst = p.rows[(long long)i * kRowB + 33];
    // forward, same arithmetic as csr_aggregate_kernel
    float m = -INFINITY;
    for (int e = e0; e < e1; ++e) m = fmaxf(m, gat_logit(p.rows[(long long)p.src[e] * kRowB + 32], adst));
    float den = 0.0f;
    for (int e = e0; e < e1; ++e)
      den = __fadd_rn(den, expf(__fsub_rn(gat_logit(p.rows[(long long)p.src[e] * kRowB + 32], adst), m)));
    den = __fadd_rn(den, 1e-16f);
    float agg[32], r[32], q[9];
#pragma unroll
    for (int cc = 0; cc < 32; ++cc) agg[cc] = 0.0f;
    for (int e = e0; e < e1; ++e) {
      const long long j = p.src[e];
      const float alpha = __fdiv_rn(expf(__fsub_rn(gat_logit(p.rows[j * kRowB + 32], adst), m)), den);
      p.alpha[e] = alpha;
      gat_accumulate(agg, alpha, reinterpret_cast<const float4*>(p.rows + j * kRowB));
    }
    float dvec[32];
    if (p.conv_only) {
      // stand-alone GATConv: the upstream gradient IS d(conv output)
      const float4* gin = reinterpret_cast<const float4*>(p.grad_q + (long long)i * 32);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 v = gin[c4];
        dvec[4 * c4] = v.x; dvec[4 * c4 + 1] = v.y; dvec[4 * c4 + 2] = v.z; dvec[4 * c4 + 3] = v.w;
      }
      store_row32(tDO, tid, dvec);
    } else {
    dqn_head(agg, tU + tid * kHPad, tR + tid * kHPad, sw, r, q);
    // head backward: dq given
    float dq[kW2Pad];
#pragma unroll
    for (int a = 0; a < kW2Pad; ++a) dq[a] = a < 9 ? p.grad_q[(long long)i * 9 + a] : 0.0f;
#pragma unroll
    for (int a = 0; a < kW2Pad; ++a) tDQ[tid * kW2Pad + a] = dq[a];
    {
      // dr[k] = sum_a W2[a][k] dq[a]; dp = dr * [r > 0], four k per iteration through the own row
      const float4* w2 = reinterpret_cast<const float4*>(sw + TW_W2T);
      const float4* r4 = reinterpret_cast<const float4*>(tR + tid * kHPad);
      float4* dp4 = reinterpret_cast<float4*>(tDP + tid * kHPad);
#pragma unroll 1
      for (int k4 = 0; k4 < 8; ++k4) {
        const float4 rk = r4[k4];
        float o[4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          float acc = 0.0f;
#pragma unroll
          for (int a4 = 0; a4 < 3; ++a4) {
            const float4 w = w2[(k4 * 4 + kk) * 3 + a4];
            acc = fmaf(w.x, dq[4 * a4 + 0], acc);
            acc = fmaf(w.y, dq[4 * a4 + 1], acc);
            acc = fmaf(w.z, dq[4 * a4 + 2], acc);
            acc = fmaf(w.w, dq[4 * a4 + 3], acc);
          }
          o[kk] = f4c(rk, kk) > 0.0f ? acc : 0.0f;
        }
        dp4[k4] = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
    load_row32(tDP, tid, dvec);
    {
      // du[k] = sum_c W1[c][k] dp[c] ; do = du * (1 - u^2)
      const float4* w1 = reinterpret_cast<const float4*>(sw + TW_W1T);
      const float4* u4 = reinterpret_cast<const float4*>(tU + tid * kHPad);
      float4* do4 = reinterpret_cast<float4*>(tDO + tid * kHPad);
#pragma unroll 1
      for (int k4 = 0; k4 < 8; ++k4) {
        const float4 uk = u4[k4];
        float o[4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          float acc = 0.0f;
#pragma unroll
          for (int c4 = 0; c4 < 8; ++c4) {
            const float4 w = w1[(k4 * 4 + kk) * 8 + c4];
            acc = fmaf(w.x, dvec[4 * c4 + 0], acc);
            acc = fmaf(w.y, dvec[4 * c4 + 1], acc);
            acc = fmaf(w.z, dvec[4 * c4 + 2], acc);
            acc = fmaf(w.w, dvec[4 * c4 + 3], acc);
          }
          const float uu = f4c(uk, kk);
          o[kk] = acc * (1.0f - uu * uu);
        }
        do4[k4] = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
    load_row32(tDO, tid, dvec);                       // dvec = d(conv output_i)
    }
    {
      float4* g = reinterpret_cast<float4*>(p.d_out + (long long)i * 32);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) g[c4] = make_float4(dvec[4 * c4], dvec[4 * c4 + 1], dvec[4 * c4 + 2], dvec[4 * c4 + 3]);
    }
    // attention backward over the in-edge group
    float dot_sum = 0.0f;
    for (int e = e0; e < e1; ++e) {
      const float4* hj = reinterpret_cast<const float4*>(p.rows + (long long)p.src[e] * kRowB);
      float da = 0.0f;
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 hv = hj[c4];
        da = fmaf(dvec[4 * c4 + 0], hv.x, da);
        da = fmaf(dvec[4 * c4 + 1], hv.y, da);
        da = fmaf(dvec[4 * c4 + 2], hv.z, da);
        da = fmaf(dvec[4 * c4 + 3], hv.w, da);
      }
      p.draw[e] = da;
      dot_sum = fmaf(p.alpha[e], da, dot_sum);
    }
    float dd_i = 0.0f;
    for (int e = e0; e < e1; ++e) {
      const float dz = p.alpha[e] * (p.draw[e] - dot_sum);
      const float raw = __fadd_rn(p.rows[(long long)p.src[e] * kRowB + 32], adst);
      const float dzz = raw > 0.0f ? dz : 0.2f * dz;
      p.draw[e] = dzz;
      dd_i += dzz;
    }
    p.dd[i] = dd_i;
  }
  __syncthreads();
  float* out = p.partials + (long long)blockIdx.x * kPartialStride;
  constexpr int G_B0 = 8, G_W1 = 256, G_B1 = 8, G_W2 = 72, G_B2 = 3;
  constexpr int G_TOTAL = G_B0 + G_W1 + G_B1 + G_W2 + G_B2;
  const int n_groups = p.conv_only ? G_B0 : G_TOTAL;      // conv-only: the partial row was zeroed by the launcher
#pragma unroll 1
  for (int grp = tid; grp < n_groups; grp += T) {
    int gi = grp;
    const float* A = nullptr;
    const float* Bm;
    int lda = 0, ac = 0, ldb = kHPad, bc, oidx, nout = 4;
    if (gi < G_B0) {                                   // d conv1.bias[c] = sum_n DO[n][c]
      Bm = tDO; bc = gi * 4; oidx = SWARM_W_CONV_BIAS + gi * 4;
    } else if ((gi -= G_B0) < G_W1) {                  // dW1[c][k] = sum_n DP[n][c] U[n][k]
      A = tDP; lda = kHPad; ac = gi >> 3; Bm = tU; bc = (gi & 7) * 4; oidx = SWARM_W_LIN1 + ac * 32 + bc;
    } else if ((gi -= G_W1) < G_B1) {                  // d lin1.bias[c] = sum_n DP[n][c]
      Bm = tDP; bc = gi * 4; oidx = SWARM_W_LIN1_BIAS + gi * 4;
    } else if ((gi -= G_B1) < G_W2) {                  // dW2[a][k] = sum_n DQ[n][a] R[n][k]
      A = tDQ; lda = kW2Pad; ac = gi >> 3; Bm = tR; bc = (gi & 7) * 4; oidx = SWARM_W_LIN2 + ac * 32 + bc;
    } else {                                           // d lin2.bias[a] = sum_n DQ[n][a]
      gi -= G_W2;
      Bm = tDQ; ldb = kW2Pad; bc = gi * 4; oidx = SWARM_W_LIN2_BIAS + gi * 4;
      nout = gi < 2 ? 4 : 1;
    }
    const float4 a = tile_gemm4(A, lda, ac, Bm, ldb, bc, T);
    float* o = out + oidx;
    o[0] = a.x;
    if (nout == 4) { o[1] = a.y; o[2] = a.z; o[3] = a.w; }
  }
  if (tid == 0) out[SWARM_W_COUNT] = 0.0f;
}

__global__ void __launch_bounds__(kTileThreads) csr_bwd_source_kernel(const __grid_constant__ CsrBwdParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int T = kTileThreads;
  float* tDH = reinterpret_cast<float*>(smem);
  float* tH = tDH + T * kHPad;
  float* tX = tH + T * kHPad;
  float* sds = tX + T * kXPad;
  float* sdd = sds + T;
  const int tid = threadIdx.x;
  const int j = blockIdx.x * T + tid;
  float4* dh_row = reinterpret_cast<float4*>(tDH + tid * kHPad);
  float4* h_row = reinterpret_cast<float4*>(tH + tid * kHPad);
  float4* x_row = reinterpret_cast<float4*>(tX + tid * kXPad);
  float ds_j = 0.0f, dd_j = 0.0f;
  if (j < p.n) {
    float dh[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) dh[k] = 0.0f;
    const int q0 = p.row_ptr_s[j], q1 = p.row_ptr_s[j + 1];
    for (int q = q0; q < q1; ++q) {
      const int pp = p.pos_s[q];
      const float a = p.alpha[pp];
      ds_j += p.draw[pp];
      const float4* dr = reinterpret_cast<const float4*>(p.d_out + (long long)p.tgt_s[q] * 32);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 dv = dr[c4];
        dh[4 * c4 + 0] = fmaf(a, dv.x, dh[4 * c4 + 0]);
        dh[4 * c4 + 1] = fmaf(a, dv.y, dh[4 * c4 + 1]);
        dh[4 * c4 + 2] = fmaf(a, dv.z, dh[4 * c4 + 2]);
        dh[4 * c4 + 3] = fmaf(a, dv.w, dh[4 * c4 + 3]);
      }
    }
    dd_j = p.dd[j];
    const float* as = p.weights + SWARM_W_ATT_SRC;
    const float* ad = p.weights + SWARM_W_ATT_DST;
#pragma unroll
    for (int k = 0; k < 32; ++k) dh[k] = fmaf(ds_j, as[k], fmaf(dd_j, ad[k], dh[k]));
    store_row32(tDH, tid, dh);
    const float4* hr = reinterpret_cast<const float4*>(p.rows + (long long)j * kRowB);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) h_row[c4] = hr[c4];
    const float* xr = p.x + (long long)j * 7;
    x_row[0] = make_float4(xr[0], xr[1], xr[2], xr[3]);
    x_row[1] = make_float4(xr[4], xr[5], xr[6], 0.0f);
  } else {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) { dh_row[c4] = z; h_row[c4] = z; }
    x_row[0] = z;
    x_row[1] = z;
  }
  sds[tid] = ds_j;
  sdd[tid] = dd_j;
  __syncthreads();
  float* out = p.partials + (long long)blockIdx.x * kPartialStride;
  constexpr int G_W0 = 64, G_AS = 8, G_AD = 8;
#pragma unroll 1
  for (int grp = tid; grp < G_W0 + G_AS + G_AD; grp += T) {
    if (grp < G_W0) {                                  // dW0[c][k] = sum_n DH[n][c] X[n][k]
      const int cc = grp >> 1, k4 = (grp & 1) * 4;
      const float4 a = tile_gemm4(tDH, kHPad, cc, tX, kXPad, k4, T);
      float* o = out + SWARM_W_CONV_LIN + cc * 7 + k4;
      o[0] = a.x; o[1] = a.y; o[2] = a.z;
      if (k4 == 0) o[3] = a.w;
    } else {
      const bool is_src = grp < G_W0 + G_AS;           // d att_src[c] = sum_n ds[n] H[n][c]; d att_dst with dd
      const int gi = is_src ? grp - G_W0 : grp - G_W0 - G_AS;
      const float4 a = tile_gemm4(is_src ? sds : sdd, 1, 0, tH, kHPad, gi * 4, T);
      float* o = out + (is_src ? SWARM_W_ATT_SRC : SWARM_W_ATT_DST) + gi * 4;
      o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w;
    }
  }
}

static size_t bwd_align(size_t v) { return (v + 255) & ~(size_t)255; }

long long gatq_backward_workspace_bytes(int n, long long E) {
  const long long ctas = (n + kTileThreads - 1) / kTileThreads;
  return (long long)(bwd_align((size_t)n * kRowB * 4) + bwd_align((size_t)n * 32 * 4) + bwd_align((size_t)n * 4) +
                     2 * bwd_align((size_t)E * 4) + 2 * bwd_align((size_t)E * 4) +
                     bwd_align((size_t)ctas * kPartialStride * 4) + 512);
}

cudaError_t launch_gatq_backward_csr(int n, long long E, const float* weights, const float* x, const int32_t* row_ptr,
                                     const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                                     const int32_t* tgt_s, const int32_t* perm_s, const float* grad_q, float* grad_w,
                                     void* workspace, cudaStream_t stream, bool conv_only) {
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  auto take = [&](size_t bytes) { char* q = base; base += bwd_align(bytes); return q; };
  float* rows = reinterpret_cast<float*>(take((size_t)n * kRowB * 4));
  float* d_out = reinterpret_cast<float*>(take((size_t)n * 32 * 4));
  float* dd = reinterpret_cast<float*>(take((size_t)n * 4));
  float* alpha = reinterpret_cast<float*>(take((size_t)E * 4));
  float* draw = reinterpret_cast<float*>(take((size_t)E * 4));
  int32_t* inv = reinterpret_cast<int32_t*>(take((size_t)E * 4));
  int32_t* pos_s = reinterpret_cast<int32_t*>(take((size_t)E * 4));
  const int ctas = (n + kTileThreads - 1) / kTileThreads;
  float* partials = reinterpret_cast<float*>(take((size_t)ctas * kPartialStride * 4));
  float* loss_dummy = reinterpret_cast<float*>(take(256));

  cudaError_t err = launch_csr_project(n, weights, x, rows, stream);
  if (err != cudaSuccess) return err;
  if (E > 0) {
    long long blocks = (E + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    csr_edge_positions_kernel<<<(int)blocks, 256, 0, stream>>>(E, perm, perm_s, inv, pos_s, 0);
    csr_edge_positions_kernel<<<(int)blocks, 256, 0, stream>>>(E, perm, perm_s, inv, pos_s, 1);
  }
  if (conv_only) {
    err = cudaMemsetAsync(partials, 0, (size_t)ctas * kPartialStride * 4, stream);
    if (err != cudaSuccess) return err;
  }
  CsrBwdParams p;
  p.conv_only = conv_only ? 1 : 0;
  p.n = n;
  p.weights = weights;
  p.x = x;
  p.row_ptr = row_ptr;
  p.src = src;
  p.row_ptr_s = row_ptr_s;
  p.tgt_s = tgt_s;
  p.pos_s = pos_s;
  p.grad_q = grad_q;
  p.rows = rows;
  p.d_out = d_out;
  p.dd = dd;
  p.alpha = alpha;
  p.draw = draw;
  p.partials = partials;
  const int smem_t = (((TW_COUNT + 3) & ~3) + 4 * kTileThreads * kHPad + kTileThreads * kW2Pad) * 4;
  err = cudaFuncSetAttribute(csr_bwd_target_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_t);
  if (err != cudaSuccess) return err;
  csr_bwd_target_kernel<<<ctas, kTileThreads, smem_t, stream>>>(p);
  const int smem_s = (2 * kTileThreads * kHPad + kTileThreads * kXPad + 2 * kTileThreads) * 4;
  csr_bwd_source_kernel<<<ctas, kTileThreads, smem_s, stream>>>(p);
  dqn_reduce_kernel<<<(SWARM_W_COUNT + 1 + 255) / 256, 256, 0, stream>>>(partials, ctas, 1.0f, grad_w, loss_dummy, nullptr, 0,
                                                                         1, 0);
  return cudaGetLastError();
}

// ---- launchers -------------------------------------------------------------------------------
int dqn_maxdeg(const SwarmConfig& c) {
  return c.graph_mode == SWARM_GRAPH_KNN ? (c.n_agents + c.knn_k + 1) : c.n_agents;
}

// graphs per CTA: as many as fit (floor(128/N)) for big batches, fewer for small ones so that the update spreads over
// the SMs (G = 32 -> one graph per CTA) and the node contractions only walk the rows that exist
int dqn_epb(const SwarmConfig& c, int n_graphs) {
  const int full = kTileThreads / c.n_agents;
  int epb = (n_graphs + 147) / 148;
  if (epb < 1) epb = 1;
  return epb < full ? epb : full;
}

long long dqn_workspace_bytes(const SwarmConfig& c, int n_graphs) {
  const int epb = dqn_epb(c, n_graphs);
  const long long ctas = (n_graphs + epb - 1) / epb;
  return ctas * kPartialStride * 4 + 256;
}

cudaError_t launch_dqn_grad(const SwarmConfig& c, const float* w_online, const float* w_target, const SwarmReplay& batch,
                            const int64_t* indices, int n_graphs, float gamma, float loss_scale, float* grad, float* loss,
                            float* td, void* workspace, cudaStream_t stream, SwarmTrainCtl* ctl, int64_t* indices_out,
                            unsigned long long sample_seed, int pushed_envs, bool skip_reduce) {
  DqnParams p;
  p.ctl = ctl;
  p.indices_out = indices_out;
  p.sample_seed = sample_seed;
  p.pushed_envs = pushed_envs;
  p.cfg = c;
  p.w_online = w_online;
  p.w_target = w_target;
  p.batch = batch;
  p.indices = indices;
  p.n_graphs = n_graphs;
  p.gamma = gamma;
  p.loss_scale = loss_scale;
  p.partials = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  p.td = td;
  p.qmax_r = sq_threshold(c.graph_radius);
  p.epb = dqn_epb(c, n_graphs);
  p.maxdeg = dqn_maxdeg(c);
  const int ctas = (n_graphs + p.epb - 1) / p.epb;
  cudaError_t err = launch_dqn_grad_tc(p, stream);
  if (err != cudaSuccess) return err;
  // skip_reduce: the caller sums the partials inside launch_reduce_clip_adam
  if (!skip_reduce)
    dqn_reduce_kernel<<<(SWARM_W_COUNT + 1 + 255) / 256, 256, 0, stream>>>(p.partials, ctas, loss_scale, grad, loss, ctl,
                                                                           pushed_envs, batch.capacity, n_graphs);
  return cudaGetLastError();
}

// The cluster launch sums an element's partials on one thread, 32 loads in flight: a win over the reduce launch while
// the gradient kernel ran on few CTAs (the reference's 32 graphs: 33.2 vs 34.8 us per tick); for the 410 CTAs of a
// 4 096-graph update seven SMs pull 2.7 MB and the tick is slower (69 vs 63.6 us), so those keep the separate launches.
bool dqn_fuse_reduce(const SwarmConfig& c, int n_graphs) {
  const int epb = dqn_epb(c, n_graphs);
  return (n_graphs + epb - 1) / epb <= 64;
}

cudaError_t launch_adam_clip(float* w, const float* grad, float* m, float* v, long long step, double lr, double beta1,
                             double beta2, double eps, double max_norm, float* target, float* grad_norm,
                             cudaStream_t stream, SwarmTrainCtl* ctl, int num_envs, long long ring_capacity,
                             int update_target_every, const SwarmPeerExchange* peers, float* grad_rw,
                             const SwarmConfig* reduce_cfg, const void* reduce_workspace, int reduce_graphs,
                             float loss_scale) {
  AdamParams p;
  p.partials = nullptr;
  p.n_ctas = 0;
  p.n_graphs = reduce_graphs;
  p.loss_scale = loss_scale;
  if (reduce_workspace && reduce_cfg && ctl && dqn_fuse_reduce(*reduce_cfg, reduce_graphs)) {
    // the partials of launch_dqn_grad(..., skip_reduce = true) on the same workspace
    const int epb = dqn_epb(*reduce_cfg, reduce_graphs);
    p.n_ctas = (reduce_graphs + epb - 1) / epb;
    p.partials = reinterpret_cast<const float*>((reinterpret_cast<uintptr_t>(reduce_workspace) + 255) & ~(uintptr_t)255);
  }
  if (peers && ctl) p.peers = *peers;
  else p.peers.world_size = 0;
  p.grad_rw = grad_rw;
  p.ctl = ctl;
  p.lr = lr;
  p.beta1 = beta1;
  p.beta2d = beta2;
  p.num_envs = num_envs;
  p.ring_capacity = ring_capacity;
  p.update_target_every = update_target_every > 0 ? update_target_every : 1;
  p.w = w;
  p.grad = grad;
  p.m = m;
  p.v = v;
  p.target = target;
  p.grad_norm = grad_norm;
  // scalars exactly as torch.optim.Adam computes them (Python doubles, cast to float where they meet tensors)
  const double b1 = beta1, b2 = beta2;
  const double bc1 = 1.0 - pow(b1, (double)step);
  const double bc2 = 1.0 - pow(b2, (double)step);
  p.lerp_w = (float)(1.0 - b1);
  p.beta2 = (float)beta2;
  p.one_minus_beta2 = (float)(1.0 - b2);
  p.neg_step_size = (float)(-(lr / bc1));
  p.bc2_sqrt = (float)sqrt(bc2);
  p.eps = (float)eps;
  p.max_norm = (float)max_norm;
  if (p.partials && p.peers.world_size > 1) reduce_clip_adam_kernel<true><<<kAdamCluster, 256, 0, stream>>>(p);
  else if (p.partials) reduce_clip_adam_kernel<false><<<kAdamCluster, 256, 0, stream>>>(p);
  else if (p.peers.world_size > 1) adam_clip_kernel<true><<<1, 256, 0, stream>>>(p);
  else adam_clip_kernel<false><<<1, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace swarm
