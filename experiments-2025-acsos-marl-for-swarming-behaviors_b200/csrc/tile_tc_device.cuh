// tile_tc_device.cuh -- the tensor-core (tcgen05, 3xTF32) variant of the per-tick Q-network forward of the
// env-tile kernels.  The three dense contractions run as UMMA tiles over the CTA's 128 node rows; attention
// softmax / aggregation, biases, tanh / ReLU and the argmax stay on the CUDA cores.
//
// Attention in INPUT space.  GATConv's projection is linear and has no bias (train:50-58: h_j = W0 x_j), so
//     sum_e alpha_e h_src(e) = W0 (sum_e alpha_e x_src(e))      and      <h_j, att> = <x_j, W0^T att>.
// The tick therefore never forms h: every node takes two 7-term dot products with the pre-multiplied attention
// vectors (v_s = W0^T att_src, v_d = W0^T att_dst, computed once per launch), the softmax-weighted mean is taken over
// the 7 input features of the neighbours -- of which four are the state already staged for the world step, two are
// the constant goal and one is the agent id -- and ONE projection MMA (K = 8) maps the mean to the 32 channels.  Per
// edge that is one 16-byte shared-memory load and three FMAs instead of eight loads and sixteen packed FMAs, the
// 18 KB tile of projected features, its publication and one block barrier per tick disappear.  Same mathematics as
// the reference's order of operations, different rounding (float32 level both ways); the bit-faithful order lives on
// in the SWARM_TC=0 path.
#ifndef SWARM_TILE_TC_DEVICE_CUH
#define SWARM_TILE_TC_DEVICE_CUH

#include "tc_device.cuh"
#include "tile_device.cuh"

namespace swarm {

// Phase clocks of the rollout tick, compiled in only with -DSWARM_PHASE_CLOCKS (scripts/time_rollout_phases.py builds
// such a library next to the regular one).  Lane 0 of every warp stamps clock64() at each phase boundary and adds the
// cycles since the previous stamp to its warp's slot in shared memory; at the end of the launch the per-warp sums go to
// g_phase_cycles[global warp][phase].  A phase's count includes the time its warp waits at the barriers inside it.
enum { PH_PUBLISH = 0, PH_ATTEND, PH_PROJ, PH_TANH, PH_LIN1, PH_RELU, PH_LIN2, PH_WORLD, PH_COUNT };
#ifdef SWARM_PHASE_CLOCKS
constexpr int kPhaseWarps = 16384;
__device__ unsigned long long g_phase_cycles[kPhaseWarps][PH_COUNT];   // (only tile_kernels.cu is built with the macro)
__device__ __forceinline__ unsigned long long* phase_slots() {
  __shared__ unsigned long long s[kTileThreads / 32][PH_COUNT + 1];     // [warp][phase]; [warp][PH_COUNT] = last stamp
  return s[threadIdx.x >> 5];
}
__device__ __forceinline__ void phase_reset() {
  if ((threadIdx.x & 31) == 0)
    for (int k = 0; k < PH_COUNT; ++k) phase_slots()[k] = 0;
}
__device__ __forceinline__ void phase_start() {
  if ((threadIdx.x & 31) == 0) phase_slots()[PH_COUNT] = clock64();
}
__device__ __forceinline__ void phase_mark(int k) {
  if ((threadIdx.x & 31) == 0) {
    unsigned long long* s = phase_slots();
    const unsigned long long now = clock64();
    s[k] += now - s[PH_COUNT];
    s[PH_COUNT] = now;
  }
}
__device__ __forceinline__ void phase_flush() {
  const long long w = (long long)blockIdx.x * (kTileThreads / 32) + (threadIdx.x >> 5);
  if ((threadIdx.x & 31) == 0 && w < kPhaseWarps)
    for (int k = 0; k < PH_COUNT; ++k) g_phase_cycles[w][k] = phase_slots()[k];
}
#define SWARM_PHASE_RESET() phase_reset()
#define SWARM_PHASE_START() phase_start()
#define SWARM_PHASE(k) phase_mark(k)
#define SWARM_PHASE_FLUSH() phase_flush()
#else
#define SWARM_PHASE_RESET() ((void)0)
#define SWARM_PHASE_START() ((void)0)
#define SWARM_PHASE(k) ((void)0)
#define SWARM_PHASE_FLUSH() ((void)0)
#endif

// float offsets inside the small vector block
// (v_s, v_d: W0^T att_src / W0^T att_dst, 7 entries + one zero each)
enum { TV_VS = 0, TV_VD = 8, TV_B0 = 16, TV_B1 = 48, TV_B2 = 80, TV_COUNT = 96 };
// TMEM columns: D tiles [0,32) projection / lin2 and [32,64) lin1; A operand (this CTA's 128 activation rows, written
// by their owner threads with tcgen05.st) hi half [64,96), lo half [96,128)
constexpr int kTmemCols = 128;
constexpr uint32_t kTmemAHi = 64, kTmemALo = 96;

struct TileTcSmem {
  unsigned char* w0;     // [32 x 8]  hi +0 (1 KB), lo +1 KB
  unsigned char* w1;     // [32 x 32] hi +0 (4 KB), lo +4 KB
  unsigned char* w2;     // [16 x 32] hi +0 (2 KB), lo +2 KB
  float* vec;            // TV_*
  uint64_t* bar;
  uint32_t* tmem_slot;
};

constexpr int kTcW0Bytes = 2 * 32 * 8 * 4, kTcW1Bytes = 2 * 32 * 32 * 4, kTcW2Bytes = 2 * 16 * 32 * 4;

// global packed weights -> split (hi, lo) UMMA B tiles + bias / attention vectors.
// All global loads of a thread are issued before the first shared-memory store (the destinations are char pointers,
// which the compiler must assume to alias the source): one exposed memory round trip instead of one per item --
// this prologue is a fifth of a single-tick launch (train tick).
// Split into a load phase (global -> registers) and a store phase (registers -> shared), so a kernel that stages
// several weight sets issues all their loads before the first store.  `vtid` = index of the thread inside the group
// that fills the vector block (tid itself, or tid - 32 * w to put the dot-product chains of v_s / v_d on warp w).
struct TcStageRegs {
  float vv;
  float4 item[(448 + kTileThreads - 1) / kTileThreads];
};

__device__ __forceinline__ void stage_weights_tc_load(const float* __restrict__ gw, TcStageRegs& r, int tid, int nthreads,
                                                      int vtid) {
  // bias vectors, and the attention vectors pulled through the projection: v[k] = sum_c att[c] W0[c][k], c ascending
  // (threads 0 .. 13 of the group; every load is issued before the FMA chain starts)
  float vv = 0.0f;
  {
    const int idx = vtid;
    if (idx >= 0 && idx < TV_B0) {
      const int k = idx & 7;
      if (k < 7) {
        const float* att = gw + ((idx < TV_VD) ? SWARM_W_ATT_SRC : SWARM_W_ATT_DST);
        float a[32], w[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) { a[c] = att[c]; w[c] = gw[SWARM_W_CONV_LIN + c * 7 + k]; }
#pragma unroll
        for (int c = 0; c < 32; ++c) vv = fmaf(a[c], w[c], vv);
      }
    } else if (idx >= TV_B0 && idx < TV_B1) vv = gw[SWARM_W_CONV_BIAS + (idx - TV_B0)];
    else if (idx >= TV_B1 && idx < TV_B2) vv = gw[SWARM_W_LIN1_BIAS + (idx - TV_B1)];
    else if (idx >= TV_B2 && idx - TV_B2 < 9) vv = gw[SWARM_W_LIN2_BIAS + (idx - TV_B2)];
  }
  r.vv = vv;
  constexpr int kItemIters = (448 + kTileThreads - 1) / kTileThreads;         // 4
  // items: (row n, k-chunk c) of W1 (256), W2 (128), W0 (64)
#pragma unroll
  for (int k = 0; k < kItemIters; ++k) {
    const int it = tid + k * nthreads;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (it < 256) {
      const float* q = gw + SWARM_W_LIN1 + (it >> 3) * 32 + 4 * (it & 7);
      v = make_float4(q[0], q[1], q[2], q[3]);
    } else if (it < 384) {
      const int j = it - 256;
      if ((j >> 3) < 9) {
        const float* q = gw + SWARM_W_LIN2 + (j >> 3) * 32 + 4 * (j & 7);
        v = make_float4(q[0], q[1], q[2], q[3]);
      }
    } else if (it < 448) {
      const int j = it - 384;
      const float* q = gw + SWARM_W_CONV_LIN + (j >> 1) * 7 + 4 * (j & 1);
      v = (j & 1) == 0 ? make_float4(q[0], q[1], q[2], q[3]) : make_float4(q[0], q[1], q[2], 0.0f);
    }
    r.item[k] = v;
  }
}

__device__ __forceinline__ void stage_weights_tc_store(const TcStageRegs& r, const TileTcSmem& s, int tid, int nthreads,
                                                       int vtid) {
  constexpr int kItemIters = (448 + kTileThreads - 1) / kTileThreads;
  if (vtid >= 0 && vtid < TV_COUNT) s.vec[vtid] = r.vv;
#pragma unroll
  for (int k = 0; k < kItemIters; ++k) {
    const int it = tid + k * nthreads;
    if (it >= 448) break;
    unsigned char* base;
    int rows, n, c, half;
    if (it < 256) {
      n = it >> 3; c = it & 7; rows = 32; base = s.w1; half = kTcW1Bytes / 2;
    } else if (it < 384) {
      const int j = it - 256;
      n = j >> 3; c = j & 7; rows = 16; base = s.w2; half = kTcW2Bytes / 2;
    } else {
      const int j = it - 384;
      n = j >> 1; c = j & 1; rows = 32; base = s.w0; half = kTcW0Bytes / 2;
    }
    float4 hi, lo;
    tc::split4(r.item[k], hi, lo);
    const int off = tc::tile_off(rows, n, c);
    *reinterpret_cast<float4*>(base + off) = hi;
    *reinterpret_cast<float4*>(base + half + off) = lo;
  }
}

__device__ __forceinline__ void stage_weights_tc(const float* __restrict__ gw, const TileTcSmem& s, int tid, int nthreads) {
  TcStageRegs r;
  stage_weights_tc_load(gw, r, tid, nthreads, tid);
  stage_weights_tc_store(r, s, tid, nthreads, tid);
}

// The A operand of the three contractions lives in TENSOR MEMORY: every thread splits its own activation row into
// (hi, lo) and writes it to its TMEM lane with two tcgen05.st -- no shared-memory stores, no shared-memory operand
// reads by the MMA (shared-memory bandwidth is the busiest resource of the rollout tick: l1tex 61 %).
__device__ __forceinline__ void tc_store_a_row(uint32_t lane_addr, const float (&v)[32]) {
  uint32_t hi[32], lo[32];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    float4 h4, l4;
    tc::split4(make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]), h4, l4);
    hi[4 * c + 0] = __float_as_uint(h4.x); hi[4 * c + 1] = __float_as_uint(h4.y);
    hi[4 * c + 2] = __float_as_uint(h4.z); hi[4 * c + 3] = __float_as_uint(h4.w);
    lo[4 * c + 0] = __float_as_uint(l4.x); lo[4 * c + 1] = __float_as_uint(l4.y);
    lo[4 * c + 2] = __float_as_uint(l4.z); lo[4 * c + 3] = __float_as_uint(l4.w);
  }
  tc::tmem_st32(lane_addr + kTmemAHi, hi);
  tc::tmem_st32(lane_addr + kTmemALo, lo);
  tc::tmem_wait_st();
}

// One UMMA round: every thread has written its operand row to TMEM; barrier; one elected thread issues the 3xTF32
// MMAs and commits to the mbarrier; everybody waits for completion.  `parity` is the per-thread phase bit.
__device__ __forceinline__ void tc_mma_round(const TileTcSmem& s, uint32_t tmem, uint32_t tmem_d, const unsigned char* b_tile,
                                             int b_half, int b_rows, int ksteps, uint32_t& parity) {
  tc::fence_before_sync();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) {
    tc::fence_after_sync();
    if (tc::elect_one()) {
      const uint32_t b = tc::smem_u32(b_tile);
      tc::mma_3xtf32_tmem_a(tmem_d, tmem + kTmemAHi, tmem + kTmemALo, b, b + b_half, b_rows, ksteps,
                            tc::make_idesc_tf32(b_rows));
      tc::mma_commit(s.bar);
    }
    __syncwarp();
  }
  tc::mbar_wait(s.bar, parity);
  parity ^= 1u;
  tc::fence_after_sync();
}

// alpha_src / alpha_dst of the node with input features x (attention vectors pulled through the projection)
__device__ __forceinline__ void tc_alpha_terms(const TileTcSmem& s, const float (&x)[7], float& asrc, float& adst) {
  const float4* v4 = reinterpret_cast<const float4*>(s.vec + TV_VS);
  const float4 s0 = v4[0], s1 = v4[1], d0 = v4[2], d1 = v4[3];
  float2 acc = make_float2(0.0f, 0.0f);
  acc = __ffma2_rn(make_float2(x[0], x[0]), make_float2(s0.x, d0.x), acc);
  acc = __ffma2_rn(make_float2(x[1], x[1]), make_float2(s0.y, d0.y), acc);
  acc = __ffma2_rn(make_float2(x[2], x[2]), make_float2(s0.z, d0.z), acc);
  acc = __ffma2_rn(make_float2(x[3], x[3]), make_float2(s0.w, d0.w), acc);
  acc = __ffma2_rn(make_float2(x[4], x[4]), make_float2(s1.x, d1.x), acc);
  acc = __ffma2_rn(make_float2(x[5], x[5]), make_float2(s1.y, d1.y), acc);
  acc = __ffma2_rn(make_float2(x[6], x[6]), make_float2(s1.z, d1.z), acc);
  asrc = acc.x;
  adst = acc.y;
}

// Softmax-weighted mean of the neighbours' input features (see the header).  `pos` = the tile's states, g.sas = the
// published alpha_src terms.  Three ways to name the in-edges of node i:
//   ATT_LIST      the in-edge list g.sin / deg in edge-list order (radius graph, large kNN swarms)
//   ATT_COMPLETE  the reference's complete graph (train:101-108): every j != i, node 0 additionally its (0,0) self loop
//   ATT_COUNTS    `counts` = 2 bits per source j: how many parallel edges j -> i the symmetrised kNN list of
//                 simulator.py:20-24 holds (0 .. 3); the sums run over j = 0 .. N - 1 with the term weighted by its
//                 multiplicity -- the same sum as over the list, term order and one rounding apart -- so the per-tick
//                 in-edge LIST (strided byte stores, two barriers) is never built
enum { ATT_LIST = 0, ATT_COMPLETE = 1, ATT_COUNTS = 2 };

//
// NT > 0 (ATT_COMPLETE only): the swarm size at compile time.  Every loop unrolls completely: the alpha_src row is read
// as float4s (an env's row starts at a multiple of 16 bytes when NT % 4 == 0), its maximum is a tree, and all NT
// exponentials are issued before the accumulation, so the dependent chains are the sums alone.  An inactive thread
// computes on env 0 of its tile instead of skipping the loops and discards the result (its UMMA row is independent of
// the others).  The sums keep the order of the run-time loop: den, acc_p, acc_v and acc_id run left to right in j, so
// the result is the same to the bit.  The maximum is exact in any order; a tree can return -0 where the chain returns
// +0 (or the reverse), but m only enters through exp(x - m), and x - (+0) and x - (-0) differ at most in the sign of a
// zero, which exp maps to 1 either way.
template <int ATT, int NT = 0>
__device__ __forceinline__ void tile_attend_inputs(const TileGraphSmem& g, const TileThread& t, const float4* __restrict__ pos,
                                                   int N, int deg, uint32_t counts, float adst, float goal_x, float goal_y,
                                                   float (&xm)[8]) {
  constexpr bool COMPLETE = (ATT == ATT_COMPLETE);
  const int T = kTileThreads;
  const float* __restrict__ sas = g.sas + t.envbase;
  const float4* __restrict__ env = pos + t.envbase;
  float den = 0.0f, acc_id = 0.0f;
  float2 acc_p = make_float2(0.0f, 0.0f), acc_v = make_float2(0.0f, 0.0f);
  // LeakyReLU and the rounded add are monotone: max_e leaky(a_e + d) = leaky(max_e a_e + d)
  if constexpr (COMPLETE && NT > 0) {
    const int base = t.active ? t.envbase : 0;
    const int self = (t.i == 0) ? -1 : t.i;
    float a[NT];
    if constexpr (NT % 4 == 0) {
      const float4* __restrict__ sas4 = reinterpret_cast<const float4*>(g.sas + base);
#pragma unroll
      for (int k = 0; k < NT / 4; ++k) {
        const float4 v = sas4[k];
        a[4 * k] = v.x; a[4 * k + 1] = v.y; a[4 * k + 2] = v.z; a[4 * k + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NT; ++j) a[j] = g.sas[base + j];
    }
    float4 sj[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) sj[j] = pos[base + j];
    // (where every term is NaN the tree returns NaN and the chain -inf: every weight is NaN either way)
    float mx[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) mx[j] = (j == self) ? -INFINITY : a[j];
#pragma unroll
    for (int w = 1; w < NT; w *= 2) {
#pragma unroll
      for (int j = 0; j + w < NT; j += 2 * w) mx[j] = fmaxf(mx[j], mx[j + w]);
    }
    const float amax = mx[0];
    const float zt = __fadd_rn(amax, adst);
    const float m = fmaxf(zt, __fmul_rn(zt, 0.2f));
    float wj[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const float zz = __fadd_rn(a[j], adst);
      const float ex = __expf(fmaxf(zz, __fmul_rn(zz, 0.2f)) - m);
      wj[j] = (j == self) ? 0.0f : ex;
    }
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const float w = wj[j];
      const float2 w2 = make_float2(w, w);
      den = __fadd_rn(den, w);
      acc_p = __ffma2_rn(w2, make_float2(sj[j].x, sj[j].y), acc_p);
      acc_v = __ffma2_rn(w2, make_float2(sj[j].z, sj[j].w), acc_v);
      acc_id = fmaf(w, (float)j, acc_id);
    }
  } else if (ATT == ATT_COUNTS) {
    const int n = t.active ? N : 0;
    float amax = -INFINITY;
    uint32_t cw = counts;
#pragma unroll 4
    for (int j = 0; j < n; ++j, cw >>= 2) amax = fmaxf(amax, (cw & 3u) ? sas[j] : -INFINITY);
    const float zt = __fadd_rn(amax, adst);
    const float m = fmaxf(zt, __fmul_rn(zt, 0.2f));
    float fj = 0.0f;
    cw = counts;
#pragma unroll 4
    for (int j = 0; j < n; ++j, cw >>= 2) {
      const float4 sj = env[j];
      const float zz = __fadd_rn(sas[j], adst);
      const float ex = __expf(fmaxf(zz, __fmul_rn(zz, 0.2f)) - m);
      const float w = ex * (float)(cw & 3u);
      const float2 w2 = make_float2(w, w);
      den = __fadd_rn(den, w);
      acc_p = __ffma2_rn(w2, make_float2(sj.x, sj.y), acc_p);
      acc_v = __ffma2_rn(w2, make_float2(sj.z, sj.w), acc_v);
      acc_id = fmaf(w, fj, acc_id);
      fj += 1.0f;
    }
  } else if (COMPLETE) {
    // Sources of node i: every j != i, and j = 0 for node 0 itself (its self loop).  The sums run over j = 0 .. N - 1
    // with the own slot weighted zero -- for node 0 the self loop is summed first instead of last, a different
    // rounding of the same sum (summing it last through a tail branch that every warp executes cost 4 % of the
    // rollout) -- so the loop needs no index arithmetic at all.
    const int self = (t.i == 0) ? -1 : t.i;
    const int n = t.active ? N : 0;
    float amax = -INFINITY;
#pragma unroll 4
    for (int j = 0; j < n; ++j) amax = fmaxf(amax, j == self ? -INFINITY : sas[j]);
    const float zt = __fadd_rn(amax, adst);
    const float m = fmaxf(zt, __fmul_rn(zt, 0.2f));
    float fj = 0.0f;
#pragma unroll 4
    for (int j = 0; j < n; ++j) {
      const float4 sj = env[j];
      const float zz = __fadd_rn(sas[j], adst);
      const float ex = __expf(fmaxf(zz, __fmul_rn(zz, 0.2f)) - m);
      const float w = (j == self) ? 0.0f : ex;
      const float2 w2 = make_float2(w, w);
      den = __fadd_rn(den, w);
      acc_p = __ffma2_rn(w2, make_float2(sj.x, sj.y), acc_p);
      acc_v = __ffma2_rn(w2, make_float2(sj.z, sj.w), acc_v);
      acc_id = fmaf(w, fj, acc_id);
      fj += 1.0f;
    }
  } else {
    const uint8_t* __restrict__ sin = g.sin + t.tid;
    float amax = -INFINITY;
#pragma unroll 4
    for (int e = 0; e < deg; ++e) amax = fmaxf(amax, sas[sin[e * T]]);
    const float zt = __fadd_rn(amax, adst);
    const float m = fmaxf(zt, __fmul_rn(zt, 0.2f));
#pragma unroll 2
    for (int e = 0; e < deg; ++e) {
      const int j = sin[e * T];
      const float4 sj = env[j];
      const float zz = __fadd_rn(sas[j], adst);
      const float w = __expf(fmaxf(zz, __fmul_rn(zz, 0.2f)) - m);
      const float2 w2 = make_float2(w, w);
      den = __fadd_rn(den, w);
      acc_p = __ffma2_rn(w2, make_float2(sj.x, sj.y), acc_p);
      acc_v = __ffma2_rn(w2, make_float2(sj.z, sj.w), acc_v);
      acc_id = fmaf(w, (float)j, acc_id);
    }
  }
  const float inv = 1.0f / __fadd_rn(den, 1e-16f);
  const float wsum = den * inv;                  // sum of the attention coefficients (the goal features are constant)
  xm[0] = acc_p.x * inv; xm[1] = acc_p.y * inv; xm[2] = acc_v.x * inv; xm[3] = acc_v.y * inv;
  xm[4] = goal_x * wsum; xm[5] = goal_y * wsum; xm[6] = acc_id * inv; xm[7] = 0.0f;
}

// Full per-tick Q forward on the tensor cores.  The caller has published g.sas[tid] = alpha_src of every node and
// passed a block barrier since (the tick's state barrier).  Contains 3 block barriers.  All 128 threads must call it.
template <int ATT, int NT = 0>
__device__ __forceinline__ int tile_q_forward_tc(const TileGraphSmem& g, const TileTcSmem& s, const TileThread& t,
                                                 uint32_t tmem, const float4* __restrict__ pos, int N, int deg,
                                                 uint32_t counts, float adst, float goal_x, float goal_y, uint32_t& parity,
                                                 float (&q)[9]) {
  const uint32_t lane_addr = tmem + ((uint32_t)(t.tid & ~31) << 16);     // this warp's 32 TMEM lanes
  // ---- attention in input space, then agg = mean W0^T (K padded 7 -> 8) ----
  {
    float xm[8];
    tile_attend_inputs<ATT, NT>(g, t, pos, N, deg, counts, adst, goal_x, goal_y, xm);
    SWARM_PHASE(PH_ATTEND);
    float4 h0, l0, h1, l1;
    tc::split4(make_float4(xm[0], xm[1], xm[2], xm[3]), h0, l0);
    tc::split4(make_float4(xm[4], xm[5], xm[6], 0.0f), h1, l1);
    const uint32_t hi[8] = {__float_as_uint(h0.x), __float_as_uint(h0.y), __float_as_uint(h0.z), __float_as_uint(h0.w),
                            __float_as_uint(h1.x), __float_as_uint(h1.y), __float_as_uint(h1.z), __float_as_uint(h1.w)};
    const uint32_t lo[8] = {__float_as_uint(l0.x), __float_as_uint(l0.y), __float_as_uint(l0.z), __float_as_uint(l0.w),
                            __float_as_uint(l1.x), __float_as_uint(l1.y), __float_as_uint(l1.z), __float_as_uint(l1.w)};
    tc::tmem_st8(lane_addr + kTmemAHi, hi);
    tc::tmem_st8(lane_addr + kTmemALo, lo);
    tc::tmem_wait_st();
  }
  tc_mma_round(s, tmem, tmem, s.w0, kTcW0Bytes / 2, 32, 1, parity);
  float a1[32];
  tc::tmem_ld32(lane_addr, a1);
  SWARM_PHASE(PH_PROJ);
  {
    // u = tanh(agg + b0) = 1 - 2 / (exp(2 (agg + b0)) + 1), two channels per packed instruction around the SFU ops
    const float4* b4 = reinterpret_cast<const float4*>(s.vec + TV_B0);
    const float2 two_log2e = make_float2(2.0f * 1.4426950408889634f, 2.0f * 1.4426950408889634f);
    const float2 one = make_float2(1.0f, 1.0f), neg2 = make_float2(-2.0f, -2.0f);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
      const float4 b = b4[c4];
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {
        const int c = 4 * c4 + 2 * h2;
        const float2 bb = h2 == 0 ? make_float2(b.x, b.y) : make_float2(b.z, b.w);
        const float2 z = __fmul2_rn(__fadd2_rn(make_float2(a1[c], a1[c + 1]), bb), two_log2e);
        const float2 e = __fadd2_rn(make_float2(exp2f_approx(z.x), exp2f_approx(z.y)), one);
        const float2 u = __ffma2_rn(neg2, make_float2(rcp_approx(e.x), rcp_approx(e.y)), one);
        a1[c] = u.x;
        a1[c + 1] = u.y;
      }
    }
  }
  tc_store_a_row(lane_addr, a1);
  SWARM_PHASE(PH_TANH);
  // ---- lin1 + ReLU ----
  tc_mma_round(s, tmem, tmem + 32, s.w1, kTcW1Bytes / 2, 32, 4, parity);
  tc::tmem_ld32(lane_addr + 32, a1);
  SWARM_PHASE(PH_LIN1);
  {
    const float4* b4 = reinterpret_cast<const float4*>(s.vec + TV_B1);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
      const float4 b = b4[c4];
      const float2 lo = __fadd2_rn(make_float2(a1[4 * c4 + 0], a1[4 * c4 + 1]), make_float2(b.x, b.y));
      const float2 hi = __fadd2_rn(make_float2(a1[4 * c4 + 2], a1[4 * c4 + 3]), make_float2(b.z, b.w));
      a1[4 * c4 + 0] = fmaxf(lo.x, 0.0f); a1[4 * c4 + 1] = fmaxf(lo.y, 0.0f);
      a1[4 * c4 + 2] = fmaxf(hi.x, 0.0f); a1[4 * c4 + 3] = fmaxf(hi.y, 0.0f);
    }
  }
  tc_store_a_row(lane_addr, a1);    // lin1 has completed (mbarrier), the A columns are free again
  SWARM_PHASE(PH_RELU);
  // ---- lin2 ----
  tc_mma_round(s, tmem, tmem, s.w2, kTcW2Bytes / 2, 16, 4, parity);
  float qq[16];
  tc::tmem_ld16(lane_addr, qq);
  float best = 0.0f;
  int action = 0;
#pragma unroll
  for (int a = 0; a < 9; ++a) {
    q[a] = __fadd_rn(qq[a], s.vec[TV_B2 + a]);
    if (a == 0 || q[a] > best) {
      best = q[a];
      action = a;
    }
  }
  SWARM_PHASE(PH_LIN2);
  return action;
}

}  // namespace swarm
#endif
