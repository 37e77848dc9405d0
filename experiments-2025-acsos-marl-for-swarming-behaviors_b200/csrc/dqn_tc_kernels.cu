// dqn_tc_kernels.cu -- the DQN gradient (train_gcn_dqn.py:112-137: target net on s', online net on s, TD error, backward
// pass) on the tensor cores.
//
// Same env-tile scheme as the rollout (thread = node, CTA = floor(128 / N) sampled transitions, per-CTA partial
// gradients reduced in CTA order by dqn_reduce_kernel -- no atomics, bit-reproducible), but every dense contraction
// runs on the tensor pipe and the attention layer is differentiated in INPUT space (tile_tc_device.cuh):
//
//   forward     xm_i = sum_e alpha_e x_src(e)           softmax-weighted mean of the 7 input features, CUDA cores
//               o_i = W0 xm_i + b0, u = tanh(o), p = W1 u + b1, r = relu(p), q = W2 r + b2
//                                                        three tcgen05 3xTF32 UMMA rounds, A rows in tensor memory
//   backward    dp = (W2[a]^T dq) * [r > 0];  du = W1^T dp (UMMA, B = W1^T tile);  do = du * (1 - u^2)
//               dxm = W0^T do (UMMA, B = W0^T tile);  d alpha_e = <dxm_i, x_src(e)>   -- a 7-term dot product; no
//               32-channel gather over the neighbours, no tile of projected features
//               softmax / LeakyReLU backward per in-edge;  d alpha_src_j gathered through a per-env dense matrix
//   weights     dW1 = sum_n dp_n (x) u_n,  dW2 = sum_n dq_n e_a (x) r_n,  dW0 = sum_n do_n (x) xm_n  contract over NODES:
//               every warp contracts its own 32 nodes with mma.sync m16n8k8 TF32 (3x split) from two warp-private
//               staging tiles (__syncwarp only), column sums give the bias gradients, and the attention vectors get
//               theirs through v = W0^T att:  d att = W0 dv,  dW0 += att (x) dv  with  dv_s = sum_j d alpha_src_j x_j.
//               The four warp partials are added in warp order.
// One transition set costs ~3 k instructions per warp instead of ~19 k on a CUDA-core kernel of the same scheme, and
// the CTA needs 2 x 5 KB of staging per warp instead of six 18 KB tiles.
#include "dqn_common.cuh"
#include "tile_tc_device.cuh"
#include "launchers.h"

namespace swarm {

constexpr int kStageLd = 40;                    // floats per staged row: conflict-free mma fragment loads
constexpr int kStageBuf = 32 * kStageLd;        // one warp-private tile (32 nodes)
// slots of a partial beyond the packed gradient: [1673] sum of squared TD errors, then dv_s[8], dv_d[8]
constexpr int kPartSse = SWARM_W_COUNT, kPartDvS = SWARM_W_COUNT + 1, kPartDvD = SWARM_W_COUNT + 9;
constexpr int kPartCount = SWARM_W_COUNT + 17;
static_assert(kPartCount <= 2 * kStageBuf, "a warp partial must fit the warp's two staging tiles");
constexpr int kTcW1tBytes = 2 * 32 * 32 * 4, kTcW0tBytes = 2 * 16 * 32 * 4;

struct DqnTcLayout {
  int tg_w0, tg_w1, tg_w2, tg_vec, on_w0, on_w1, on_w2, on_vec, w1t, w0t, plain, bar, st, asrc, wt, inl, kv, ki, nbr, mz,
      sdq, sact, sdasrc, sdadst, sx, xbar, stage, total;
};
// plain float32 copies of online tensors read by the CUDA-core parts: W2 [9][32], att_src [32], att_dst [32], W0 [32][7]
enum { PL_W2 = 0, PL_ATT_S = 288, PL_ATT_D = 320, PL_W0 = 352, PL_DV = 576, PL_COUNT = 592 };

__host__ __device__ inline DqnTcLayout dqn_tc_layout(int n, int k, int maxdeg, int epb, int graph_mode) {
  const int T = kTileThreads;
  DqnTcLayout L;
  int off = 0;
  auto take = [&](int bytes, int align) { off = (off + align - 1) & ~(align - 1); const int o = off; off += bytes; return o; };
  const bool knn = graph_mode == SWARM_GRAPH_KNN;
  const bool knn_rows = knn && n > 16;
  const bool complete = graph_mode == SWARM_GRAPH_COMPLETE;
  L.tg_w0 = take(kTcW0Bytes, 128); L.tg_w1 = take(kTcW1Bytes, 128); L.tg_w2 = take(kTcW2Bytes, 128);
  L.on_w0 = take(kTcW0Bytes, 128); L.on_w1 = take(kTcW1Bytes, 128); L.on_w2 = take(kTcW2Bytes, 128);
  L.w1t = take(kTcW1tBytes, 128); L.w0t = take(kTcW0tBytes, 128);
  L.tg_vec = take(TV_COUNT * 4, 16); L.on_vec = take(TV_COUNT * 4, 16);
  L.plain = take(PL_COUNT * 4, 16);
  L.bar = take(16, 16);
  L.st = take(T * 16, 16);
  L.asrc = take(T * 4, 16);
  L.wt = take(maxdeg * T * 4, 16);
  L.inl = take(complete ? 0 : maxdeg * T, 16);
  L.kv = take(knn ? (knn_rows ? n : 1) * T * 4 : 0, 16);
  L.ki = take(knn_rows ? n * T : 0, 16);
  L.nbr = take(knn_rows ? k * T : 0, 16);
  L.mz = take(epb * n * n * 4, 16);
  L.sdq = take(T * 4, 16); L.sact = take(T * 4, 16); L.sdasrc = take(T * 4, 16); L.sdadst = take(T * 4, 16);
  L.sx = take(T * 8 * 4, 16);
  L.xbar = take(T * 8 * 4, 16);
  L.stage = take(4 * 2 * kStageBuf * 4, 16);
  L.total = off;
  return L;
}

// ---- extra B tiles of the backward pass --------------------------------------------------------------------------
// w1t: B[n = k][K = c] = W1[c][k]  (du = W1^T dp);  w0t: B[n = k < 7, padded to 16][K = c] = W0[c][k]  (dxm = W0^T do)
struct BwdStageRegs {
  float4 item[(256 + 128) / kTileThreads];                     // 3
  float pv[(PL_DV + kTileThreads - 1) / kTileThreads];         // 5
};

__device__ __forceinline__ void stage_backward_load(const float* __restrict__ gw, BwdStageRegs& r, int tid, int nthreads) {
  constexpr int kItems = (256 + 128) / kTileThreads;
  constexpr int kPlain = (PL_DV + kTileThreads - 1) / kTileThreads;
#pragma unroll
  for (int q = 0; q < kItems; ++q) {
    const int it = tid + q * nthreads;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (it < 256) {
      const int n = it >> 3, c = it & 7;
      const float* col = gw + SWARM_W_LIN1 + n;                 // W1[4c + j][n]
      v = make_float4(col[(4 * c + 0) * 32], col[(4 * c + 1) * 32], col[(4 * c + 2) * 32], col[(4 * c + 3) * 32]);
    } else if (it < 384) {
      const int j = it - 256, n = j >> 3, c = j & 7;
      if (n < 7) {
        const float* col = gw + SWARM_W_CONV_LIN + n;           // W0[4c + j][n]
        v = make_float4(col[(4 * c + 0) * 7], col[(4 * c + 1) * 7], col[(4 * c + 2) * 7], col[(4 * c + 3) * 7]);
      }
    }
    r.item[q] = v;
  }
#pragma unroll
  for (int q = 0; q < kPlain; ++q) {
    const int o = tid + q * nthreads;
    float v = 0.0f;
    if (o < PL_ATT_S) v = gw[SWARM_W_LIN2 + o];
    else if (o < PL_ATT_D) v = gw[SWARM_W_ATT_SRC + (o - PL_ATT_S)];
    else if (o < PL_W0) v = gw[SWARM_W_ATT_DST + (o - PL_ATT_D)];
    else if (o < PL_DV) v = gw[SWARM_W_CONV_LIN + (o - PL_W0)];
    r.pv[q] = v;
  }
}

__device__ __forceinline__ void stage_backward_store(const BwdStageRegs& r, unsigned char* w1t, unsigned char* w0t, float* plain,
                                                     int tid, int nthreads) {
  constexpr int kItems = (256 + 128) / kTileThreads;
  constexpr int kPlain = (PL_DV + kTileThreads - 1) / kTileThreads;
#pragma unroll
  for (int q = 0; q < kItems; ++q) {
    const int it = tid + q * nthreads;
    if (it >= 384) break;
    unsigned char* base;
    int rows, n, c, half;
    if (it < 256) {
      n = it >> 3; c = it & 7; rows = 32; base = w1t; half = kTcW1tBytes / 2;
    } else {
      const int j = it - 256;
      n = j >> 3; c = j & 7; rows = 16; base = w0t; half = kTcW0tBytes / 2;
    }
    float4 hi, lo;
    tc::split4(r.item[q], hi, lo);
    const int off = tc::tile_off(rows, n, c);
    *reinterpret_cast<float4*>(base + off) = hi;
    *reinterpret_cast<float4*>(base + half + off) = lo;
  }
#pragma unroll
  for (int q = 0; q < kPlain; ++q) {
    const int o = tid + q * nthreads;
    if (o < PL_DV) plain[o] = r.pv[q];
  }
}

// ---- warp-level node contraction on mma.sync (m16n8k8, TF32, 3x split) --------------------------------------------
__device__ __forceinline__ void split_frag(float x, uint32_t& hi, uint32_t& lo) {
  float h, l;
  tc::split_tf32(x, h, l);
  hi = __float_as_uint(h);
  lo = __float_as_uint(l);
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// acc[mt][nt] += sum over this warp's 32 nodes of left(node, m) * right(node, n); m = mt * 16 + row, n = nt * 8 + col.
// Fragment ownership (g = lane / 4, tg = lane % 4): A (g | g + 8, tg | tg + 4), B (k = tg | tg + 4, n = g),
// C (g | g + 8, 2 tg | 2 tg + 1).  Small terms first, like the UMMA path.
// `ksteps` = groups of 8 nodes that can be non-zero (a CTA with one 12-node graph contracts 2 groups in warp 0, none elsewhere)
template <int MT, int NT, typename FL, typename FR>
__device__ __forceinline__ void warp_node_gemm(float (&acc)[MT][NT][4], int lane, int ksteps, FL left, FR right) {
  const int g = lane >> 2, tg = lane & 3;
#pragma unroll 1
  for (int ks = 0; ks < ksteps; ++ks) {
    const int n0 = ks * 8 + tg, n1 = n0 + 4;
    uint32_t ah[MT][4], al[MT][4], bh[NT][2], bl[NT][2];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      split_frag(left(n0, mt * 16 + g), ah[mt][0], al[mt][0]);
      split_frag(left(n0, mt * 16 + g + 8), ah[mt][1], al[mt][1]);
      split_frag(left(n1, mt * 16 + g), ah[mt][2], al[mt][2]);
      split_frag(left(n1, mt * 16 + g + 8), ah[mt][3], al[mt][3]);
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      split_frag(right(n0, nt * 8 + g), bh[nt][0], bl[nt][0]);
      split_frag(right(n1, nt * 8 + g), bh[nt][1], bl[nt][1]);
    }
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        mma_tf32(acc[mt][nt], al[mt], bh[nt]);
        mma_tf32(acc[mt][nt], ah[mt], bl[nt]);
        mma_tf32(acc[mt][nt], ah[mt], bh[nt]);
      }
  }
}

__device__ __forceinline__ void stage_row(float* buf, int lane, const float (&v)[32]) {
  float4* r = reinterpret_cast<float4*>(buf + lane * kStageLd);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) r[c4] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
}

// softmax weights and weighted mean of the neighbours' input features, keeping what the backward pass needs:
// the unnormalised weights w_e in swt[e][tid] and 1 / (sum + 1e-16).  Exact expf / division here -- the TD error is a
// small difference of large Q values, so the forward pass of the update keeps float32-level accuracy throughout.
template <bool COMPLETE, bool KEEP>
__device__ __forceinline__ float dqn_attend(const TileGraphSmem& g, const TileThread& t, const float4* __restrict__ pos,
                                            int N, int deg, float adst, float goal_x, float goal_y, float (&xm)[8]) {
  const int T = kTileThreads;
  const float* __restrict__ sas = g.sas + t.envbase;
  const float4* __restrict__ env = pos + t.envbase;
  float* __restrict__ swt = g.swt + t.tid;
  const uint8_t* __restrict__ sin = g.sin + t.tid;
  const int self = (t.i == 0) ? -1 : t.i;                      // complete graph: node 0 keeps its (0,0) self loop
  const int n_edges = COMPLETE ? (t.active ? N : 0) : deg;
  float amax = -INFINITY;
#pragma unroll 4
  for (int e = 0; e < n_edges; ++e) {
    const int j = COMPLETE ? e : (int)sin[e * T];
    amax = fmaxf(amax, (COMPLETE && j == self) ? -INFINITY : sas[j]);
  }
  const float zt = __fadd_rn(amax, adst);
  const float m = fmaxf(zt, __fmul_rn(zt, 0.2f));
  float den = 0.0f, acc_id = 0.0f;
  float2 acc_p = make_float2(0.0f, 0.0f), acc_v = make_float2(0.0f, 0.0f);
#pragma unroll 2
  for (int e = 0; e < n_edges; ++e) {
    const int j = COMPLETE ? e : (int)sin[e * T];
    const float4 sj = env[j];
    const float zz = __fadd_rn(sas[j], adst);
    float w = expf(__fsub_rn(fmaxf(zz, __fmul_rn(zz, 0.2f)), m));
    if (COMPLETE && j == self) w = 0.0f;
    if (KEEP) swt[e * T] = w;
    const float2 w2 = make_float2(w, w);
    den = __fadd_rn(den, w);
    acc_p = __ffma2_rn(w2, make_float2(sj.x, sj.y), acc_p);
    acc_v = __ffma2_rn(w2, make_float2(sj.z, sj.w), acc_v);
    acc_id = fmaf(w, (float)j, acc_id);
  }
  const float inv = __fdiv_rn(1.0f, __fadd_rn(den, 1e-16f));
  const float wsum = den * inv;
  xm[0] = acc_p.x * inv; xm[1] = acc_p.y * inv; xm[2] = acc_v.x * inv; xm[3] = acc_v.y * inv;
  xm[4] = goal_x * wsum; xm[5] = goal_y * wsum; xm[6] = acc_id * inv; xm[7] = 0.0f;
  return inv;
}

// complete graph, online and target pass in one loop (two independent dependency chains per iteration)
__device__ __forceinline__ float dqn_attend_pair(const TileGraphSmem& go, const TileGraphSmem& gt, const TileThread& t,
                                                 const float4* __restrict__ pos_o, const float4* __restrict__ pos_t, int N,
                                                 float adst_o, float adst_t, float goal_x, float goal_y, float (&xo)[8],
                                                 float (&xt)[8]) {
  const int T = kTileThreads;
  const float* __restrict__ sas_o = go.sas + t.envbase;
  const float* __restrict__ sas_t = gt.sas + t.envbase;
  const float4* __restrict__ env_o = pos_o + t.envbase;
  const float4* __restrict__ env_t = pos_t + t.envbase;
  float* __restrict__ swt = go.swt + t.tid;
  const int self = (t.i == 0) ? -1 : t.i;
  const int n = t.active ? N : 0;
  float amax_o = -INFINITY, amax_t = -INFINITY;
#pragma unroll 4
  for (int j = 0; j < n; ++j) {
    amax_o = fmaxf(amax_o, j == self ? -INFINITY : sas_o[j]);
    amax_t = fmaxf(amax_t, j == self ? -INFINITY : sas_t[j]);
  }
  const float zo = __fadd_rn(amax_o, adst_o), zt = __fadd_rn(amax_t, adst_t);
  const float mo = fmaxf(zo, __fmul_rn(zo, 0.2f)), mt = fmaxf(zt, __fmul_rn(zt, 0.2f));
  float den_o = 0.0f, den_t = 0.0f, id_o = 0.0f, id_t = 0.0f, fj = 0.0f;
  float2 po = make_float2(0.f, 0.f), vo = po, pt = po, vt = po;
#pragma unroll 4
  for (int j = 0; j < n; ++j) {
    const float4 so = env_o[j], st = env_t[j];
    const float ao = __fadd_rn(sas_o[j], adst_o), at = __fadd_rn(sas_t[j], adst_t);
    float wo = expf(__fsub_rn(fmaxf(ao, __fmul_rn(ao, 0.2f)), mo));
    float wt = expf(__fsub_rn(fmaxf(at, __fmul_rn(at, 0.2f)), mt));
    if (j == self) { wo = 0.0f; wt = 0.0f; }
    swt[j * T] = wo;
    den_o = __fadd_rn(den_o, wo);
    den_t = __fadd_rn(den_t, wt);
    po = __ffma2_rn(make_float2(wo, wo), make_float2(so.x, so.y), po);
    vo = __ffma2_rn(make_float2(wo, wo), make_float2(so.z, so.w), vo);
    pt = __ffma2_rn(make_float2(wt, wt), make_float2(st.x, st.y), pt);
    vt = __ffma2_rn(make_float2(wt, wt), make_float2(st.z, st.w), vt);
    id_o = fmaf(wo, fj, id_o);
    id_t = fmaf(wt, fj, id_t);
    fj += 1.0f;
  }
  const float inv_o = __fdiv_rn(1.0f, __fadd_rn(den_o, 1e-16f)), inv_t = __fdiv_rn(1.0f, __fadd_rn(den_t, 1e-16f));
  const float ws_o = den_o * inv_o, ws_t = den_t * inv_t;
  xo[0] = po.x * inv_o; xo[1] = po.y * inv_o; xo[2] = vo.x * inv_o; xo[3] = vo.y * inv_o;
  xo[4] = goal_x * ws_o; xo[5] = goal_y * ws_o; xo[6] = id_o * inv_o; xo[7] = 0.0f;
  xt[0] = pt.x * inv_t; xt[1] = pt.y * inv_t; xt[2] = vt.x * inv_t; xt[3] = vt.y * inv_t;
  xt[4] = goal_x * ws_t; xt[5] = goal_y * ws_t; xt[6] = id_t * inv_t; xt[7] = 0.0f;
  return inv_o;
}

__device__ __forceinline__ void tc_store_a8(uint32_t lane_addr, const float (&v)[8]) {
  float4 h0, l0, h1, l1;
  tc::split4(make_float4(v[0], v[1], v[2], v[3]), h0, l0);
  tc::split4(make_float4(v[4], v[5], v[6], v[7]), h1, l1);
  const uint32_t hi[8] = {__float_as_uint(h0.x), __float_as_uint(h0.y), __float_as_uint(h0.z), __float_as_uint(h0.w),
                          __float_as_uint(h1.x), __float_as_uint(h1.y), __float_as_uint(h1.z), __float_as_uint(h1.w)};
  const uint32_t lo[8] = {__float_as_uint(l0.x), __float_as_uint(l0.y), __float_as_uint(l0.z), __float_as_uint(l0.w),
                          __float_as_uint(l1.x), __float_as_uint(l1.y), __float_as_uint(l1.z), __float_as_uint(l1.w)};
  tc::tmem_st8(lane_addr + kTmemAHi, hi);
  tc::tmem_st8(lane_addr + kTmemALo, lo);
  tc::tmem_wait_st();
}

// TMEM columns: the online network uses [0, 128) as in the rollout (D tiles [0, 64), A hi / lo [64, 128)), the target
// network the same layout 128 columns further on, so both forward passes advance together: every thread writes both
// operand rows, ONE round issues the two 3xTF32 products (target weights for the target rows, online weights for the
// online rows) behind one barrier and one mbarrier wait.  Halves the number of round trips of the forward passes and
// gives each thread two independent epilogue chains.
constexpr int kDqnTmemCols = 256;
constexpr uint32_t kTmemTarget = 128;

__device__ __forceinline__ void tc_mma_round2(uint64_t* bar, uint32_t tmem, uint32_t d_off, const unsigned char* b_on,
                                              const unsigned char* b_tg, int b_half, int b_rows, int ksteps,
                                              uint32_t& parity) {
  tc::fence_before_sync();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) {
    tc::fence_after_sync();
    if (tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc_tf32(b_rows);
      const uint32_t bo = tc::smem_u32(b_on), bt = tc::smem_u32(b_tg);
      tc::mma_3xtf32_tmem_a(tmem + kTmemTarget + d_off, tmem + kTmemTarget + kTmemAHi, tmem + kTmemTarget + kTmemALo, bt,
                            bt + b_half, b_rows, ksteps, idesc);
      tc::mma_3xtf32_tmem_a(tmem + d_off, tmem + kTmemAHi, tmem + kTmemALo, bo, bo + b_half, b_rows, ksteps, idesc);
      tc::mma_commit(bar);
    }
    __syncwarp();
  }
  tc::mbar_wait(bar, parity);
  parity ^= 1u;
  tc::fence_after_sync();
}

// u = tanh(o + b0) = 1 - 2 / (exp(2 (o + b0)) + 1) on the SFU like the rollout's forward (absolute error ~1e-7; tanhf
// costs 17 instructions per channel and was a sixth of this kernel)
__device__ __forceinline__ void dqn_tanh_bias(float (&u)[32], const float* __restrict__ b0) {
  const float4* b4 = reinterpret_cast<const float4*>(b0);
  const float2 two_log2e = make_float2(2.0f * 1.4426950408889634f, 2.0f * 1.4426950408889634f);
  const float2 one = make_float2(1.0f, 1.0f), neg2 = make_float2(-2.0f, -2.0f);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) {
    const float4 b = b4[c4];
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {
      const int k = 4 * c4 + 2 * h2;
      const float2 bb = h2 == 0 ? make_float2(b.x, b.y) : make_float2(b.z, b.w);
      const float2 z = __fmul2_rn(__fadd2_rn(make_float2(u[k], u[k + 1]), bb), two_log2e);
      const float2 e = __fadd2_rn(make_float2(exp2f_approx(z.x), exp2f_approx(z.y)), one);
      const float2 uu = __ffma2_rn(neg2, make_float2(rcp_approx(e.x), rcp_approx(e.y)), one);
      u[k] = uu.x;
      u[k + 1] = uu.y;
    }
  }
}
__device__ __forceinline__ void dqn_relu_bias(float (&r)[32], const float* __restrict__ b1) {
#pragma unroll
  for (int k = 0; k < 32; ++k) r[k] = fmaxf(__fadd_rn(r[k], b1[k]), 0.0f);
}

template <bool COMPLETE>
__global__ void __launch_bounds__(kTileThreads, 2) dqn_grad_tc_kernel(const __grid_constant__ DqnParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const SwarmConfig& c = p.cfg;
  const int T = kTileThreads;
  const int N = c.n_agents;
  const int K = c.knn_k;
  const bool knn = c.graph_mode == SWARM_GRAPH_KNN;
  const bool radius = c.graph_mode == SWARM_GRAPH_RADIUS;
  TileThread t = tile_thread(N, p.epb, p.n_graphs);
  const int tid = t.tid, lane = tid & 31, warp = tid >> 5;

  long long ring_size = 0;
  if (p.ctl) {
    ring_size = train_ring_size(p.ctl, p.pushed_envs, p.batch.capacity);
    if (ring_size < p.n_graphs) return;        // replay ring not filled yet (train:113-115)
  }

  const DqnTcLayout L = dqn_tc_layout(N, K, p.maxdeg, p.epb, c.graph_mode);
  TileTcSmem ts_tg, ts_on;
  ts_tg.w0 = smem + L.tg_w0; ts_tg.w1 = smem + L.tg_w1; ts_tg.w2 = smem + L.tg_w2;
  ts_tg.vec = reinterpret_cast<float*>(smem + L.tg_vec);
  ts_on.w0 = smem + L.on_w0; ts_on.w1 = smem + L.on_w1; ts_on.w2 = smem + L.on_w2;
  ts_on.vec = reinterpret_cast<float*>(smem + L.on_vec);
  ts_tg.bar = ts_on.bar = reinterpret_cast<uint64_t*>(smem + L.bar);
  ts_tg.tmem_slot = ts_on.tmem_slot = reinterpret_cast<uint32_t*>(smem + L.bar + 8);
  unsigned char* w1t = smem + L.w1t;
  unsigned char* w0t = smem + L.w0t;
  float* plain = reinterpret_cast<float*>(smem + L.plain);
  float4* sst = reinterpret_cast<float4*>(smem + L.st);
  TileGraphSmem g;
  g.sh = nullptr;
  g.sas = reinterpret_cast<float*>(smem + L.asrc);
  g.swt = reinterpret_cast<float*>(smem + L.wt);
  g.sin = smem + L.inl;
  g.skv = reinterpret_cast<float*>(smem + L.kv);
  g.ski = smem + L.ki;
  g.snbr = smem + L.nbr;
  float* mZ = reinterpret_cast<float*>(smem + L.mz);
  float* sdq = reinterpret_cast<float*>(smem + L.sdq);
  int* sact = reinterpret_cast<int*>(smem + L.sact);
  float* sdasrc = reinterpret_cast<float*>(smem + L.sdasrc);
  float* sdadst = reinterpret_cast<float*>(smem + L.sdadst);
  float* sx = reinterpret_cast<float*>(smem + L.sx);
  float* sxbar = reinterpret_cast<float*>(smem + L.xbar);
  float* stage_all = reinterpret_cast<float*>(smem + L.stage);
  float* buf0 = stage_all + (warp * 2 + 0) * kStageBuf;         // U, then (with buf1) this warp's partial
  float* buf1 = stage_all + (warp * 2 + 1) * kStageBuf;         // R, then DP, then DO
  // node rows of this warp that belong to a graph (the rest contribute exact zeros: dq = 0)
  const int wnodes = min(32, max(0, min(p.epb, p.n_graphs - (int)blockIdx.x * p.epb) * N - warp * 32));
  const int wsteps = (wnodes + 7) >> 3;

  // ---- the sampled transition of this node (loads in flight while the weights are staged) -------------------------
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s;
  int act = 0;
  float rew = 0.0f;
  if (t.active) {
    long long slot = t.env;
    if (p.ctl) {
      const uint64_t rnd = rng_draw(p.sample_seed, (uint64_t)t.env, (uint64_t)(p.ctl->tick + 1), 0x5A17u);
      slot = (long long)__umul64hi(rnd, (uint64_t)ring_size);
      if (p.indices_out && t.i == 0) p.indices_out[t.env] = slot;
    } else if (p.indices) {
      slot = p.indices[t.env];
      slot = slot < 0 ? 0 : (slot >= p.batch.capacity ? p.batch.capacity - 1 : slot);
    }
    const long long ri = slot * N + t.i;
    s = reinterpret_cast<const float4*>(p.batch.state)[ri];
    s2 = reinterpret_cast<const float4*>(p.batch.next_state)[ri];
    act = sanitize_action(p.batch.actions[ri]);
    rew = p.batch.rewards[ri];
  }

  {
    // all global loads of the three weight sets first (the v_s / v_d chains of the two networks on warps 0 and 1; the vector block takes 96 threads),
    // then the shared-memory stores: one exposed round trip to L2 for the whole prologue
    TcStageRegs rt, ro;
    BwdStageRegs rb;
    stage_weights_tc_load(p.w_target, rt, tid, T, tid - 32);
    stage_weights_tc_load(p.w_online, ro, tid, T, tid);
    stage_backward_load(p.w_online, rb, tid, T);
    stage_weights_tc_store(rt, ts_tg, tid, T, tid - 32);
    stage_weights_tc_store(ro, ts_on, tid, T, tid);
    stage_backward_store(rb, w1t, w0t, plain, tid, T);
  }
  if (tid == 0) tc::mbar_init(ts_on.bar, 1);
  if (warp == 0) tc::tmem_alloc(ts_on.tmem_slot, kDqnTmemCols);
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *ts_on.tmem_slot;
  const uint32_t lane_addr = tmem + ((uint32_t)(tid & ~31) << 16);
  uint32_t parity = 0;

  float u[32], r[32], xm[8];
  float adst = 0.0f, inv = 0.0f, y = 0.0f, v_taken = 0.0f;
  int deg = 0;

  // target network on s' -> y = r + gamma * max_a Q_target(s')  (train:120-121) and online network on s (train:119),
  // advancing together.  The target pass's state / alpha_src / edge list live in the (still unused) staging tiles.
  {
    float4* sst_t = reinterpret_cast<float4*>(stage_all);
    TileGraphSmem gt = g;
    gt.sas = stage_all + 4 * T;
    gt.sin = reinterpret_cast<uint8_t*>(stage_all + 5 * T);
    const float x_o[7] = {s.x, s.y, s.z, s.w, c.goal_x, c.goal_y, (float)t.i};
    const float x_t[7] = {s2.x, s2.y, s2.z, s2.w, c.goal_x, c.goal_y, (float)t.i};
    float asrc_o, asrc_t, adst_t;
    tc_alpha_terms(ts_on, x_o, asrc_o, adst);
    tc_alpha_terms(ts_tg, x_t, asrc_t, adst_t);
    sst[tid] = s;
    g.sas[tid] = asrc_o;
    sst_t[tid] = s2;
    gt.sas[tid] = asrc_t;
    {
      float4* xr = reinterpret_cast<float4*>(sx + tid * 8);
      xr[0] = make_float4(x_o[0], x_o[1], x_o[2], x_o[3]);
      xr[1] = make_float4(x_o[4], x_o[5], x_o[6], 0.f);
    }
    __syncthreads();
    int deg_t = 0;
    if (!COMPLETE) {
      auto in_edges = [&](const TileGraphSmem& gg, const float4* pos, const float4& sp) -> int {
        if (knn && N <= kKnnSmallMax) {
          uint64_t cache_rank = ~0ull, cache_nbr = 0;
          const uint64_t nbr_word = tile_knn_small(t, pos, sp, N, K, cache_rank, cache_nbr);
          return tile_in_edges_knn_small(gg, t, N, K, nbr_word, reinterpret_cast<uint32_t*>(gg.skv));
        } else if (knn) {
          tile_knn_rows(gg, t, pos, sp, N, K);
          return tile_in_edges_knn(gg, t, N, K, reinterpret_cast<uint32_t*>(gg.skv));
        }
        return t.active ? tile_in_edges_radius(gg, t, pos, sp, N, p.qmax_r) : 0;
      };
      deg_t = in_edges(gt, sst_t, s2);
      __syncthreads();                             // the kNN scratch is shared by the two builds
      deg = in_edges(g, sst, s);
    }
    float xm_t[8];
    if (COMPLETE) {
      inv = dqn_attend_pair(g, gt, t, sst, sst_t, N, adst, adst_t, c.goal_x, c.goal_y, xm, xm_t);
    } else {
      dqn_attend<COMPLETE, false>(gt, t, sst_t, N, deg_t, adst_t, c.goal_x, c.goal_y, xm_t);
      inv = dqn_attend<COMPLETE, true>(g, t, sst, N, deg, adst, c.goal_x, c.goal_y, xm);
    }
    tc_store_a8(lane_addr + kTmemTarget, xm_t);
    tc_store_a8(lane_addr, xm);
    tc_mma_round2(ts_on.bar, tmem, 0, ts_on.w0, ts_tg.w0, kTcW0Bytes / 2, 32, 1, parity);
    float ut[32];
    tc::tmem_ld32(lane_addr + kTmemTarget, ut);
    tc::tmem_ld32(lane_addr, u);
    dqn_tanh_bias(ut, ts_tg.vec + TV_B0);
    dqn_tanh_bias(u, ts_on.vec + TV_B0);
    tc_store_a_row(lane_addr + kTmemTarget, ut);
    tc_store_a_row(lane_addr, u);
    tc_mma_round2(ts_on.bar, tmem, 32, ts_on.w1, ts_tg.w1, kTcW1Bytes / 2, 32, 4, parity);
    tc::tmem_ld32(lane_addr + kTmemTarget + 32, ut);
    tc::tmem_ld32(lane_addr + 32, r);
    dqn_relu_bias(ut, ts_tg.vec + TV_B1);
    dqn_relu_bias(r, ts_on.vec + TV_B1);
    tc_store_a_row(lane_addr + kTmemTarget, ut);
    tc_store_a_row(lane_addr, r);
    tc_mma_round2(ts_on.bar, tmem, 0, ts_on.w2, ts_tg.w2, kTcW2Bytes / 2, 16, 4, parity);
    float qt[16], qo[16];
    tc::tmem_ld16(lane_addr + kTmemTarget, qt);
    tc::tmem_ld16(lane_addr, qo);
    float qmax = __fadd_rn(qt[0], ts_tg.vec[TV_B2]);
#pragma unroll
    for (int a = 1; a < 9; ++a) qmax = fmaxf(qmax, __fadd_rn(qt[a], ts_tg.vec[TV_B2 + a]));
    y = __fadd_rn(rew, __fmul_rn(p.gamma, qmax));
    v_taken = __fadd_rn(qo[0], ts_on.vec[TV_B2]);
#pragma unroll
    for (int a = 1; a < 9; ++a) v_taken = (act == a) ? __fadd_rn(qo[a], ts_on.vec[TV_B2 + a]) : v_taken;   // Q(s).gather(1, a)
  }

  // ---- TD error --------------------------------------------------------------------------------------------------
  float delta = 0.0f, dq = 0.0f;
  if (t.active) {
    delta = __fsub_rn(v_taken, y);
    dq = 2.0f * delta * p.loss_scale;             // d mean((v - y)^2) / dv
    if (p.td) p.td[t.gidx] = delta;
  }
  sdq[tid] = dq;
  sact[tid] = act;
  stage_row(buf0, lane, u);
  stage_row(buf1, lane, r);
  {
    float4* xb = reinterpret_cast<float4*>(sxbar + tid * 8);
    xb[0] = make_float4(xm[0], xm[1], xm[2], xm[3]);
    xb[1] = make_float4(xm[4], xm[5], xm[6], 0.f);
  }
  __syncwarp();

  // ---- dW2 = sum_n dq_n e_{a_n} (x) r_n ;  d lin2.bias ---------------------------------------------------------------
  float acc2[1][4][4];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt)
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4) acc2[0][nt][q4] = 0.0f;
  {
    const float* wdq = sdq + warp * 32;
    const int* wact = sact + warp * 32;
    warp_node_gemm<1, 4>(acc2, lane, wsteps, [&](int n, int m) { return wact[n] == m ? wdq[n] : 0.0f; },
                         [&](int n, int col) { return buf1[n * kStageLd + col]; });
  }
  float db2 = 0.0f;
  if (lane < 9) {
    for (int n = 0; n < 32; ++n) db2 += (sact[warp * 32 + n] == lane) ? sdq[warp * 32 + n] : 0.0f;
  }

  // ---- backward through lin2 / ReLU:  dp = (W2[a]^T dq) * [r > 0] --------------------------------------------------
  float dvec[32];
  {
    const float4* w2a = reinterpret_cast<const float4*>(plain + PL_W2 + act * 32);
#pragma unroll
    for (int k4 = 0; k4 < 8; ++k4) {
      const float4 w = w2a[k4];
      dvec[4 * k4 + 0] = r[4 * k4 + 0] > 0.0f ? w.x * dq : 0.0f;
      dvec[4 * k4 + 1] = r[4 * k4 + 1] > 0.0f ? w.y * dq : 0.0f;
      dvec[4 * k4 + 2] = r[4 * k4 + 2] > 0.0f ? w.z * dq : 0.0f;
      dvec[4 * k4 + 3] = r[4 * k4 + 3] > 0.0f ? w.w * dq : 0.0f;
    }
  }
  __syncwarp();                                    // every lane is done with the R tile
  stage_row(buf1, lane, dvec);
  tc_store_a_row(lane_addr, dvec);
  __syncwarp();

  // ---- dW1 = sum_n dp_n (x) u_n ;  d lin1.bias ----------------------------------------------------------------------
  float acc1[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) acc1[mt][nt][q4] = 0.0f;
  warp_node_gemm<2, 4>(acc1, lane, wsteps, [&](int n, int m) { return buf1[n * kStageLd + m]; },
                       [&](int n, int col) { return buf0[n * kStageLd + col]; });
  float db1 = 0.0f;
  for (int n = 0; n < 32; ++n) db1 += buf1[n * kStageLd + lane];

  // ---- du = W1^T dp (UMMA);  do = du * (1 - u^2) ---------------------------------------------------------------------
  tc_mma_round(ts_on, tmem, tmem + 32, w1t, kTcW1tBytes / 2, 32, 4, parity);
  tc::tmem_ld32(lane_addr + 32, dvec);
#pragma unroll
  for (int k = 0; k < 32; ++k) dvec[k] = dvec[k] * (1.0f - u[k] * u[k]);     // dvec = d(o_i) from here on
  __syncwarp();                                    // every lane is done with the DP tile
  stage_row(buf1, lane, dvec);
  tc_store_a_row(lane_addr, dvec);
  __syncwarp();

  // ---- dW0 = sum_n do_n (x) xm_n ;  d conv1.bias --------------------------------------------------------------------
  float acc0[2][1][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4) acc0[mt][0][q4] = 0.0f;
  {
    const float* wxb = sxbar + warp * 32 * 8;
    warp_node_gemm<2, 1>(acc0, lane, wsteps, [&](int n, int m) { return buf1[n * kStageLd + m]; },
                         [&](int n, int col) { return wxb[n * 8 + col]; });
  }
  float db0 = 0.0f;
  for (int n = 0; n < 32; ++n) db0 += buf1[n * kStageLd + lane];

  // ---- dxm = W0^T do (UMMA);  attention backward in input space ---------------------------------------------------------
  tc_mma_round(ts_on, tmem, tmem, w0t, kTcW0tBytes / 2, 16, 4, parity);
  float dxm[16];
  tc::tmem_ld16(lane_addr, dxm);
  float dadst = 0.0f;
  {
    const int T_ = T;
    const float* __restrict__ sas = g.sas + t.envbase;
    const float4* __restrict__ env = sst + t.envbase;
    const float* __restrict__ swt = g.swt + tid;
    const uint8_t* __restrict__ sin = g.sin + tid;
    float* rz = mZ + (t.el * N + t.i) * N;
    const int n_edges = COMPLETE ? (t.active ? N : 0) : deg;
    if (!COMPLETE && t.active)
      for (int j = 0; j < N; ++j) rz[j] = 0.0f;
    const float cg = fmaf(dxm[4], c.goal_x, dxm[5] * c.goal_y);
    auto dalpha = [&](int j) {
      const float4 sj = env[j];
      return fmaf(dxm[0], sj.x, fmaf(dxm[1], sj.y, fmaf(dxm[2], sj.z, fmaf(dxm[3], sj.w, fmaf(dxm[6], (float)j, cg)))));
    };
    // softmax backward: d z_e = alpha_e (d alpha_e - sum_e' alpha_e' d alpha_e')
    float dot_sum = 0.0f;
#pragma unroll 2
    for (int e = 0; e < n_edges; ++e) {
      const int j = COMPLETE ? e : (int)sin[e * T_];
      dot_sum = fmaf(swt[e * T_] * inv, dalpha(j), dot_sum);
    }
#pragma unroll 2
    for (int e = 0; e < n_edges; ++e) {
      const int j = COMPLETE ? e : (int)sin[e * T_];
      const float alpha = swt[e * T_] * inv;
      const float dz = alpha * (dalpha(j) - dot_sum);
      const float raw = __fadd_rn(sas[j], adst);
      const float dzz = raw > 0.0f ? dz : 0.2f * dz;
      if (COMPLETE) rz[j] = dzz;
      else rz[j] += dzz;                          // parallel edges (duplicates, double self loops) accumulate
      dadst += dzz;
    }
  }
  sdadst[tid] = dadst;
  __syncthreads();            // mZ complete (an env may straddle two warps)
  {
    float ds = 0.0f;
    if (t.active)
      for (int ii = 0; ii < N; ++ii) ds += mZ[(t.el * N + ii) * N + t.i];
    sdasrc[tid] = ds;
  }
  __syncwarp();

  // ---- dv_s = sum_j d alpha_src_j x_j,  dv_d = sum_i d alpha_dst_i x_i over this warp's nodes; squared TD errors -----
  float dv = 0.0f;
  if (lane < 16) {
    const float* coef = (lane < 8 ? sdasrc : sdadst) + warp * 32;
    const float* xr = sx + warp * 32 * 8 + (lane & 7);
    for (int n = 0; n < 32; ++n) dv = fmaf(coef[n], xr[n * 8], dv);
  }
  float sse = delta * delta;
#pragma unroll
  for (int sh = 16; sh > 0; sh >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, sh);

  // ---- this warp's partial into its own staging tiles (every lane is done reading them) ---------------------------
  __syncwarp();
  float* part = buf0;                              // buf0 and buf1 are contiguous; every slot read below is written here
  {
    const int gq = lane >> 2, tg = lane & 3;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int k0 = nt * 8 + 2 * tg;
      if (gq < 9) {
        part[SWARM_W_LIN2 + gq * 32 + k0] = acc2[0][nt][0];
        part[SWARM_W_LIN2 + gq * 32 + k0 + 1] = acc2[0][nt][1];
      }
      if (gq + 8 < 9) {
        part[SWARM_W_LIN2 + (gq + 8) * 32 + k0] = acc2[0][nt][2];
        part[SWARM_W_LIN2 + (gq + 8) * 32 + k0 + 1] = acc2[0][nt][3];
      }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const int c0 = mt * 16 + gq;
        part[SWARM_W_LIN1 + c0 * 32 + k0] = acc1[mt][nt][0];
        part[SWARM_W_LIN1 + c0 * 32 + k0 + 1] = acc1[mt][nt][1];
        part[SWARM_W_LIN1 + (c0 + 8) * 32 + k0] = acc1[mt][nt][2];
        part[SWARM_W_LIN1 + (c0 + 8) * 32 + k0 + 1] = acc1[mt][nt][3];
      }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int c0 = mt * 16 + gq, k0 = 2 * tg;
      if (k0 < 7) {
        part[SWARM_W_CONV_LIN + c0 * 7 + k0] = acc0[mt][0][0];
        part[SWARM_W_CONV_LIN + (c0 + 8) * 7 + k0] = acc0[mt][0][2];
      }
      if (k0 + 1 < 7) {
        part[SWARM_W_CONV_LIN + c0 * 7 + k0 + 1] = acc0[mt][0][1];
        part[SWARM_W_CONV_LIN + (c0 + 8) * 7 + k0 + 1] = acc0[mt][0][3];
      }
    }
    part[SWARM_W_LIN1_BIAS + lane] = db1;
    part[SWARM_W_CONV_BIAS + lane] = db0;
    if (lane < 9) part[SWARM_W_LIN2_BIAS + lane] = db2;
    if (lane < 8) part[kPartDvS + lane] = dv;
    else if (lane < 16) part[kPartDvD + (lane - 8)] = dv;
    if (lane == 0) part[kPartSse] = sse;
  }
  __syncthreads();

  // ---- warp partials added in warp order; the attention vectors' gradients through v = W0^T att ------------------------
  auto warp_sum = [&](int o) {
    float a = stage_all[0 * 2 * kStageBuf + o];
    a += stage_all[1 * 2 * kStageBuf + o];
    a += stage_all[2 * 2 * kStageBuf + o];
    a += stage_all[3 * 2 * kStageBuf + o];
    return a;
  };
  if (tid < 16) plain[PL_DV + tid] = warp_sum(kPartDvS + tid);         // dv_s[8] and dv_d[8] are contiguous
  __syncthreads();
  const float* dvs = plain + PL_DV;
  const float* dvd = plain + PL_DV + 8;
  float* out = p.partials + (long long)blockIdx.x * kPartialStride;
  for (int o = tid; o <= SWARM_W_COUNT; o += T) {
    float val;
    if (o < SWARM_W_ATT_SRC) {                                  // conv1.lin.weight[c][k] += att_s[c] dv_s[k] + att_d[c] dv_d[k]
      const int cc = o / 7, k = o - cc * 7;
      val = warp_sum(o) + plain[PL_ATT_S + cc] * dvs[k] + plain[PL_ATT_D + cc] * dvd[k];
    } else if (o < SWARM_W_CONV_BIAS) {                         // d att_src[c] = sum_k W0[c][k] dv_s[k]  (att_dst alike)
      const bool src = o < SWARM_W_ATT_DST;
      const int cc = o - (src ? SWARM_W_ATT_SRC : SWARM_W_ATT_DST);
      const float* dvv = src ? dvs : dvd;
      val = 0.0f;
#pragma unroll
      for (int k = 0; k < 7; ++k) val = fmaf(plain[PL_W0 + cc * 7 + k], dvv[k], val);
    } else {
      val = warp_sum(o);                                        // o == SWARM_W_COUNT: sum of squared TD errors
    }
    out[o] = val;
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, kDqnTmemCols);
}

int dqn_maxdeg(const SwarmConfig& c);

// the largest tile (floor(128 / N) transitions per CTA) that launch_dqn_grad_tc can ask for
int dqn_smem_bytes(const SwarmConfig& c) {
  return dqn_tc_layout(c.n_agents, c.knn_k, dqn_maxdeg(c), kTileThreads / c.n_agents, c.graph_mode).total;
}

cudaError_t launch_dqn_grad_tc(DqnParams& p, cudaStream_t stream) {
  const SwarmConfig& c = p.cfg;
  const int smem = dqn_tc_layout(c.n_agents, c.knn_k, p.maxdeg, p.epb, c.graph_mode).total;
  const int ctas = (p.n_graphs + p.epb - 1) / p.epb;
  cudaError_t err;
  if (c.graph_mode == SWARM_GRAPH_COMPLETE) {
    err = cudaFuncSetAttribute(dqn_grad_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    dqn_grad_tc_kernel<true><<<ctas, kTileThreads, smem, stream>>>(p);
  } else {
    err = cudaFuncSetAttribute(dqn_grad_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    dqn_grad_tc_kernel<false><<<ctas, kTileThreads, smem, stream>>>(p);
  }
  return cudaGetLastError();
}

}  // namespace swarm
