// grid_kernels.cu -- uniform-grid broad phase for large swarms (n_agents <= 4096; SURVEY 8(f) rank 4, BASELINE config
// "1024 agents x 1024 envs" with the radius / complete graph).
//
// One CTA owns one env.  Its agents are binned into square cells at least one graph radius wide (at most 64 x 64 cells
// over the env's bounding box), the (cell, agent) keys are sorted by a bitonic network in shared memory -- agents of a
// cell end up contiguous AND in ascending agent order, so every walk over the grid is deterministic -- and a node only
// ever looks at the 3 x 3 cells around its own.  Membership is decided by the exact test of the small-swarm radius
// graph (tile_device.cuh radius_hit: squared distance against the largest q whose rounded sqrt is <= r), the grid only
// prunes candidates.  On top of it:
//   radius_csr_kernel     the radius graph (batched_oracle.edges_radius: the complete builder of train_gcn_dqn.py:94-110
//                         filtered by distance) as a compact CSR grouped by target -- in-degrees, then sources in
//                         ascending order through a 9-way merge of the cell lists, which is exactly the order the edge
//                         list -> stable sort by target gives; feeds swarm_gatq_forward_csr (bit-faithful forward)
//   gatq_large_x_kernel   GCN.forward (train_gcn_dqn.py:59-70) + argmax for a large env on the radius graph with the
//                         attention in input space (see large_kernels.cu gatq_knn_large_x_kernel): no edge list at all
//   gatq_large_sorted_kernel  the same on the complete graph in O(N log N) -- the complete graph of 1 024 agents would
//                         be 1.07e9 edges per tick at C4.
#include <cstdlib>

#include "gatq_device.cuh"
#include "grid_device.cuh"
#include "launchers.h"

namespace swarm {

// ---- radius graph as CSR ----------------------------------------------------------------------------------------
struct RadiusCsrParams {
  SwarmConfig cfg;
  const float4* state;
  int32_t* degree;            // [B*N]   (count pass)
  const int32_t* row_ptr;     // [B*N+1] (fill pass)
  int32_t* src;               // [E]     (fill pass): global node ids b*N + j
  float qmax_r;
};

__host__ __device__ inline size_t radius_csr_smem_bytes(int N) {
  return (size_t)N * 8 + (size_t)grid_pow2(N) * 4 + (size_t)kGridCells * 4 + 64 * 4 + 64;
}

template <bool FILL>
__global__ void __launch_bounds__(kGridThreads) radius_csr_kernel(const __grid_constant__ RadiusCsrParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.cfg.n_agents, P = grid_pow2(N);
  float2* spos = reinterpret_cast<float2*>(smem_raw);
  uint32_t* keys = reinterpret_cast<uint32_t*>(spos + N);
  uint16_t* cbeg = reinterpret_cast<uint16_t*>(keys + P);
  uint16_t* cend = cbeg + kGridCells;
  float* sred = reinterpret_cast<float*>(cend + kGridCells);
  const long long env = blockIdx.x;
  for (int j = threadIdx.x; j < N; j += kGridThreads) {
    const float4 s = p.state[env * N + j];
    spos[j] = make_float2(s.x, s.y);
  }
  __syncthreads();
  const CellGrid g = grid_build([&](int j) { return spos[j]; }, N, P, p.cfg.graph_radius, keys, cbeg, cend, sred);
  const long long base = env * N;
  for (int i = threadIdx.x; i < N; i += kGridThreads) {
    const float2 pi = spos[i];
    const float2 neg = make_float2(-pi.x, -pi.y);
    const int cx = g.cx(pi.x), cy = g.cy(pi.y);
    if (!FILL) {
      int deg = (i == 0) ? 1 : 0;                           // the trailing (0 -> 0)
      for (int yy = max(cy - 1, 0); yy <= min(cy + 1, g.ny - 1); ++yy)
        for (int xx = max(cx - 1, 0); xx <= min(cx + 1, g.nx - 1); ++xx) {
          const int c = yy * g.nx + xx;
          for (int q = cbeg[c], e = cend[c]; q < e; ++q) {
            const int j = (int)(keys[q] & kIdxMask);
            deg += (j != i && grid_hit(spos[j], neg, p.qmax_r)) ? 1 : 0;
          }
        }
      p.degree[base + i] = deg;
    } else {
      // sources in ascending order: 9-way merge of the (ascending) cell lists
      int h[9], e[9];
      uint32_t v[9];
#pragma unroll
      for (int c9 = 0; c9 < 9; ++c9) {
        const int yy = cy - 1 + c9 / 3, xx = cx - 1 + c9 % 3;
        const bool ok = yy >= 0 && yy < g.ny && xx >= 0 && xx < g.nx;
        const int c = ok ? yy * g.nx + xx : 0;
        h[c9] = ok ? (int)cbeg[c] : 0;
        e[c9] = ok ? (int)cend[c] : 0;
        v[c9] = h[c9] < e[c9] ? (keys[h[c9]] & kIdxMask) : 0xFFFFu;
      }
      int32_t* out = p.src + p.row_ptr[base + i];
      int n = 0;
      while (true) {
        uint32_t m = v[0];
#pragma unroll
        for (int c9 = 1; c9 < 9; ++c9) m = min(m, v[c9]);
        if (m == 0xFFFFu) break;
#pragma unroll
        for (int c9 = 0; c9 < 9; ++c9) {
          if (v[c9] == m) {
            ++h[c9];
            v[c9] = h[c9] < e[c9] ? (keys[h[c9]] & kIdxMask) : 0xFFFFu;
          }
        }
        if ((int)m != i && grid_hit(spos[m], neg, p.qmax_r)) out[n++] = (int32_t)(base + m);
      }
      if (i == 0) out[n++] = (int32_t)base;
    }
  }
}

cudaError_t launch_radius_csr(const SwarmConfig& c, const float* state, int32_t* degree, const int32_t* row_ptr,
                              int32_t* src, cudaStream_t stream) {
  RadiusCsrParams p;
  p.cfg = c;
  p.state = reinterpret_cast<const float4*>(state);
  p.degree = degree;
  p.row_ptr = row_ptr;
  p.src = src;
  p.qmax_r = sq_threshold(c.graph_radius);
  const size_t smem = radius_csr_smem_bytes(c.n_agents);
  if (src) {
    cudaError_t err = cudaFuncSetAttribute(radius_csr_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    radius_csr_kernel<true><<<c.num_envs, kGridThreads, smem, stream>>>(p);
  } else {
    cudaError_t err = cudaFuncSetAttribute(radius_csr_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    radius_csr_kernel<false><<<c.num_envs, kGridThreads, smem, stream>>>(p);
  }
  return cudaGetLastError();
}

// ---- world step of a large env: contact partners from the grid ---------------------------------------------------
// vmas World.step for one env per CTA (large_kernels.cu sim_step_large_kernel sweeps all N partners per agent: 1 M pair
// tests per env at N = 1 024).  Agents in contact are at most dmin = 2 r apart, so with cells of that size the partners
// of an agent sit in its 3 x 3 cells; they are visited in ASCENDING agent order (9-way merge of the cell lists, as
// radius_csr_kernel does) because the reference adds the contact forces in entity order and float addition does not
// commute -- same pair test, same contact_force, same order as the full sweep, hence the same bits.  An agent whose
// neighbourhood holds more than kGridBruteAbove candidates (a collapsed swarm) falls back to the full sweep.
constexpr int kGridBruteAbove = 96;

__global__ void __launch_bounds__(kGridThreads) sim_step_grid_kernel(const __grid_constant__ SimStepArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_hits;
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, P = grid_pow2(N);
  float2* spos = reinterpret_cast<float2*>(smem_raw);
  uint32_t* keys = reinterpret_cast<uint32_t*>(spos + N);
  uint16_t* cbeg = reinterpret_cast<uint16_t*>(keys + P);
  uint16_t* cend = cbeg + kGridCells;
  float* sred = reinterpret_cast<float*>(cend + kGridCells);
  const long long env = blockIdx.x;
  const float4* env_state = p.state_in + env * N;
  if (threadIdx.x == 0) s_hits = 0;
  for (int j = threadIdx.x; j < N; j += kGridThreads) {
    const float4 s = env_state[j];
    spos[j] = make_float2(s.x, s.y);
  }
  __syncthreads();
  // every pre-step position is staged before any thread writes a post-step state: state_out may alias state_in
  const WorldConsts& w = p.world;
  const CellGrid g = grid_build([&](int j) { return spos[j]; }, N, P, w.dmin_aa, keys, cbeg, cend, sred);
  int my_hits = 0;
  const bool oa = c.scenario == SWARM_SCENARIO_OBSTACLE_AVOIDANCE;
  for (int i = threadIdx.x; i < N; i += kGridThreads) {
    const long long gidx = env * N + i;
    float4 s = env_state[i];               // only this thread ever writes index i
    float fx, fy;
    decode_action(p.actions[gidx], fx, fy);
    uint8_t flags = 0;
    if (oa) obstacle_contact(s, c, w, fx, fy, flags);
    {
      const float2 neg = make_float2(-s.x, -s.y);
      const int cx = g.cx(s.x), cy = g.cy(s.y);
      int h[9], e[9], cand = 0;
      uint32_t v[9];
#pragma unroll
      for (int c9 = 0; c9 < 9; ++c9) {
        const int yy = cy - 1 + c9 / 3, xx = cx - 1 + c9 % 3;
        const bool ok = yy >= 0 && yy < g.ny && xx >= 0 && xx < g.nx;
        const int cc = ok ? yy * g.nx + xx : 0;
        h[c9] = ok ? (int)cbeg[cc] : 0;
        e[c9] = ok ? (int)cend[cc] : 0;
        cand += e[c9] - h[c9];
        v[c9] = h[c9] < e[c9] ? (keys[h[c9]] & kIdxMask) : 0xFFFFu;
      }
      if (cand > kGridBruteAbove) {
        uint32_t cmask = 0;
        agent_contacts(spos, N, i, s.x, s.y, w.qmax_aa, w.dmin_aa, c.collision_force, c.contact_margin, fx, fy, cmask);
      } else {
        while (true) {
          uint32_t m = v[0];
#pragma unroll
          for (int c9 = 1; c9 < 9; ++c9) m = min(m, v[c9]);
          if (m == 0xFFFFu) break;
#pragma unroll
          for (int c9 = 0; c9 < 9; ++c9) {
            if (v[c9] == m) {
              ++h[c9];
              v[c9] = h[c9] < e[c9] ? (keys[h[c9]] & kIdxMask) : 0xFFFFu;
            }
          }
          const float2 o = spos[m];
          float gx, gy;
          if ((int)m != i && grid_hit(o, neg, w.qmax_aa)) {
            if (contact_force(s.x, s.y, o.x, o.y, w.dmin_aa, c.collision_force, c.contact_margin, gx, gy)) {
              fx = __fadd_rn(fx, gx);
              fy = __fadd_rn(fy, gy);
            }
          }
        }
      }
    }
    integrate(s, fx, fy, c.dt, w.one_minus_drag);
    float dgoal, dobs;
    const float reward = post_step_reward(s, oa, c, dgoal, dobs, flags);
    if (oa) {
      if (p.rewards) p.rewards[gidx] = reward;
      if (p.returns) p.returns[gidx] = __fadd_rn(p.returns[gidx], reward);
      my_hits += (flags & SWARM_FLAG_HIT) ? 1 : 0;
    }
    p.state_out[gidx] = s;
    store_step_outputs(p, gidx, s, dgoal, dobs, flags, 0u);     // no contact masks above 32 agents
  }
  if (p.hits) {
    if (my_hits) atomicAdd(&s_hits, my_hits);          // integer: order-independent
    __syncthreads();
    if (threadIdx.x == 0) p.hits[env] += s_hits;
  }
}

// default: from 512 agents on (measured: 256 agents x 4 096 envs 0.155 ms against 0.083 ms for the full sweep -- the sort
// does not pay yet; 1 024 x 1 024: 0.086 against 0.305 ms; 4 096 x 256: 0.090 against 1.44 ms); SWARM_STEP_GRID=0 / 1 forces
bool sim_step_grid_enabled(int n_agents) {
  const char* e = std::getenv("SWARM_STEP_GRID");
  if (e && e[0] == '0') return false;
  if (e && e[0] == '1') return true;
  return n_agents >= 512;
}

cudaError_t launch_sim_step_grid(const SimStepArgs& p, cudaStream_t stream) {
  const SwarmConfig& c = p.cfg;
  const size_t smem = radius_csr_smem_bytes(c.n_agents);
  cudaError_t err = cudaFuncSetAttribute(sim_step_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  sim_step_grid_kernel<<<c.num_envs, kGridThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

// ---- Q forward with the attention in input space, radius / complete graph -----------------------------------------
struct LargeXParams {
  SwarmConfig cfg;
  const float4* state;
  const float* weights;
  float* q_out;              // [B*N][9] or nullptr
  int32_t* act_out;          // [B*N] or nullptr
  float qmax_r;
};

__host__ __device__ inline size_t large_x_smem_bytes(int N) {
  size_t b = (size_t)((TW_COUNT + 3) & ~3) * 4 + 64;        // weights, v_s / v_d
  b += (size_t)N * 16 + (size_t)N * 4;                       // states, alpha_src
  b += 64 * 4;                                               // reduction scratch
  b += (size_t)grid_pow2(N) * 4 + (size_t)kGridCells * 4;    // grid keys, cell ranges
  return b + 64;
}

__global__ void __launch_bounds__(kGridThreads, 2) gatq_large_x_kernel(const __grid_constant__ LargeXParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, P = grid_pow2(N);
  const int tid = threadIdx.x;
  const long long env = blockIdx.x;
  float* sw = reinterpret_cast<float*>(smem_raw);
  float* sv = sw + ((TW_COUNT + 3) & ~3);                 // v_s[8], v_d[8]
  float4* sst = reinterpret_cast<float4*>(sv + 16);
  float* sas = reinterpret_cast<float*>(sst + N);
  float* sred = sas + N;                                  // [64]
  uint32_t* keys = reinterpret_cast<uint32_t*>(sred + 64);
  uint16_t* cbeg = reinterpret_cast<uint16_t*>(keys + P);
  uint16_t* cend = cbeg + kGridCells;

  stage_weights(p.weights, sw, tid, kGridThreads);
  for (int i = tid; i < N; i += kGridThreads) sst[i] = p.state[env * N + i];
  __syncthreads();
  if (tid < 16) {
    // attention vectors pulled through the projection: v[k] = sum_c att[c] W0[c][k]
    const int k = tid & 7;
    const float* att = sw + (tid < 8 ? TW_ATT_S : TW_ATT_D);
    float v = 0.0f;
    if (k < 7)
      for (int cc = 0; cc < 32; ++cc) v = fmaf(att[cc], sw[TW_W0T + k * 32 + cc], v);
    sv[tid] = v;
  }
  const CellGrid g = grid_build([&](int j) { const float4 s = sst[j]; return make_float2(s.x, s.y); }, N, P,
                                c.graph_radius, keys, cbeg, cend, sred);
  __syncthreads();
  for (int i = tid; i < N; i += kGridThreads) {
    const float4 st = sst[i];
    sas[i] = fmaf(st.x, sv[0], fmaf(st.y, sv[1], fmaf(st.z, sv[2], fmaf(st.w, sv[3],
             fmaf(c.goal_x, sv[4], fmaf(c.goal_y, sv[5], (float)i * sv[6]))))));
  }
  __syncthreads();

  for (int i = tid; i < N; i += kGridThreads) {
    const float4 st = sst[i];
    const float adst = fmaf(st.x, sv[8], fmaf(st.y, sv[9], fmaf(st.z, sv[10], fmaf(st.w, sv[11],
                       fmaf(c.goal_x, sv[12], fmaf(c.goal_y, sv[13], (float)i * sv[14]))))));
    // in-edges: agents j != i within the radius (train:94-110 filtered by distance) + the trailing (0,0) of node 0
    const float2 neg = make_float2(-st.x, -st.y);
    const int cx = g.cx(st.x), cy = g.cy(st.y);
    const int y0 = max(cy - 1, 0), y1 = min(cy + 1, g.ny - 1), x0 = max(cx - 1, 0), x1 = min(cx + 1, g.nx - 1);
    float amax = (i == 0) ? sas[0] : -INFINITY;
    for (int yy = y0; yy <= y1; ++yy)
      for (int xx = x0; xx <= x1; ++xx) {
        const int cc = yy * g.nx + xx;
        for (int q = cbeg[cc], e = cend[cc]; q < e; ++q) {
          const int j = (int)(keys[q] & kIdxMask);
          const float4 sj = sst[j];
          if (j != i && grid_hit(make_float2(sj.x, sj.y), neg, p.qmax_r)) amax = fmaxf(amax, sas[j]);
        }
      }
    const float m = gat_logit(amax, adst);                // LeakyReLU and the rounded add are monotone
    float den = 0.0f, acc_id = 0.0f;
    float2 acc_p = make_float2(0.f, 0.f), acc_v = make_float2(0.f, 0.f);
    auto add = [&](int j) {
      const float4 sj = sst[j];
      const float w = __expf(gat_logit(sas[j], adst) - m);
      den = __fadd_rn(den, w);
      acc_p = __ffma2_rn(make_float2(w, w), make_float2(sj.x, sj.y), acc_p);
      acc_v = __ffma2_rn(make_float2(w, w), make_float2(sj.z, sj.w), acc_v);
      acc_id = fmaf(w, (float)j, acc_id);
    };
    for (int yy = y0; yy <= y1; ++yy)
      for (int xx = x0; xx <= x1; ++xx) {
        const int cc = yy * g.nx + xx;
        for (int q = cbeg[cc], e = cend[cc]; q < e; ++q) {
          const int j = (int)(keys[q] & kIdxMask);
          const float4 sj = sst[j];
          if (j != i && grid_hit(make_float2(sj.x, sj.y), neg, p.qmax_r)) add(j);
        }
      }
    if (i == 0) add(0);
    const float inv = 1.0f / __fadd_rn(den, 1e-16f);
    const float wsum = den * inv;
    const float xm[7] = {acc_p.x * inv, acc_p.y * inv, acc_v.x * inv, acc_v.y * inv, c.goal_x * wsum, c.goal_y * wsum,
                         acc_id * inv};
    // agg = W0 xm (the projection of gat_project without its attention terms), then the head
    float a1[32];
#pragma unroll
    for (int cc = 0; cc < 32; ++cc) a1[cc] = 0.0f;
    const float4* w0 = reinterpret_cast<const float4*>(sw + TW_W0T);
#pragma unroll
    for (int k = 0; k < 7; ++k) {
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        fma4_packed(xm[k], w0[k * 8 + c4], a1[4 * c4 + 0], a1[4 * c4 + 1], a1[4 * c4 + 2], a1[4 * c4 + 3]);
      }
    }
    float q[9];
    const int action = gat_head_fast(a1, sw, q);
    const long long gi = env * N + i;
    if (p.q_out) {
#pragma unroll
      for (int a = 0; a < 9; ++a) p.q_out[gi * 9 + a] = q[a];
    }
    if (p.act_out) p.act_out[gi] = action;
  }
}

// ---- complete graph in O(N log N) ---------------------------------------------------------------------------------
// On the complete graph (train:94-110) the attention logit of edge (j -> i) is LeakyReLU(a_j + d_i) with a = alpha_src,
// d = alpha_dst: for a fixed target the sources split by the SIGN of a_j + d_i, i.e. -- with the sources sorted by a --
// into a prefix (slope 0.2) and a suffix (slope 1), and inside each part the weight factorises:
//     exp(a_j + d_i - m_i)       = exp(d_i + A - m_i)           * exp(a_j - A)             (suffix, a_j > -d_i)
//     exp(0.2 (a_j + d_i) - m_i) = exp(0.2 (d_i + A) - m_i)     * exp(0.2 (a_j - A))       (prefix)
// with A = the env's largest a and m_i the softmax shift (largest logit of the row).  So one sort of the env's a values,
// one suffix scan and one prefix scan of the six weighted quantities (1, x, y, vx, vy, id), and per target a binary
// search, two scan look-ups, and the removal of its own term (no self loop except node 0's (0, 0)).  Everything that is
// added is positive and the two factors are <= 1 (m_i = LeakyReLU(A + d_i) is the row's largest logit), so there is no
// overflow and no cancellation -- except for the ONE node that holds A itself (its row's largest logit comes from the
// second largest a): that node sums its row directly.  1 M pair evaluations per env at N = 1 024 become ~20 k operations.
// Same mathematics as the bit-faithful CSR forward (swarm_gatq_forward_csr), float32-level different rounding (tests: Q
// within 1e-5).
struct SortedScan {
  float v[6];
};

__host__ __device__ inline size_t large_sorted_smem_bytes(int N) {
  size_t b = (size_t)((TW_COUNT + 3) & ~3) * 4 + 64;        // weights, v_s / v_d
  b += (size_t)N * 16 + (size_t)N * 4 * 2;                   // states, alpha_src, alpha_dst
  b += 64 * 4;                                               // reduction scratch
  b += (size_t)grid_pow2(N) * 4 + (size_t)grid_pow2(N) * 2;  // sort keys, permutation
  b += (size_t)N * 4;                                        // sorted a
  b += (size_t)((N >> 2) + 2) * 6 * 4 * 2;                   // prefix / suffix scans of six quantities, every 4th position
  b += 32 * 6 * 4 * 2;                                       // warp totals of the scans
  return b + 128;
}

__global__ void __launch_bounds__(kGridThreads, 2) gatq_large_sorted_kernel(const __grid_constant__ LargeXParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const SwarmConfig& c = p.cfg;
  const int N = c.n_agents, P = grid_pow2(N);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kGridThreads / 32;
  const long long env = blockIdx.x;
  float* sw = reinterpret_cast<float*>(smem_raw);
  float* sv = sw + ((TW_COUNT + 3) & ~3);                 // v_s[8], v_d[8]
  float4* sst = reinterpret_cast<float4*>(sv + 16);
  float* sas = reinterpret_cast<float*>(sst + N);
  float* sad = sas + N;
  float* sred = sad + N;                                  // [64]
  uint32_t* keys = reinterpret_cast<uint32_t*>(sred + 64);
  float* sa_sorted = reinterpret_cast<float*>(keys + P);
  // scans are kept at every FOURTH sorted position (12 B per agent instead of 48: envs of 4 096 agents fit); a look-up
  // adds the at most three elements between the stored position and the one asked for
  const int NC = (N >> 2) + 2;
  float* pre = sa_sorted + N;                             // [NC][6]  pre[c] = sum over positions <  4 c, slope-0.2 weights
  float* suf = pre + (size_t)NC * 6;                      // [NC][6]  suf[c] = sum over positions >= 4 c, slope-1 weights
  float* wtot = suf + (size_t)NC * 6;                     // [2][kWarps][6]
  uint16_t* perm = reinterpret_cast<uint16_t*>(wtot + 2 * 32 * 6);

  stage_weights(p.weights, sw, tid, kGridThreads);
  for (int i = tid; i < N; i += kGridThreads) sst[i] = p.state[env * N + i];
  __syncthreads();
  if (tid < 16) {
    const int k = tid & 7;
    const float* att = sw + (tid < 8 ? TW_ATT_S : TW_ATT_D);
    float v = 0.0f;
    if (k < 7)
      for (int cc = 0; cc < 32; ++cc) v = fmaf(att[cc], sw[TW_W0T + k * 32 + cc], v);
    sv[tid] = v;
  }
  __syncthreads();
  // alpha terms, sort keys, the two largest alpha_src
  float t1 = -INFINITY, t2 = -INFINITY;
  int t1i = -1;
  for (int i = tid; i < P; i += kGridThreads) {
    uint32_t key = 0xFFFFFFFFu;
    if (i < N) {
      const float4 st = sst[i];
      const float a = fmaf(st.x, sv[0], fmaf(st.y, sv[1], fmaf(st.z, sv[2], fmaf(st.w, sv[3],
                      fmaf(c.goal_x, sv[4], fmaf(c.goal_y, sv[5], (float)i * sv[6]))))));
      const float d = fmaf(st.x, sv[8], fmaf(st.y, sv[9], fmaf(st.z, sv[10], fmaf(st.w, sv[11],
                      fmaf(c.goal_x, sv[12], fmaf(c.goal_y, sv[13], (float)i * sv[14]))))));
      sas[i] = a;
      sad[i] = d;
      key = float_order_key(a);
      if (key == 0xFFFFFFFFu) key = 0xFFFFFFFEu;            // padding stays last
      if (a > t1) { t2 = t1; t1 = a; t1i = i; }
      else if (a > t2) t2 = a;
    }
    keys[i] = key;
    perm[i] = (uint16_t)(i < N ? i : 0);
  }
  {
    auto merge = [&](float o1, int oi, float o2) {
      if (o1 > t1) { t2 = fmaxf(t1, o2); t1 = o1; t1i = oi; }
      else t2 = fmaxf(t2, o1);
    };
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) {
      const float o1 = __shfl_xor_sync(0xffffffffu, t1, sh), o2 = __shfl_xor_sync(0xffffffffu, t2, sh);
      const int oi = __shfl_xor_sync(0xffffffffu, t1i, sh);
      merge(o1, oi, o2);
    }
    if (lane == 0) {
      sred[warp * 3 + 0] = t1;
      sred[warp * 3 + 1] = __int_as_float(t1i);
      sred[warp * 3 + 2] = t2;
    }
    __syncthreads();
    t1 = -INFINITY; t2 = -INFINITY; t1i = -1;
    for (int w = 0; w < kWarps; ++w) merge(sred[w * 3 + 0], __float_as_int(sred[w * 3 + 1]), sred[w * 3 + 2]);
  }
  const float A = t1;
  // bitonic sort of (key, index) pairs (see grid_build for the barrier scheme)
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < (P >> 1); t += kGridThreads) {
        const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int hi = lo | j;
        const bool up = (lo & k) == 0;
        const uint32_t ka = keys[lo], kb = keys[hi];
        if ((ka > kb) == up) {
          keys[lo] = kb; keys[hi] = ka;
          const uint16_t pa = perm[lo];
          perm[lo] = perm[hi]; perm[hi] = pa;
        }
      }
      const int jn = (j > 1) ? (j >> 1) : k;
      if (j > 32 || jn > 32) __syncthreads(); else __syncwarp();
    }
  }
  __syncthreads();
  // scans over the sorted order: thread t owns the contiguous positions [t * per, (t + 1) * per)
  const int per = (N + kGridThreads - 1) / kGridThreads;
  const int p0 = tid * per;
  {
    SortedScan lp, ls;                                      // this thread's chunk totals: prefix weights, suffix weights
#pragma unroll
    for (int q = 0; q < 6; ++q) { lp.v[q] = 0.0f; ls.v[q] = 0.0f; }
    for (int k = 0; k < per; ++k) {
      const int pp = p0 + k;
      if (pp < N) {
        const int j = perm[pp];
        const float a = sas[j];
        sa_sorted[pp] = a;
        const float4 sj = sst[j];
        const float e2 = __expf(0.2f * (a - A)), e1 = __expf(a - A);
        const float qv[6] = {1.0f, sj.x, sj.y, sj.z, sj.w, (float)j};
#pragma unroll
        for (int q = 0; q < 6; ++q) { lp.v[q] = fmaf(e2, qv[q], lp.v[q]); ls.v[q] = fmaf(e1, qv[q], ls.v[q]); }
      }
    }
    // inclusive warp scans: prefix ascending in tid, suffix descending in tid
    SortedScan ip = lp, is = ls;
#pragma unroll
    for (int sh = 1; sh < 32; sh <<= 1) {
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        const float up = __shfl_up_sync(0xffffffffu, ip.v[q], sh);
        const float dn = __shfl_down_sync(0xffffffffu, is.v[q], sh);
        if (lane >= sh) ip.v[q] += up;
        if (lane + sh < 32) is.v[q] += dn;
      }
    }
    if (lane == 31)
#pragma unroll
      for (int q = 0; q < 6; ++q) wtot[(0 * 32 + warp) * 6 + q] = ip.v[q];
    if (lane == 0)
#pragma unroll
      for (int q = 0; q < 6; ++q) wtot[(1 * 32 + warp) * 6 + q] = is.v[q];
    __syncthreads();
    SortedScan bp, bs;                                      // totals of the warps before / after this one
#pragma unroll
    for (int q = 0; q < 6; ++q) { bp.v[q] = 0.0f; bs.v[q] = 0.0f; }
    for (int w = 0; w < warp; ++w)
#pragma unroll
      for (int q = 0; q < 6; ++q) bp.v[q] += wtot[(0 * 32 + w) * 6 + q];
    for (int w = kWarps - 1; w > warp; --w)
#pragma unroll
      for (int q = 0; q < 6; ++q) bs.v[q] += wtot[(1 * 32 + w) * 6 + q];
    // exclusive prefix at the chunk start / suffix just after the chunk end (the neighbour lane's inclusive value: no
    // subtraction), then walk the chunk
    SortedScan runp, runs;
#pragma unroll
    for (int q = 0; q < 6; ++q) {
      const float upx = __shfl_up_sync(0xffffffffu, ip.v[q], 1);
      const float dnx = __shfl_down_sync(0xffffffffu, is.v[q], 1);
      runp.v[q] = bp.v[q] + (lane > 0 ? upx : 0.0f);
      runs.v[q] = bs.v[q] + (lane < 31 ? dnx : 0.0f);
    }
    // prefix: ascending walk writes pre[pp] = sum over positions < pp
    for (int k = 0; k < per; ++k) {
      const int pp = p0 + k;
      if (pp < N) {
        if ((pp & 3) == 0) {
#pragma unroll
          for (int q = 0; q < 6; ++q) pre[(size_t)(pp >> 2) * 6 + q] = runp.v[q];
        }
        const int j = perm[pp];
        const float a = sas[j];
        const float4 sj = sst[j];
        const float e2 = __expf(0.2f * (a - A));
        const float qv[6] = {1.0f, sj.x, sj.y, sj.z, sj.w, (float)j};
#pragma unroll
        for (int q = 0; q < 6; ++q) runp.v[q] = fmaf(e2, qv[q], runp.v[q]);
      }
    }
    if ((N & 3) == 0 && p0 <= N - 1 && N - 1 < p0 + per) {  // the owner of the last position: the total at position N
#pragma unroll
      for (int q = 0; q < 6; ++q) pre[(size_t)(N >> 2) * 6 + q] = runp.v[q];
    }
    // suffix: descending walk writes suf[pp] = sum over positions >= pp
    for (int k = per - 1; k >= 0; --k) {
      const int pp = p0 + k;
      if (pp < N) {
        const int j = perm[pp];
        const float a = sas[j];
        const float4 sj = sst[j];
        const float e1 = __expf(a - A);
        const float qv[6] = {1.0f, sj.x, sj.y, sj.z, sj.w, (float)j};
#pragma unroll
        for (int q = 0; q < 6; ++q) runs.v[q] = fmaf(e1, qv[q], runs.v[q]);
        if ((pp & 3) == 0) {
#pragma unroll
          for (int q = 0; q < 6; ++q) suf[(size_t)(pp >> 2) * 6 + q] = runs.v[q];
        }
      }
    }
    if (tid == 0) {                                         // positions >= 4 ceil(N / 4): nothing
#pragma unroll
      for (int q = 0; q < 6; ++q) suf[(size_t)((N + 3) >> 2) * 6 + q] = 0.0f;
    }
  }
  if (warp == 0 && t1i > 0) {
    // direct row of the holder of the largest alpha_src, 32 lanes over the sources (fixed lane order: deterministic)
    const float adst = sad[t1i];
    const float m = gat_logit(t2, adst);
    float ds[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) ds[q] = 0.0f;
    for (int j = lane; j < N; j += 32) {
      if (j == t1i) continue;
      const float4 sj = sst[j];
      const float w = __expf(gat_logit(sas[j], adst) - m);
      ds[0] += w;
      ds[1] = fmaf(w, sj.x, ds[1]); ds[2] = fmaf(w, sj.y, ds[2]);
      ds[3] = fmaf(w, sj.z, ds[3]); ds[4] = fmaf(w, sj.w, ds[4]);
      ds[5] = fmaf(w, (float)j, ds[5]);
    }
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1)
#pragma unroll
      for (int q = 0; q < 6; ++q) ds[q] += __shfl_xor_sync(0xffffffffu, ds[q], sh);
    if (lane == 0)
#pragma unroll
      for (int q = 0; q < 6; ++q) sred[48 + q] = ds[q];
  }
  __syncthreads();

  for (int i = tid; i < N; i += kGridThreads) {
    const float4 st = sst[i];
    const float adst = sad[i], ai = sas[i];
    float sum[6];
    if (i == t1i && i != 0) {
      // the holder of the largest alpha_src: its row's largest logit comes from the second largest.  Its row was summed
      // directly by warp 0 (below the scans): pick the sums up
#pragma unroll
      for (int q = 0; q < 6; ++q) sum[q] = sred[48 + q];
    } else {
      const float zA = A + adst;
      const float m = zA > 0.0f ? zA : 0.2f * zA;             // the row's largest logit (node 0 keeps its own source)
      // split position: number of sorted a values <= -adst (their logits take the 0.2 slope)
      int lo = 0, hi = N;
      const float thr = -adst;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sa_sorted[mid] <= thr) lo = mid + 1; else hi = mid;
      }
      const float c1 = __expf(zA - m), c2 = __expf(0.2f * zA - m);
      // prefix over positions < lo = stored prefix at 4 floor(lo / 4) + the positions up to lo - 1;
      // suffix over positions >= lo = stored suffix at 4 ceil(lo / 4) + the positions from lo up to it
      float ps[6], ss[6];
      const int cp = lo >> 2, cs = (lo + 3) >> 2;
#pragma unroll
      for (int q = 0; q < 6; ++q) { ps[q] = pre[(size_t)cp * 6 + q]; ss[q] = suf[(size_t)cs * 6 + q]; }
      for (int pp = cp << 2; pp < lo; ++pp) {
        const int j = perm[pp];
        const float4 sj = sst[j];
        const float e2 = __expf(0.2f * (sa_sorted[pp] - A));
        ps[0] += e2;
        ps[1] = fmaf(e2, sj.x, ps[1]); ps[2] = fmaf(e2, sj.y, ps[2]);
        ps[3] = fmaf(e2, sj.z, ps[3]); ps[4] = fmaf(e2, sj.w, ps[4]);
        ps[5] = fmaf(e2, (float)j, ps[5]);
      }
      const int top = min(cs << 2, N);
      for (int pp = top - 1; pp >= lo; --pp) {
        const int j = perm[pp];
        const float4 sj = sst[j];
        const float e1 = __expf(sa_sorted[pp] - A);
        ss[0] += e1;
        ss[1] = fmaf(e1, sj.x, ss[1]); ss[2] = fmaf(e1, sj.y, ss[2]);
        ss[3] = fmaf(e1, sj.z, ss[3]); ss[4] = fmaf(e1, sj.w, ss[4]);
        ss[5] = fmaf(e1, (float)j, ss[5]);
      }
#pragma unroll
      for (int q = 0; q < 6; ++q) sum[q] = fmaf(c1, ss[q], c2 * ps[q]);
      if (i != 0) {
        const float wown = __expf(gat_logit(ai, adst) - m);
        sum[0] -= wown;
        sum[1] = fmaf(-wown, st.x, sum[1]); sum[2] = fmaf(-wown, st.y, sum[2]);
        sum[3] = fmaf(-wown, st.z, sum[3]); sum[4] = fmaf(-wown, st.w, sum[4]);
        sum[5] = fmaf(-wown, (float)i, sum[5]);
      }
    }
    const float den = sum[0];
    const float inv = 1.0f / __fadd_rn(den, 1e-16f);
    const float wsum = den * inv;
    const float xm[7] = {sum[1] * inv, sum[2] * inv, sum[3] * inv, sum[4] * inv, c.goal_x * wsum, c.goal_y * wsum,
                         sum[5] * inv};
    float a1[32];
#pragma unroll
    for (int cc = 0; cc < 32; ++cc) a1[cc] = 0.0f;
    const float4* w0 = reinterpret_cast<const float4*>(sw + TW_W0T);
#pragma unroll
    for (int k = 0; k < 7; ++k) {
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4)
        fma4_packed(xm[k], w0[k * 8 + c4], a1[4 * c4 + 0], a1[4 * c4 + 1], a1[4 * c4 + 2], a1[4 * c4 + 3]);
    }
    float q[9];
    const int action = gat_head_fast(a1, sw, q);
    const long long gi = env * N + i;
    if (p.q_out) {
#pragma unroll
      for (int a = 0; a < 9; ++a) p.q_out[gi * 9 + a] = q[a];
    }
    if (p.act_out) p.act_out[gi] = action;
  }
}

bool gatq_large_x_fits(int N, bool radius) {
  return N <= (1 << kIdxBits) && (radius ? large_x_smem_bytes(N) : large_sorted_smem_bytes(N)) <= 227 * 1024;
}

cudaError_t launch_gatq_large_x(const SwarmConfig& c, const float* weights, const float* state, float* q, int32_t* actions,
                                cudaStream_t stream) {
  LargeXParams p;
  p.cfg = c;
  p.state = reinterpret_cast<const float4*>(state);
  p.weights = weights;
  p.q_out = q;
  p.act_out = actions;
  const bool radius = c.graph_mode == SWARM_GRAPH_RADIUS;
  p.qmax_r = radius ? sq_threshold(c.graph_radius) : 0.0f;
  if (radius) {
    const size_t smem = large_x_smem_bytes(c.n_agents);
    cudaError_t err = cudaFuncSetAttribute(gatq_large_x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    gatq_large_x_kernel<<<c.num_envs, kGridThreads, smem, stream>>>(p);
  } else {
    // complete graph in O(N log N): sorted sources, prefix / suffix scans
    const size_t smem = large_sorted_smem_bytes(c.n_agents);
    cudaError_t err = cudaFuncSetAttribute(gatq_large_sorted_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    gatq_large_sorted_kernel<<<c.num_envs, kGridThreads, smem, stream>>>(p);
  }
  return cudaGetLastError();
}

}  // namespace swarm
