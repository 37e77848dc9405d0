// swarm_device.cuh -- device-side building blocks shared by every kernel of the swarm hot path.
//
// Rounding discipline (SURVEY.md A.5): the reference executes the world step as a chain of separately
// rounded float32 torch ops, with the 2-norm evaluated as sqrtf(fmaf(y, y, x*x)).  All physics / reward
// arithmetic below therefore uses the __f*_rn intrinsics (never contracted into FMAs by nvcc) in exactly
// that order, which makes positions, velocities, rewards, contact masks and kNN edge lists bit-identical
// to the CPU oracle whenever no contact force is active (the contact magnitude goes through
// logaddexp = log1p(exp(.)), whose CUDA and SLEEF implementations differ in the last ulp).
#ifndef SWARM_DEVICE_CUH
#define SWARM_DEVICE_CUH

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/swarm_b200.h"

namespace swarm {

// largest float q with sqrtf(q) <= dmin: makes a squared-distance test exactly equivalent to the reference's
// `vector_norm(delta) <= dmin` test on the rounded norm (host side)
inline float sq_threshold(float dmin) {
  if (!(dmin < 1e18f)) return INFINITY;
  float q = dmin * dmin;
  while (sqrtf(q) > dmin) q = nextafterf(q, 0.0f);
  while (sqrtf(nextafterf(q, INFINITY)) <= dmin) q = nextafterf(q, INFINITY);
  return q;
}

// the world step's constants, computed once on the host (world_consts)
struct WorldConsts {
  float one_minus_drag;
  float dmin_aa, dmin_ao;        // contact distances agent-agent / agent-obstacle (sum of radii, f32 add)
  float qmax_aa, qmax_ao;        // largest squared distance whose rounded sqrt is <= dmin (exact pre-filter)
};

inline WorldConsts world_consts(const SwarmConfig& c) {
  WorldConsts w;
  w.one_minus_drag = (float)(1.0 - (double)c.drag);
  w.dmin_aa = c.agent_radius + c.agent_radius;
  w.dmin_ao = c.landmark_radius + c.agent_radius;
  w.qmax_aa = sq_threshold(w.dmin_aa);
  w.qmax_ao = sq_threshold(w.dmin_ao);
  return w;
}

// parameter block of the stand-alone world-step kernels (step_kernels.cu, large_kernels.cu, grid_kernels.cu)
struct SimStepArgs {
  SwarmConfig cfg;
  const float4* state_in;
  const int32_t* actions;
  float4* state_out;
  float* rewards;                // optional outputs from here on
  uint8_t* flags;
  uint32_t* contact;
  float* obs;
  float2* dist;
  int32_t epb;                   // envs per block (step_kernels.cu)
  WorldConsts world;
  float* returns;                // += reward (large swarms)
  int32_t* hits;                 // += agents inside hit_distance (large swarms)
};

// ---- 2-norm exactly like torch.linalg.vector_norm over two floats -------------------------------
__device__ __forceinline__ float norm2(float x, float y) {
  return __fsqrt_rn(__fmaf_rn(y, y, __fmul_rn(x, x)));
}

// ---- torch CPU sum over a contiguous float row --------------------------------------------------------------------
// `x.mean(-1)` / `x.sum(-1)` over a contiguous row of m floats is NOT a left-to-right sum on the CPU: ATen's
// SumKernel.cpp (vectorized_inner_sum -> row_sum -> multi_row_sum) adds the row as 8-lane vectors, four vector
// accumulators interleaved over groups of four chunks, the chunks left over into accumulator 0, the accumulators into
// accumulator 0, and finally  0 + tail elements (k >= 8 * (m / 8)) + lane 0 + ... + lane 7; rows shorter than a vector
// use four interleaved scalar accumulators instead.  Only for m <= 4 and m = 8 is that a left-to-right sum; otherwise
// it differs in the last bit (observed on flocking_scenario.py:109-121 with 12 agents: 2 of 12
// shaping terms).  elem(k) yields element k; it is called exactly once per k.  (m < 16 * 32: no cascade levels.)
template <typename F>
__device__ __forceinline__ float torch_row_sum(int m, F elem) {
  if (m < 8) {
    // rows shorter than one vector take ATen's scalar path (scalar_inner_sum -> row_sum with four interleaved scalar
    // accumulators): p[k] = e[k] (k < 4), the rest into p[0], then p[0] + p[1] + p[2] + p[3]
    float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
    int k = 0;
    if (m >= 4) {
      p0 = elem(0); p1 = elem(1); p2 = elem(2); p3 = elem(3);
      k = 4;
    }
    for (; k < m; ++k) p0 = __fadd_rn(p0, elem(k));
    return __fadd_rn(__fadd_rn(__fadd_rn(p0, p1), p2), p3);
  }
  const int chunks = m >> 3, groups = chunks >> 2;
  float a0[8];
#pragma unroll
  for (int l = 0; l < 8; ++l) a0[l] = 0.0f;
  int c = 0;
  if (groups > 0) {
    float a1[8], a2[8], a3[8];
#pragma unroll
    for (int l = 0; l < 8; ++l) a1[l] = a2[l] = a3[l] = 0.0f;
    for (int gI = 0; gI < groups; ++gI, c += 4) {
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        a0[l] = __fadd_rn(a0[l], elem((c + 0) * 8 + l));
        a1[l] = __fadd_rn(a1[l], elem((c + 1) * 8 + l));
        a2[l] = __fadd_rn(a2[l], elem((c + 2) * 8 + l));
        a3[l] = __fadd_rn(a3[l], elem((c + 3) * 8 + l));
      }
    }
    for (; c < chunks; ++c) {
#pragma unroll
      for (int l = 0; l < 8; ++l) a0[l] = __fadd_rn(a0[l], elem(c * 8 + l));
    }
#pragma unroll
    for (int l = 0; l < 8; ++l) a0[l] = __fadd_rn(__fadd_rn(__fadd_rn(a0[l], a1[l]), a2[l]), a3[l]);
  } else {
    for (; c < chunks; ++c) {
#pragma unroll
      for (int l = 0; l < 8; ++l) a0[l] = __fadd_rn(a0[l], elem(c * 8 + l));
    }
  }
  float fin = 0.0f;
  for (int k = chunks * 8; k < m; ++k) fin = __fadd_rn(fin, elem(k));
#pragma unroll
  for (int l = 0; l < 8; ++l) fin = __fadd_rn(fin, a0[l]);
  return fin;
}

// The same row sum for rows of up to 8 191 non-negative elements, with the cascade of ATen's multi_row_sum that
// torch_row_sum leaves out.  multi_row_sum keeps four levels of the four vector accumulators, level_power =
// max(4, CeilLog2(groups) / 4) = 4 below 2^16 groups: after every 16th group of four chunks (512 floats) the level-0
// accumulators a0..a3 are added into the level-1 accumulators b0..b3 and cleared; after the last group the levels are
// added back into level 0, and row_sum goes on as torch_row_sum does (leftover chunks, accumulators, tail, lanes).
// Below 256 groups (m < 8 192) levels 2 and 3 stay zero, and so does level 1 below 16 groups: adding a zero changes no
// sum of non-negative elements, so those adds are left out.  Up to 17 groups (m < 576) the result equals
// torch_row_sum's, as float addition is commutative; from m = 576 on the two orders differ
// (tests/test_torch_sum_order_cascade.py).  elem(k) is called exactly once per k.
template <typename F>
__device__ __forceinline__ float torch_row_sum_cascade(int m, F elem) {
  if (m < 8) {
    float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
    int k = 0;
    if (m >= 4) {
      p0 = elem(0); p1 = elem(1); p2 = elem(2); p3 = elem(3);
      k = 4;
    }
    for (; k < m; ++k) p0 = __fadd_rn(p0, elem(k));
    return __fadd_rn(__fadd_rn(__fadd_rn(p0, p1), p2), p3);
  }
  const int chunks = m >> 3, groups = chunks >> 2;
  float a0[8], a1[8], a2[8], a3[8], b0[8], b1[8], b2[8], b3[8];
#pragma unroll
  for (int l = 0; l < 8; ++l) a0[l] = a1[l] = a2[l] = a3[l] = b0[l] = b1[l] = b2[l] = b3[l] = 0.0f;
  int c = 0;
  for (int gI = 0; gI < groups; ++gI, c += 4) {
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      a0[l] = __fadd_rn(a0[l], elem((c + 0) * 8 + l));
      a1[l] = __fadd_rn(a1[l], elem((c + 1) * 8 + l));
      a2[l] = __fadd_rn(a2[l], elem((c + 2) * 8 + l));
      a3[l] = __fadd_rn(a3[l], elem((c + 3) * 8 + l));
    }
    if ((gI & 15) == 15) {                                  // a full block of 16 groups: level 0 -> level 1
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        b0[l] = __fadd_rn(b0[l], a0[l]); a0[l] = 0.0f;
        b1[l] = __fadd_rn(b1[l], a1[l]); a1[l] = 0.0f;
        b2[l] = __fadd_rn(b2[l], a2[l]); a2[l] = 0.0f;
        b3[l] = __fadd_rn(b3[l], a3[l]); a3[l] = 0.0f;
      }
    }
  }
  if (groups >= 16) {                                       // level 1 -> level 0
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      a0[l] = __fadd_rn(a0[l], b0[l]);
      a1[l] = __fadd_rn(a1[l], b1[l]);
      a2[l] = __fadd_rn(a2[l], b2[l]);
      a3[l] = __fadd_rn(a3[l], b3[l]);
    }
  }
  for (; c < chunks; ++c) {
#pragma unroll
    for (int l = 0; l < 8; ++l) a0[l] = __fadd_rn(a0[l], elem(c * 8 + l));
  }
  if (groups > 0) {
#pragma unroll
    for (int l = 0; l < 8; ++l) a0[l] = __fadd_rn(__fadd_rn(__fadd_rn(a0[l], a1[l]), a2[l]), a3[l]);
  }
  float fin = 0.0f;
  for (int k = chunks * 8; k < m; ++k) fin = __fadd_rn(fin, elem(k));
#pragma unroll
  for (int l = 0; l < 8; ++l) fin = __fadd_rn(fin, a0[l]);
  return fin;
}

// Flocking's partner sweep of agent i at (px, py) (flocking_scenario.py:109-121,148-168): element k of the stacked
// distance list is partner j = k + (k >= i) -- the list comprehension skips the agent itself --
//   sum   = torch sum of (|p_i - p_j| - desired)^2 in torch's CPU row order (torch_row_sum, exact for N <= 128;
//           CASCADE = true: torch_row_sum_cascade, exact for N <= 4 096)
//   close = number of partners with world.get_distance <= min_collision_distance (centre distance minus both radii)
// pos(j) yields partner j's position.
template <bool CASCADE = false, typename P>
__device__ __forceinline__ void flocking_partner_sweep(float px, float py, int i, int N, P pos, float desired,
                                                       float radius, float min_collision_distance, float& sum,
                                                       int& close) {
  int cnt = 0;
  auto elem = [&](int k) -> float {
    const int j = k + (k >= i ? 1 : 0);
    const float2 q = pos(j);
    const float dx = __fsub_rn(px, q.x), dy = __fsub_rn(py, q.y);
    const float d = __fsqrt_rn(__fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    const float e = __fsub_rn(d, desired);
    const float gap = __fsub_rn(__fsub_rn(d, radius), radius);
    cnt += (gap <= min_collision_distance) ? 1 : 0;
    return __fmul_rn(e, e);
  };
  if constexpr (CASCADE)
    sum = torch_row_sum_cascade(N - 1, elem);
  else
    sum = torch_row_sum(N - 1, elem);
  close = cnt;
}

// ---- vmas Environment._set_action for discrete_action_nvec = [3, 3] -----------------------------
// flat a -> (a / 3, a % 3); index 0 -> 0, 1 -> -1, 2 -> +1
__device__ __forceinline__ float action_component(int idx) {
  return idx == 0 ? 0.0f : (idx == 1 ? -1.0f : 1.0f);
}
// Flat actions outside [0, 8] are a caller error (vmas raises; the Python seam asserts on them): every kernel treats
// them as action 0 (no force) and the replay ring stores 0, so no table or weight row is ever indexed out of range.
__device__ __forceinline__ int sanitize_action(int a) { return (unsigned)a > 8u ? 0 : a; }
__device__ __forceinline__ void decode_action(int a, float& ux, float& uy) {
  a = sanitize_action(a);
  ux = action_component(a / 3);
  uy = action_component(a % 3);
}

// ---- vmas World._get_constraint_forces, sphere-sphere, force on the entity at (ax, ay) ----------
// delta = a - b; dist_min = r_a + r_b; k = contact_margin
//   pen   = logaddexp(0, (dist_min - d) / k) * k
//   force = ((collision_force * delta) / (d > 0 ? d : 1e-8)) * pen; 0 if d < 1e-6 or d > dist_min
// Returns true when the pair passes vmas' collides() pre-filter (d <= dist_min), i.e. when the force
// (possibly zero) is added to the accumulator.
__device__ __forceinline__ bool contact_force(float ax, float ay, float bx, float by, float dist_min,
                                              float collision_force, float k, float& fx, float& fy) {
  const float dx = __fsub_rn(ax, bx);
  const float dy = __fsub_rn(ay, by);
  const float d = norm2(dx, dy);
  fx = 0.0f;
  fy = 0.0f;
  if (!(d <= dist_min)) return false;
  if (d < 1e-6f) return true;
  const float z = __fdiv_rn(__fsub_rn(dist_min, d), k);
  // torch.logaddexp(0, z) = max(0, z) + log1p(exp(-|0 - z|));  z >= 0 here
  const float pen = __fmul_rn(__fadd_rn(fmaxf(0.0f, z), log1pf(expf(-fabsf(z)))), k);
  const float dd = d > 0.0f ? d : 1e-8f;
  fx = __fmul_rn(__fdiv_rn(__fmul_rn(collision_force, dx), dd), pen);
  fy = __fmul_rn(__fdiv_rn(__fmul_rn(collision_force, dy), dd), pen);
  return true;
}

// ---- agent-agent contacts of one agent against the N agents of its env ---------------------------------
// `partners` = positions of the env's agents (float2 or float4 elements, .x/.y used), `self` = own index.
// Phase 1 is a branch-free sweep that records, 32 partners at a time, which squared distances pass the exact
// pre-filter q <= qmax (qmax = largest float whose rounded sqrt is <= r_a + r_b, see api.cu).  The difference is
// formed as partner - self with one packed add (sm_100 FADD2) against the negated own position: b - a = -(a - b)
// exactly under round-to-nearest, and only squares of the components are used.  Four partners share one shift: their
// hits are collected in a nibble of immediates first.  Phase 2 walks the set bits in ascending partner order and
// adds the contact forces in vmas' accumulation order; late in an episode, when the swarm has gathered at the goal,
// almost every warp has some lane in phase 2, so it has to stay proportional to the number of contacts.
__device__ __forceinline__ float2 xy_of(const float2& v) { return v; }
__device__ __forceinline__ float2 xy_of(const float4& v) { return *reinterpret_cast<const float2*>(&v); }

template <typename P>
__device__ __forceinline__ void agent_contacts(const P* __restrict__ partners, int N, int self, float sx, float sy,
                                               float qmax, float dist_min, float collision_force, float k, float& fx,
                                               float& fy, uint32_t& cmask) {
  const float2 neg = make_float2(-sx, -sy);
  auto hit = [&](int j) -> bool {
    const float2 d = __fadd2_rn(xy_of(partners[j]), neg);
    return __fmaf_rn(d.y, d.y, __fmul_rn(d.x, d.x)) <= qmax;
  };
  for (int base = 0; base < N; base += 32) {
    const int end = (N - base < 32) ? N : base + 32;
    uint32_t m = 0;
    int j = base;
    for (; j + 4 <= end; j += 4) {
      const uint32_t nib = (hit(j) ? 1u : 0u) | (hit(j + 1) ? 2u : 0u) | (hit(j + 2) ? 4u : 0u) | (hit(j + 3) ? 8u : 0u);
      m |= nib << (j - base);
    }
    for (; j < end; ++j) m |= (hit(j) ? 1u : 0u) << (j - base);
    if ((unsigned)(self - base) < 32u) m &= ~(1u << (self - base));
    while (m) {
      const int jj = __ffs(m) - 1;
      m &= m - 1;
      const float2 o = xy_of(partners[base + jj]);
      float gx, gy;
      if (contact_force(sx, sy, o.x, o.y, dist_min, collision_force, k, gx, gy)) {
        fx = __fadd_rn(fx, gx);
        fy = __fadd_rn(fy, gy);
        if (base + jj < 32) cmask |= (1u << (base + jj));
      }
    }
  }
}

// ---- vmas World._integrate_state (substeps = 1, mass = 1) ----------------------------------------
// accel = F / mass with mass = 1.0 is F itself (x / 1.0f == x exactly), so no division is issued.
__device__ __forceinline__ void integrate(float4& s, float fx, float fy, float dt, float one_minus_drag) {
  float vx = __fmul_rn(s.z, one_minus_drag);
  float vy = __fmul_rn(s.w, one_minus_drag);
  vx = __fadd_rn(vx, __fmul_rn(fx, dt));
  vy = __fadd_rn(vy, __fmul_rn(fy, dt));
  s.x = __fadd_rn(s.x, __fmul_rn(vx, dt));
  s.y = __fadd_rn(s.y, __fmul_rn(vy, dt));
  s.z = vx;
  s.w = vy;
}

// ---- scenario reward pieces ------------------------------------------------------------------------
// distance_to_goal_reward (go_to:117-122, oa:138-144): returns ||p - goal||
__device__ __forceinline__ float goal_distance(float x, float y, const SwarmConfig& c) {
  return norm2(__fsub_rn(x, c.goal_x), __fsub_rn(y, c.goal_y));
}
// world.get_distance(agent, obstacle): centre distance minus the two radii, one after the other
__device__ __forceinline__ float obstacle_distance(float x, float y, const SwarmConfig& c) {
  const float d = norm2(__fsub_rn(x, c.obstacle_x), __fsub_rn(y, c.obstacle_y));
  return __fsub_rn(__fsub_rn(d, c.agent_radius), c.landmark_radius);
}
// ObstacleAvoidanceScenario.reward (oa:135-152): -d_goal + w * (-(pen - d_obs) if d_obs <= pen else 0)
__device__ __forceinline__ float oa_reward(float d_goal, float d_obs, const SwarmConfig& c, uint8_t& flags) {
  float avoid = 0.0f;
  if (d_obs <= c.penalty_distance) {
    avoid = -__fsub_rn(c.penalty_distance, d_obs);
    flags |= SWARM_FLAG_PENALTY;
  }
  if (d_obs <= c.hit_distance) flags |= SWARM_FLAG_HIT;
  return __fadd_rn(-d_goal, __fmul_rn(c.obstacle_weight, avoid));
}

// ---- vmas World.step of one agent -----------------------------------------------------------------
// The ObstacleAvoidance landmark's contact force on the agent at s, behind the exact squared-distance pre-filter: added
// to (fx, fy), with the contact flag.
__device__ __forceinline__ void obstacle_contact(const float4& s, const SwarmConfig& c, const WorldConsts& w, float& fx,
                                                 float& fy, uint8_t& flags) {
  const float dx = __fsub_rn(s.x, c.obstacle_x), dy = __fsub_rn(s.y, c.obstacle_y);
  if (__fmaf_rn(dy, dy, __fmul_rn(dx, dx)) <= w.qmax_ao) {
    float gx, gy;
    if (contact_force(s.x, s.y, c.obstacle_x, c.obstacle_y, w.dmin_ao, c.collision_force, c.contact_margin, gx, gy)) {
      fx = __fadd_rn(fx, gx);
      fy = __fadd_rn(fy, gy);
      flags |= SWARM_FLAG_OBSTACLE_CONTACT;
    }
  }
}

// Force = decoded action u, + the obstacle's (oa: ObstacleAvoidance; pass a constant where there is one, so the branch
// folds), + the agents' in ascending partner order (`partners` = the env's positions, `self` = own index); then
// integration of s.
template <typename P>
__device__ __forceinline__ void agent_step(float4& s, float2 u, const P* __restrict__ partners, int N, int self, bool oa,
                                           const SwarmConfig& c, const WorldConsts& w, uint8_t& flags, uint32_t& cmask) {
  float fx = u.x, fy = u.y;
  if (oa) obstacle_contact(s, c, w, fx, fy, flags);
  agent_contacts(partners, N, self, s.x, s.y, w.qmax_aa, w.dmin_aa, c.collision_force, c.contact_margin, fx, fy, cmask);
  integrate(s, fx, fy, c.dt, w.one_minus_drag);
}

// scenario.reward(agent) on the post-step state s: d_goal, d_obs (0 for GoTo) and the ObstacleAvoidance reward with its
// flags (0 for GoTo, whose collective sum over the env's d_goal each caller adds from its own shared-memory layout)
__device__ __forceinline__ float post_step_reward(const float4& s, bool oa, const SwarmConfig& c, float& dgoal,
                                                  float& dobs, uint8_t& flags) {
  dgoal = goal_distance(s.x, s.y, c);
  dobs = 0.0f;
  if (!oa) return 0.0f;
  dobs = obstacle_distance(s.x, s.y, c);
  return oa_reward(dgoal, dobs, c, flags);
}

// the optional per-agent outputs of a stand-alone world step: observation [pos, vel, goal], (d_goal, d_obs), flags and
// agent-contact mask
__device__ __forceinline__ void store_step_outputs(const SimStepArgs& p, long long gidx, const float4& s, float dgoal,
                                                   float dobs, uint8_t flags, uint32_t cmask) {
  if (p.flags) p.flags[gidx] = flags;
  if (p.contact) p.contact[gidx] = cmask;
  if (p.obs) {
    float2* o = reinterpret_cast<float2*>(p.obs + gidx * 6);
    o[0] = make_float2(s.x, s.y);
    o[1] = make_float2(s.z, s.w);
    o[2] = make_float2(p.cfg.goal_x, p.cfg.goal_y);
  }
  if (p.dist) p.dist[gidx] = make_float2(dgoal, dobs);
}

// ---- generate_grid (go_to:52-80): offsets are Python doubles, cast to f32, added to the f32 centre ----
__device__ __forceinline__ float2 grid_position(float cx, float cy, int i, int cols, int rows, double spacing) {
  const int r = i / cols, q = i % cols;
  const double ox = ((double)q - (double)(cols - 1) / 2.0) * spacing;
  const double oy = ((double)r - (double)(rows - 1) / 2.0) * spacing;
  return make_float2(__fadd_rn(cx, (float)ox), __fadd_rn(cy, (float)oy));
}

}  // namespace swarm
#endif  // SWARM_DEVICE_CUH
