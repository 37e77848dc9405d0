// api.cu -- extern "C" entry points of libswarm_b200.so (see include/swarm_b200.h).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "launchers.h"
#include "tile_kernels.cuh"

namespace swarm {
namespace {
thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return SWARM_OK;
  return fail(SWARM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

constexpr int kMaxLargeAgents = 4096;

int validate(const SwarmConfig* cfg, bool need_graph, bool allow_large = false) {
  if (!cfg) return fail(SWARM_ERR_INVALID_ARG, "cfg is NULL");
  if (cfg->num_envs <= 0) return fail(SWARM_ERR_INVALID_ARG, "num_envs must be positive");
  if (cfg->n_agents <= 0) return fail(SWARM_ERR_INVALID_ARG, "n_agents must be positive");
  if (cfg->scenario != SWARM_SCENARIO_GOTO && cfg->scenario != SWARM_SCENARIO_OBSTACLE_AVOIDANCE)
    return fail(SWARM_ERR_INVALID_ARG, "unknown scenario id");
  if (cfg->n_agents > kTileThreads && !allow_large)
    return fail(SWARM_ERR_UNSUPPORTED, "n_agents > 128 is not supported by the fused env-tile kernels (use swarm_sim_step / "
                                       "swarm_graph_build / swarm_gatq_forward_csr for large swarms)");
  if (cfg->n_agents > kMaxLargeAgents) return fail(SWARM_ERR_UNSUPPORTED, "n_agents > 4096");
  if (need_graph) {
    if (cfg->graph_mode != SWARM_GRAPH_COMPLETE && cfg->graph_mode != SWARM_GRAPH_KNN &&
        cfg->graph_mode != SWARM_GRAPH_RADIUS)
      return fail(SWARM_ERR_INVALID_ARG, "unknown graph mode");
    if (cfg->graph_mode == SWARM_GRAPH_RADIUS) {
      if (!(cfg->graph_radius >= 0.0f)) return fail(SWARM_ERR_INVALID_ARG, "graph_radius must be >= 0");
      if (cfg->n_agents > kTileThreads && !allow_large)
        return fail(SWARM_ERR_UNSUPPORTED, "the padded radius edge block is implemented for n_agents <= 128 (large swarms: "
                                           "swarm_graph_build_radius_csr / swarm_gatq_forward_large / swarm_rollout_large)");
    }
    if (cfg->graph_mode == SWARM_GRAPH_KNN) {
      // torch.topk raises "selected index k out of range" for k > n (simulator.py:19 with n_agents < 10)
      if (cfg->knn_k <= 0 || cfg->knn_k > cfg->n_agents)
        return fail(SWARM_ERR_INVALID_ARG, "selected index k out of range");
    }
  }
  return SWARM_OK;
}

// above 128 agents the kNN table comes from torch.topk's partial_sort branch, the only one implemented
int validate_large_knn(const SwarmConfig& c) {
  if (c.graph_mode == SWARM_GRAPH_KNN && c.n_agents > kTileThreads && (int64_t)c.knn_k * 64 > c.n_agents)
    return fail(SWARM_ERR_UNSUPPORTED,
                "large-swarm kNN implements torch.topk's partial_sort branch only (needs 64 * k <= n_agents)");
  return SWARM_OK;
}

// what: "replay ring" or "batch"; need_capacity: the call writes into the ring
int validate_ring(const SwarmReplay* r, const char* what, bool need_capacity) {
  if (!r || !r->state || !r->next_state || !r->actions || !r->rewards || (need_capacity && r->capacity <= 0))
    return fail(SWARM_ERR_INVALID_ARG,
                std::string(what) + (need_capacity ? " has NULL arrays or no capacity" : " has NULL arrays"));
  return SWARM_OK;
}

// torch.optim.Adam's ValueError checks
int validate_adam(double lr, double beta1, double beta2, double eps) {
  if (!(lr >= 0.0) || !(beta1 >= 0.0 && beta1 < 1.0) || !(beta2 >= 0.0 && beta2 < 1.0) || !(eps >= 0.0))
    return fail(SWARM_ERR_INVALID_ARG, "invalid Adam hyper-parameter");
  return SWARM_OK;
}

// the Flocking / Cohesion rewards of a rollout tick on cfg's world; same_shape: the spec must cover cfg's envs and agents
int validate_reward_cfg(const SwarmConfig* cfg, const SwarmRewardSpec& s, bool same_shape) {
  if (cfg->scenario != SWARM_SCENARIO_GOTO)
    return fail(SWARM_ERR_INVALID_ARG,
                "the Flocking / Cohesion rewards run on the GoTo world (cfg->scenario = SWARM_SCENARIO_GOTO)");
  if (same_shape && (s.num_envs != cfg->num_envs || s.n_agents != cfg->n_agents))
    return fail(SWARM_ERR_INVALID_ARG, "reward spec and cfg disagree on num_envs / n_agents");
  if (cfg->n_agents < 2) return fail(SWARM_ERR_INVALID_ARG, "the scenario rewards need at least two agents");
  return SWARM_OK;
}

// Flocking's shaping memory and Cohesion's parameters; per_agent_reward: the call writes the reward array (a rollout
// adds it to returns instead)
int validate_reward_buffers(const SwarmRewardSpec& s, const float* shaping, bool per_agent_reward, const float* reward) {
  if (s.kind == SWARM_REWARD_FLOCKING) {
    if (!shaping) return fail(SWARM_ERR_INVALID_ARG, "Flocking needs the shaping buffer");
    if (per_agent_reward && !s.reset && !reward) return fail(SWARM_ERR_INVALID_ARG, "reward is NULL");
  } else {
    if (s.reset) return fail(SWARM_ERR_INVALID_ARG, "Cohesion keeps no shaping memory (reset must be 0)");
    if (per_agent_reward && !reward) return fail(SWARM_ERR_INVALID_ARG, "reward is NULL");
    if (!(s.sigma > 0.0f)) return fail(SWARM_ERR_INVALID_ARG, "sigma must be > 0");
  }
  return SWARM_OK;
}

template <class T> T align256(T x) { return (x + 255) & ~(T)255; }

// the start grid of reset_grid: math.ceil(math.sqrt(num_points)) columns, math.ceil(num_points / num_cols) rows
struct GridShape {
  int cols, rows;
  explicit GridShape(int n) : cols((int)std::ceil(std::sqrt((double)n))), rows((int)std::ceil((double)n / (double)cols)) {}
};

// The workspace of a large-swarm rollout: the byte count its *_workspace_bytes call reports and, in a buffer of that
// size, where each piece starts (256-byte aligned). One function per call computes both, so they cannot disagree.
struct RolloutWorkspace {
  int64_t bytes = 0;
  int32_t* actions = nullptr;
  int32_t* nbr = nullptr;       // the kNN graph's topk table
  void* forward = nullptr;      // the large stacked forward's workspace
  void* reward = nullptr;       // the large scenario reward's per-agent terms
};

int64_t knn_table_k(const SwarmConfig& c) { return c.graph_mode == SWARM_GRAPH_KNN && c.knn_k > 0 ? c.knn_k : 0; }

// swarm_rollout_large: topk table, then actions
RolloutWorkspace rollout_large_workspace(const SwarmConfig& c, void* ws = nullptr) {
  const int64_t bn = (int64_t)c.num_envs * c.n_agents;
  const uintptr_t base = align256(reinterpret_cast<uintptr_t>(ws));
  RolloutWorkspace w;
  w.bytes = bn * knn_table_k(c) * 4 + bn * 4 + 512;
  w.nbr = reinterpret_cast<int32_t*>(base);
  w.actions = reinterpret_cast<int32_t*>(base + bn * knn_table_k(c) * 4);
  return w;
}

// swarm_rollout_stack above 128 agents: actions, topk table, then the large forward's workspace at the widest layer
// (hidden 32). The n_agents <= 128 rollout is one launch that does not touch the workspace; its size is kept as the
// ABI states it.
RolloutWorkspace rollout_stack_workspace(const SwarmConfig& c, void* ws = nullptr) {
  const int64_t bn = (int64_t)c.num_envs * c.n_agents;
  RolloutWorkspace w;
  if (c.n_agents <= kTileThreads) {
    w.bytes = bn * 4 + bn * 4 + bn + 1024;
    return w;
  }
  const int64_t tables = align256(bn * 4 + bn * knn_table_k(c) * 4);
  const uintptr_t base = align256(reinterpret_cast<uintptr_t>(ws));
  w.bytes = 256 + tables + stack_large_workspace_bytes(c, 32);
  w.actions = reinterpret_cast<int32_t*>(base);
  w.nbr = reinterpret_cast<int32_t*>(base + bn * 4);
  w.forward = reinterpret_cast<void*>(base + tables);
  return w;
}

// swarm_rollout_stack_large: the stacked layout, then (reward) the large scenario reward's per-agent terms
RolloutWorkspace rollout_stack_large_workspace(const SwarmConfig& c, const SwarmRewardSpec* reward, void* ws = nullptr) {
  RolloutWorkspace w = rollout_stack_workspace(c, ws);
  if (!reward) return w;
  SwarmRewardSpec rs = *reward;
  rs.num_envs = c.num_envs;
  rs.n_agents = c.n_agents;
  w.reward = reinterpret_cast<void*>(align256(reinterpret_cast<uintptr_t>(ws) + (uintptr_t)w.bytes));
  w.bytes += 256 + scenario_reward_large_workspace_bytes(rs);
  return w;
}

int fill_params(TileParams& p, const SwarmConfig* cfg, int mode) {
  std::memset(&p, 0, sizeof(p));
  p.cfg = *cfg;
  const int n = cfg->n_agents;
  p.epb = n <= kTileThreads ? kTileThreads / n : 1;
  p.ticks = 1;
  const bool knn = cfg->graph_mode == SWARM_GRAPH_KNN;
  p.maxdeg = knn ? (n + cfg->knn_k + 1) : n;
  p.edges_per_env = (int32_t)swarm_edges_per_env(cfg);
  p.world = world_consts(*cfg);
  p.qmax_r = cfg->graph_mode == SWARM_GRAPH_RADIUS ? sq_threshold(cfg->graph_radius) : 0.0f;
  // dense contractions on the tensor cores (tcgen05 3xTF32) unless SWARM_TC=0 selects the CUDA-core FFMA path
  const char* tc_env = std::getenv("SWARM_TC");
  p.use_tc = (mode == MODE_ROLLOUT || mode == MODE_FORWARD) && !(tc_env && tc_env[0] == '0');
  const char* ord_env = std::getenv("SWARM_KNN_ORDERED");
  p.knn_ordered = (ord_env && ord_env[0] == '1') ? 1 : 0;
  const TileLayout L = tile_layout(mode, kTileThreads, n, cfg->knn_k, p.maxdeg, cfg->graph_mode, p.use_tc != 0);
  if (L.total > 227 * 1024) return fail(SWARM_ERR_UNSUPPORTED, "shared-memory tile exceeds 227 KB for this (N, k)");
  return SWARM_OK;
}

SimStepArgs step_args(const SwarmConfig& c, const float* state_in, const int32_t* actions, float* state_out) {
  SimStepArgs p;
  std::memset(&p, 0, sizeof(p));
  p.cfg = c;
  p.world = world_consts(c);
  p.state_in = reinterpret_cast<const float4*>(state_in);
  p.actions = actions;
  p.state_out = reinterpret_cast<float4*>(state_out);
  return p;
}
}  // namespace
}  // namespace swarm

using namespace swarm;

extern "C" {

int swarm_abi_version(void) { return SWARM_ABI_VERSION; }

const char* swarm_last_error(void) { return g_last_error.c_str(); }

void swarm_default_config(SwarmConfig* cfg, int32_t scenario, int32_t num_envs, int32_t n_agents) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->grid_spacing = 0.15;
  cfg->num_envs = num_envs;
  cfg->n_agents = n_agents;
  cfg->scenario = scenario;
  cfg->graph_mode = SWARM_GRAPH_COMPLETE;
  cfg->knn_k = 10;
  cfg->dt = 0.1f;
  cfg->drag = 0.25f;
  cfg->collision_force = 100.0f;
  cfg->contact_margin = 1e-3f;
  cfg->agent_radius = 0.05f;
  cfg->landmark_radius = 0.05f;
  cfg->goal_x = -0.8f;
  cfg->goal_y = 0.8f;
  cfg->obstacle_x = -0.1f;
  cfg->obstacle_y = 0.1f;
  cfg->hit_distance = 0.2f;
  cfg->penalty_distance = 1.0f;
  cfg->obstacle_weight = 2.5f;
  cfg->graph_radius = 0.35f;       // extension default: <= 20 neighbours on the 0.15-spaced start grid
}

int64_t swarm_edges_per_env(const SwarmConfig* cfg) {
  if (!cfg) return 0;
  const int64_t n = cfg->n_agents;
  if (cfg->graph_mode == SWARM_GRAPH_KNN) return 2 * (int64_t)cfg->knn_k * n + 1;
  return n * (n - 1) + 1;
}

int swarm_reset_grid(const SwarmConfig* cfg, const float* centers, float* state, void* stream) {
  if (int rc = validate(cfg, false, true)) return rc;
  if (!centers || !state) return fail(SWARM_ERR_INVALID_ARG, "centers/state is NULL");
  const GridShape g(cfg->n_agents);
  return check_cuda(launch_reset_grid(*cfg, g.cols, g.rows, centers, state, (cudaStream_t)stream), "swarm_reset_grid");
}

int swarm_sim_step(const SwarmConfig* cfg, const float* state_in, const int32_t* actions, float* state_out,
                   float* rewards, uint8_t* flags, uint32_t* contact, float* obs, float* dist, void* stream) {
  if (int rc = validate(cfg, false, true)) return rc;
  if (!state_in || !actions || !state_out) return fail(SWARM_ERR_INVALID_ARG, "state_in/actions/state_out is NULL");
  if (contact && cfg->n_agents > 32) return fail(SWARM_ERR_UNSUPPORTED, "contact masks need n_agents <= 32");
  SimStepArgs p = step_args(*cfg, state_in, actions, state_out);
  p.rewards = rewards;
  p.flags = flags;
  p.contact = contact;
  p.obs = obs;
  p.dist = reinterpret_cast<float2*>(dist);
  // n_agents <= 128: whole envs per CTA, TMA-streamed for small swarms where the tiles allow (step_kernels.cu); above:
  // one env per CTA (large_kernels.cu) -- both run the same device arithmetic
  if (cfg->n_agents > kTileThreads) return check_cuda(launch_sim_step_large(p, (cudaStream_t)stream), "swarm_sim_step");
  return check_cuda(launch_sim_step(p, (cudaStream_t)stream), "swarm_sim_step");
}

int swarm_graph_build(const SwarmConfig* cfg, const float* state, int32_t* edges, int32_t* neighbours, void* stream) {
  if (int rc = validate(cfg, true, true)) return rc;
  if (!state) return fail(SWARM_ERR_INVALID_ARG, "state is NULL");
  if (!edges && !neighbours) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  if (cfg->graph_mode == SWARM_GRAPH_RADIUS)
    return fail(SWARM_ERR_INVALID_ARG, "radius graphs have a per-env edge count: use swarm_graph_build_radius");
  if (cfg->n_agents > kTileThreads) {
    if (int rc = validate_large_knn(*cfg)) return rc;
    if (cfg->graph_mode == SWARM_GRAPH_KNN && cfg->knn_k > 64) return fail(SWARM_ERR_UNSUPPORTED, "knn_k > 64");
    return check_cuda(launch_graph_large(*cfg, state, edges, neighbours, (int)swarm_edges_per_env(cfg), (cudaStream_t)stream),
                      "swarm_graph_build");
  }
  TileParams p;
  if (int rc = fill_params(p, cfg, MODE_GRAPH)) return rc;
  p.state_in = state;
  p.edges_out = edges;
  p.nbr_out = neighbours;
  return check_cuda(launch_tile(MODE_GRAPH, p, (cudaStream_t)stream), "swarm_graph_build");
}

int swarm_graph_build_radius(const SwarmConfig* cfg, const float* state, int32_t* edges, int32_t* counts, void* stream) {
  if (int rc = validate(cfg, true)) return rc;
  if (cfg->graph_mode != SWARM_GRAPH_RADIUS) return fail(SWARM_ERR_INVALID_ARG, "cfg->graph_mode must be SWARM_GRAPH_RADIUS");
  if (!state || !edges) return fail(SWARM_ERR_INVALID_ARG, "state/edges is NULL");
  TileParams p;
  if (int rc = fill_params(p, cfg, MODE_GRAPH)) return rc;
  p.state_in = state;
  p.edges_out = edges;
  p.counts_out = counts;
  return check_cuda(launch_tile(MODE_GRAPH, p, (cudaStream_t)stream), "swarm_graph_build_radius");
}

int swarm_gatq_forward(const SwarmConfig* cfg, const float* weights, const float* state, float* q, int32_t* actions,
                       void* stream) {
  if (int rc = validate(cfg, true)) return rc;
  if (!weights || !state) return fail(SWARM_ERR_INVALID_ARG, "weights/state is NULL");
  if (!q && !actions) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  TileParams p;
  if (int rc = fill_params(p, cfg, MODE_FORWARD)) return rc;
  p.weights = weights;
  p.state_in = state;
  p.q_out = q;
  p.act_out = actions;
  return check_cuda(launch_tile(MODE_FORWARD, p, (cudaStream_t)stream), "swarm_gatq_forward");
}

int64_t swarm_gatq_workspace_bytes(int32_t n_nodes) { return n_nodes > 0 ? gatq_workspace_bytes(n_nodes) : 0; }

int swarm_gatq_forward_csr(int32_t n_nodes, const float* weights, const float* x, const int32_t* row_ptr,
                           const int32_t* src, float* q, int32_t* actions, void* workspace, int64_t workspace_bytes,
                           void* stream) {
  if (n_nodes < 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes must be >= 0");
  if (n_nodes == 0) return SWARM_OK;
  if (!weights || !x || !row_ptr || !workspace) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (!q && !actions) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  if (workspace_bytes < gatq_workspace_bytes(n_nodes)) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  float* rows = reinterpret_cast<float*>(align256(reinterpret_cast<uintptr_t>(workspace)));
  return check_cuda(launch_gatq_csr(n_nodes, weights, x, row_ptr, src, q, actions, rows, (cudaStream_t)stream),
                    "swarm_gatq_forward_csr");
}

int swarm_gatq_forward_knn_large(const SwarmConfig* cfg, const float* weights, const float* state,
                                 const int32_t* neighbours, float* q, int32_t* actions, void* stream) {
  if (int rc = validate(cfg, true, true)) return rc;
  if (cfg->graph_mode != SWARM_GRAPH_KNN) return fail(SWARM_ERR_INVALID_ARG, "cfg->graph_mode must be SWARM_GRAPH_KNN");
  if (!weights || !state || !neighbours) return fail(SWARM_ERR_INVALID_ARG, "weights/state/neighbours is NULL");
  if (!q && !actions) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  if (!gatq_knn_large_fits(cfg->n_agents, cfg->knn_k))
    return fail(SWARM_ERR_UNSUPPORTED, "the env does not fit shared memory: use swarm_graph_build + swarm_csr_from_edges + "
                                       "swarm_gatq_forward_csr");
  return check_cuda(launch_gatq_knn_large(*cfg, weights, state, neighbours, q, actions, (cudaStream_t)stream),
                    "swarm_gatq_forward_knn_large");
}

int swarm_graph_build_radius_csr(const SwarmConfig* cfg, const float* state, int32_t* degree, const int32_t* row_ptr,
                                 int32_t* src, void* stream) {
  if (int rc = validate(cfg, true, true)) return rc;
  if (cfg->graph_mode != SWARM_GRAPH_RADIUS) return fail(SWARM_ERR_INVALID_ARG, "cfg->graph_mode must be SWARM_GRAPH_RADIUS");
  if (!state) return fail(SWARM_ERR_INVALID_ARG, "state is NULL");
  if ((src == nullptr) == (degree == nullptr))
    return fail(SWARM_ERR_INVALID_ARG, "pass degree (count pass) or row_ptr + src (fill pass), not both");
  if (src && !row_ptr) return fail(SWARM_ERR_INVALID_ARG, "the fill pass needs row_ptr");
  if ((int64_t)cfg->num_envs * cfg->n_agents > 0x7fffffffLL) return fail(SWARM_ERR_UNSUPPORTED, "more than 2^31 - 1 nodes");
  return check_cuda(launch_radius_csr(*cfg, state, degree, row_ptr, src, (cudaStream_t)stream), "swarm_graph_build_radius_csr");
}

int swarm_gatq_forward_large(const SwarmConfig* cfg, const float* weights, const float* state, float* q, int32_t* actions,
                             void* stream) {
  if (int rc = validate(cfg, true, true)) return rc;
  if (cfg->graph_mode != SWARM_GRAPH_RADIUS && cfg->graph_mode != SWARM_GRAPH_COMPLETE)
    return fail(SWARM_ERR_INVALID_ARG, "cfg->graph_mode must be SWARM_GRAPH_RADIUS or SWARM_GRAPH_COMPLETE "
                                       "(kNN: swarm_gatq_forward_knn_large)");
  if (!weights || !state) return fail(SWARM_ERR_INVALID_ARG, "weights/state is NULL");
  if (!q && !actions) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  if (!gatq_large_x_fits(cfg->n_agents, cfg->graph_mode == SWARM_GRAPH_RADIUS))
    return fail(SWARM_ERR_UNSUPPORTED, "the env does not fit shared memory");
  return check_cuda(launch_gatq_large_x(*cfg, weights, state, q, actions, (cudaStream_t)stream), "swarm_gatq_forward_large");
}

int64_t swarm_rollout_large_workspace_bytes(const SwarmConfig* cfg) {
  if (!cfg || cfg->num_envs <= 0 || cfg->n_agents <= 0) return 0;
  return rollout_large_workspace(*cfg).bytes;
}

int swarm_rollout_large(const SwarmConfig* cfg, const float* weights, float* state, int32_t ticks, float* returns,
                        int32_t* hits, void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = validate(cfg, true, true)) return rc;
  if (cfg->n_agents <= kTileThreads) return fail(SWARM_ERR_INVALID_ARG, "n_agents <= 128: use swarm_rollout");
  if (!weights || !state || !workspace) return fail(SWARM_ERR_INVALID_ARG, "weights/state/workspace is NULL");
  if (ticks < 0) return fail(SWARM_ERR_INVALID_ARG, "ticks must be >= 0");
  if (int rc = validate_large_knn(*cfg)) return rc;
  const bool knn = cfg->graph_mode == SWARM_GRAPH_KNN;
  // attention in input space (no projected-feature tile: envs up to 4 096 agents fit) unless SWARM_TC=0 asks for the
  // bit-faithful forward of swarm_gatq_forward_knn_large (kNN only; the radius / complete graph of a large swarm has
  // the input-space forward alone -- their bit-faithful path is the CSR one)
  const char* tc_env = std::getenv("SWARM_TC");
  const bool xspace = !knn || !(tc_env && tc_env[0] == '0');
  const bool fits = !knn ? gatq_large_x_fits(cfg->n_agents, cfg->graph_mode == SWARM_GRAPH_RADIUS)
                         : (xspace ? gatq_knn_large_x_fits(cfg->n_agents, cfg->knn_k)
                                   : gatq_knn_large_fits(cfg->n_agents, cfg->knn_k));
  if (!fits)
    return fail(SWARM_ERR_UNSUPPORTED, "the env does not fit shared memory: step it with swarm_graph_build + "
                                       "swarm_csr_from_edges + swarm_gatq_forward_csr + swarm_sim_step");
  const RolloutWorkspace w = rollout_large_workspace(*cfg, workspace);
  if (workspace_bytes < w.bytes) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  int32_t *nbr = w.nbr, *actions = w.actions;
  // in place: one CTA owns a whole env and stages its positions first
  SimStepArgs p = step_args(*cfg, state, actions, state);
  p.returns = returns;
  p.hits = hits;
  cudaStream_t st = (cudaStream_t)stream;
  for (int t = 0; t < ticks; ++t) {
    // simulator.py:59-68 per tick: topk table -> GCN forward + argmax straight from the table -> Environment.step,
    // returns / hits accumulated by the step kernel: three launches, nothing but the state leaves the device
    // (radius / complete graph: the forward finds its own sources -- uniform-grid broad phase / every other agent --
    // so a tick is two launches)
    if (knn) {
      if (cudaError_t e = launch_graph_large(*cfg, state, nullptr, nbr, (int)swarm_edges_per_env(cfg), st); e != cudaSuccess)
        return check_cuda(e, "swarm_rollout_large (graph)");
      if (cudaError_t e = xspace ? launch_gatq_knn_large_x(*cfg, weights, state, nbr, nullptr, actions, st)
                                 : launch_gatq_knn_large(*cfg, weights, state, nbr, nullptr, actions, st);
          e != cudaSuccess)
        return check_cuda(e, "swarm_rollout_large (forward)");
    } else if (cudaError_t e = launch_gatq_large_x(*cfg, weights, state, nullptr, actions, st); e != cudaSuccess) {
      return check_cuda(e, "swarm_rollout_large (forward)");
    }
    if (cudaError_t e = launch_sim_step_large(p, st); e != cudaSuccess) return check_cuda(e, "swarm_rollout_large (step)");
  }
  return SWARM_OK;
}

int swarm_gatconv_forward_csr(int32_t n_nodes, const float* weights, const float* x, const int32_t* row_ptr,
                              const int32_t* src, float* out, void* workspace, int64_t workspace_bytes, void* stream) {
  if (n_nodes < 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes must be >= 0");
  if (n_nodes == 0) return SWARM_OK;
  if (!weights || !x || !row_ptr || !out || !workspace) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (workspace_bytes < gatq_workspace_bytes(n_nodes)) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  float* rows = reinterpret_cast<float*>(align256(reinterpret_cast<uintptr_t>(workspace)));
  return check_cuda(launch_gatq_csr(n_nodes, weights, x, row_ptr, src, out, nullptr, rows, (cudaStream_t)stream, true),
                    "swarm_gatconv_forward_csr");
}

int swarm_gatconv_backward_csr(int32_t n_nodes, int64_t n_edges, const float* weights, const float* x,
                               const int32_t* row_ptr, const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                               const int32_t* tgt_s, const int32_t* perm_s, const float* grad_out, float* grad_weights,
                               void* workspace, int64_t workspace_bytes, void* stream) {
  if (n_nodes <= 0 || n_edges < 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes must be > 0 and n_edges >= 0");
  if (n_edges >= (1LL << 31)) return fail(SWARM_ERR_UNSUPPORTED, "more than 2^31 - 1 edges");
  if (!weights || !x || !row_ptr || !row_ptr_s || !grad_out || !grad_weights || !workspace)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (n_edges > 0 && (!src || !perm || !tgt_s || !perm_s)) return fail(SWARM_ERR_INVALID_ARG, "NULL edge array");
  if (workspace_bytes < gatq_backward_workspace_bytes(n_nodes, n_edges))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_gatq_backward_csr(n_nodes, n_edges, weights, x, row_ptr, src, perm, row_ptr_s, tgt_s, perm_s,
                                             grad_out, grad_weights, workspace, (cudaStream_t)stream, true),
                    "swarm_gatconv_backward_csr");
}

static int gat_layer_check_dims(int32_t n_nodes, int64_t n_edges, int32_t ci, int32_t co) {
  if (n_nodes < 0 || n_edges < 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes and n_edges must be >= 0");
  if (n_edges >= (1LL << 31)) return fail(SWARM_ERR_UNSUPPORTED, "more than 2^31 - 1 edges");
  if (ci < 1 || co < 1) return fail(SWARM_ERR_INVALID_ARG, "in_channels and out_channels must be >= 1");
  if (ci > 64 || co > 64) return fail(SWARM_ERR_UNSUPPORTED, "the GAT layer kernels cover in_channels, out_channels <= 64");
  if ((int64_t)n_nodes * 68 >= (1LL << 31)) return fail(SWARM_ERR_UNSUPPORTED, "too many nodes for one call");
  return SWARM_OK;
}

int64_t swarm_gat_layer_workspace_bytes(int32_t n_nodes, int64_t n_edges, int32_t in_channels, int32_t out_channels,
                                        int32_t backward) {
  if (gat_layer_check_dims(n_nodes, n_edges, in_channels, out_channels)) return -1;
  return gat_layer_workspace_bytes(n_nodes, n_edges, in_channels, out_channels, backward != 0);
}

int swarm_gat_layer_forward(int32_t n_nodes, int32_t in_channels, int32_t out_channels, const float* lin_weight,
                            const float* att_src, const float* att_dst, const float* bias, const float* x,
                            const int32_t* row_ptr, const int32_t* src, float* out, void* workspace,
                            int64_t workspace_bytes, void* stream) {
  if (int rc = gat_layer_check_dims(n_nodes, 0, in_channels, out_channels)) return rc;
  if (n_nodes == 0) return SWARM_OK;
  if (!lin_weight || !att_src || !att_dst || !bias || !x || !row_ptr || !out || !workspace)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (workspace_bytes < gat_layer_workspace_bytes(n_nodes, 0, in_channels, out_channels, false))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_gat_layer_forward(n_nodes, in_channels, out_channels, lin_weight, att_src, att_dst, bias, x,
                                             row_ptr, src, out, workspace, (cudaStream_t)stream),
                    "swarm_gat_layer_forward");
}

int swarm_gat_layer_backward(int32_t n_nodes, int64_t n_edges, int32_t in_channels, int32_t out_channels,
                             const float* lin_weight, const float* att_src, const float* att_dst, const float* x,
                             const int32_t* row_ptr, const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                             const int32_t* tgt_s, const int32_t* perm_s, const float* grad_out, float* grad_lin_weight,
                             float* grad_att_src, float* grad_att_dst, float* grad_bias, float* grad_x, void* workspace,
                             int64_t workspace_bytes, void* stream) {
  if (int rc = gat_layer_check_dims(n_nodes, n_edges, in_channels, out_channels)) return rc;
  if (n_nodes == 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes must be > 0");
  if (!lin_weight || !att_src || !att_dst || !x || !row_ptr || !row_ptr_s || !grad_out || !grad_lin_weight ||
      !grad_att_src || !grad_att_dst || !grad_bias || !workspace)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (n_edges > 0 && (!src || !perm || !tgt_s || !perm_s)) return fail(SWARM_ERR_INVALID_ARG, "NULL edge array");
  if (workspace_bytes < gat_layer_workspace_bytes(n_nodes, n_edges, in_channels, out_channels, true))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_gat_layer_backward(n_nodes, n_edges, in_channels, out_channels, lin_weight, att_src, att_dst, x,
                                              row_ptr, src, perm, row_ptr_s, tgt_s, perm_s, grad_out, grad_lin_weight,
                                              grad_att_src, grad_att_dst, grad_bias, grad_x, workspace,
                                              (cudaStream_t)stream),
                    "swarm_gat_layer_backward");
}

int64_t swarm_gatq_backward_workspace_bytes(int32_t n_nodes, int64_t n_edges) {
  if (n_nodes <= 0 || n_edges < 0) return 0;
  return gatq_backward_workspace_bytes(n_nodes, n_edges);
}

int swarm_gatq_backward_csr(int32_t n_nodes, int64_t n_edges, const float* weights, const float* x, const int32_t* row_ptr,
                            const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s, const int32_t* tgt_s,
                            const int32_t* perm_s, const float* grad_q, float* grad_weights, void* workspace,
                            int64_t workspace_bytes, void* stream) {
  if (n_nodes <= 0 || n_edges < 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes must be > 0 and n_edges >= 0");
  if (n_edges >= (1LL << 31)) return fail(SWARM_ERR_UNSUPPORTED, "more than 2^31 - 1 edges");
  if (!weights || !x || !row_ptr || !row_ptr_s || !grad_q || !grad_weights || !workspace)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (n_edges > 0 && (!src || !perm || !tgt_s || !perm_s)) return fail(SWARM_ERR_INVALID_ARG, "NULL edge array");
  if (workspace_bytes < gatq_backward_workspace_bytes(n_nodes, n_edges))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_gatq_backward_csr(n_nodes, n_edges, weights, x, row_ptr, src, perm, row_ptr_s, tgt_s, perm_s,
                                             grad_q, grad_weights, workspace, (cudaStream_t)stream),
                    "swarm_gatq_backward_csr");
}

int64_t swarm_csr_workspace_bytes(int32_t n_nodes, int64_t n_edges) {
  if (n_nodes <= 0 || n_edges < 0) return 0;
  return csr_workspace_bytes(n_nodes, n_edges);
}

int swarm_csr_from_edges(int32_t n_nodes, int64_t n_edges, const int64_t* edge_src, const int64_t* edge_dst,
                         int32_t* row_ptr, int32_t* src, int32_t* perm, void* workspace, int64_t workspace_bytes,
                         void* stream) {
  if (n_nodes <= 0 || n_edges < 0) return fail(SWARM_ERR_INVALID_ARG, "n_nodes must be > 0 and n_edges >= 0");
  if (n_edges >= (1LL << 31)) return fail(SWARM_ERR_UNSUPPORTED, "more than 2^31 - 1 edges");
  if (!row_ptr || !workspace) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (n_edges > 0 && (!edge_src || !edge_dst || !src || !perm)) return fail(SWARM_ERR_INVALID_ARG, "NULL edge array");
  if (workspace_bytes < csr_workspace_bytes(n_nodes, n_edges)) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_csr_from_edges(n_nodes, n_edges, edge_src, edge_dst, row_ptr, src, perm, workspace,
                                          workspace_bytes, (cudaStream_t)stream),
                    "swarm_csr_from_edges");
}

// SwarmRolloutOptions / SwarmTrainHyper: the optional Flocking reward of the fused tick
static int attach_flocking(TileParams& p, const SwarmConfig* cfg, const SwarmRewardSpec* fs, float* shaping) {
  if (!fs) return SWARM_OK;
  if (fs->kind != SWARM_REWARD_FLOCKING) return fail(SWARM_ERR_INVALID_ARG, "`flocking` must be a Flocking reward spec");
  if (int rc = validate_reward_cfg(cfg, *fs, false)) return rc;
  if (int rc = validate_reward_buffers(*fs, shaping, false, nullptr)) return rc;
  p.flock = *fs;
  p.shaping = reinterpret_cast<float2*>(shaping);
  p.use_flock = 1;
  return SWARM_OK;
}

int swarm_rollout(const SwarmConfig* cfg, const float* weights, float* state, int32_t ticks,
                  const SwarmRolloutOptions* opts, float* returns, int32_t* hits, const SwarmTrace* trace, void* stream) {
  if (int rc = validate(cfg, true)) return rc;
  if (!weights || !state) return fail(SWARM_ERR_INVALID_ARG, "weights/state is NULL");
  if (ticks < 0) return fail(SWARM_ERR_INVALID_ARG, "ticks must be >= 0");
  if (ticks == 0) return SWARM_OK;
  if (trace && trace->contact && cfg->n_agents > 32)
    return fail(SWARM_ERR_UNSUPPORTED, "contact masks need n_agents <= 32");
  if (trace && trace->edges && cfg->graph_mode == SWARM_GRAPH_RADIUS)
    return fail(SWARM_ERR_UNSUPPORTED, "per-tick edge traces are not available for radius graphs (variable edge count)");
  TileParams p;
  if (int rc = fill_params(p, cfg, MODE_ROLLOUT)) return rc;
  p.weights = weights;
  p.state_in = state;
  p.state_out = state;
  p.ticks = ticks;
  p.returns = returns;
  p.hits = hits;
  if (opts) {
    if (opts->epsilon < 0.0f || opts->epsilon > 1.0f) return fail(SWARM_ERR_INVALID_ARG, "epsilon must be in [0, 1]");
    p.actions_in = opts->forced_actions;
    p.epsilon = opts->epsilon;
    p.rng_seed = opts->rng_seed;
    p.rng_tick0 = opts->rng_tick0;
    p.env_offset = opts->env_offset;
    if (opts->replay) {
      if (int rc = validate_ring(opts->replay, "replay ring", true)) return rc;
      const SwarmReplay& r = *opts->replay;
      if ((int64_t)ticks * cfg->num_envs > r.capacity)
        return fail(SWARM_ERR_INVALID_ARG, "ticks * num_envs exceeds the replay capacity (slots would be overwritten inside one call)");
      p.replay = r;
      p.replay_cursor = opts->replay_cursor % r.capacity;
    }
    if (int rc = attach_flocking(p, cfg, opts->flocking, opts->flocking_shaping)) return rc;
    if (opts->knn_memo) {
      const int64_t n = opts->knn_memo_entries;
      if (n <= 0 || (n & (n - 1)) != 0 || n > (1LL << 32))
        return fail(SWARM_ERR_INVALID_ARG, "knn_memo_entries must be a power of two (<= 2^32)");
      p.knn_memo = reinterpret_cast<unsigned long long*>(opts->knn_memo);
      p.knn_memo_mask = (uint32_t)(n - 1);
    }
  }
  if (trace) p.trace = *trace;
  return check_cuda(launch_tile(MODE_ROLLOUT, p, (cudaStream_t)stream), "swarm_rollout");
}

int swarm_replay_push(const SwarmConfig* cfg, const SwarmReplay* replay, int64_t cursor, const float* state,
                      const int32_t* actions, const float* rewards, const float* next_state, void* stream) {
  if (int rc = validate(cfg, false)) return rc;
  if (int rc = validate_ring(replay, "replay ring", true)) return rc;
  if (!state || !actions || !rewards || !next_state) return fail(SWARM_ERR_INVALID_ARG, "NULL transition array");
  if (cfg->num_envs > replay->capacity) return fail(SWARM_ERR_INVALID_ARG, "num_envs exceeds the replay capacity");
  if (cursor < 0) return fail(SWARM_ERR_INVALID_ARG, "cursor must be >= 0");
  return check_cuda(launch_replay_push(*replay, cursor % replay->capacity, cfg->num_envs, cfg->n_agents, state, actions,
                                       rewards, next_state, (cudaStream_t)stream),
                    "swarm_replay_push");
}

int swarm_replay_gather(const SwarmConfig* cfg, const SwarmReplay* replay, const int64_t* indices, int32_t n_graphs,
                        float* state, int32_t* actions, float* rewards, float* next_state, void* stream) {
  if (!cfg || cfg->n_agents <= 0) return fail(SWARM_ERR_INVALID_ARG, "cfg is NULL or n_agents <= 0");
  if (int rc = validate_ring(replay, "replay ring", false)) return rc;
  if (n_graphs < 0) return fail(SWARM_ERR_INVALID_ARG, "n_graphs must be >= 0");
  if (n_graphs == 0) return SWARM_OK;
  if (!indices || !state || !actions || !rewards || !next_state) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  return check_cuda(launch_replay_gather(*replay, indices, n_graphs, cfg->n_agents, state, actions, rewards, next_state,
                                         (cudaStream_t)stream),
                    "swarm_replay_gather");
}

static int validate_dqn(const SwarmConfig* cfg, int32_t n_graphs) {
  if (!cfg) return fail(SWARM_ERR_INVALID_ARG, "cfg is NULL");
  SwarmConfig c = *cfg;
  c.num_envs = n_graphs > 0 ? n_graphs : 1;
  if (int rc = validate(&c, true)) return rc;
  if (n_graphs <= 0) return fail(SWARM_ERR_INVALID_ARG, "n_graphs must be positive");
  if (dqn_smem_bytes(c) > 227 * 1024)
    return fail(SWARM_ERR_UNSUPPORTED, "the DQN gradient tile exceeds 227 KB of shared memory for this (N, k)");
  return SWARM_OK;
}

int64_t swarm_dqn_workspace_bytes(const SwarmConfig* cfg, int32_t n_graphs) {
  if (validate_dqn(cfg, n_graphs) != SWARM_OK) return 0;
  return dqn_workspace_bytes(*cfg, n_graphs);
}

int swarm_dqn_grad(const SwarmConfig* cfg, const float* online_weights, const float* target_weights,
                   const SwarmReplay* batch, const int64_t* indices, int32_t n_graphs, float gamma, float loss_scale,
                   float* grad, float* loss, float* td, void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = validate_dqn(cfg, n_graphs)) return rc;
  if (!online_weights || !target_weights || !grad || !loss || !workspace) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (int rc = validate_ring(batch, "batch", false)) return rc;
  if (workspace_bytes < dqn_workspace_bytes(*cfg, n_graphs)) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_dqn_grad(*cfg, online_weights, target_weights, *batch, indices, n_graphs, gamma, loss_scale,
                                    grad, loss, td, workspace, (cudaStream_t)stream),
                    "swarm_dqn_grad");
}

int swarm_adam_clip_step(float* weights, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t step, double lr,
                         double beta1, double beta2, double eps, double max_norm, float* target_weights,
                         float* grad_norm, void* stream) {
  if (!weights || !grad || !exp_avg || !exp_avg_sq) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (step < 1) return fail(SWARM_ERR_INVALID_ARG, "step is 1-based");
  if (int rc = validate_adam(lr, beta1, beta2, eps)) return rc;
  return check_cuda(launch_adam_clip(weights, grad, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, max_norm,
                                     target_weights, grad_norm, (cudaStream_t)stream),
                    "swarm_adam_clip_step");
}

static int validate_hyper(const SwarmTrainHyper* h) {
  if (!h) return fail(SWARM_ERR_INVALID_ARG, "hyper is NULL");
  if (h->graphs_per_update <= 0) return fail(SWARM_ERR_INVALID_ARG, "graphs_per_update must be positive");
  if (h->update_target_every <= 0) return fail(SWARM_ERR_INVALID_ARG, "update_target_every must be positive");
  return validate_adam(h->lr, h->beta1, h->beta2, h->eps);
}

// shared argument checks and rollout-tick parameters of swarm_train_tick_grad / swarm_train_tick
static int train_tick_rollout(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl, const float* weights,
                              const float* target_weights, float* state, float* returns, int32_t* hits,
                              const SwarmReplay* ring, float* grad, float* loss, void* workspace, int64_t workspace_bytes,
                              cudaStream_t st, const char* what) {
  if (int rc = validate(cfg, true)) return rc;
  if (int rc = validate_hyper(hyper)) return rc;
  if (int rc = validate_dqn(cfg, hyper->graphs_per_update)) return rc;
  if (!ctl || !weights || !target_weights || !state || !grad || !loss || !workspace)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (int rc = validate_ring(ring, "replay ring", true)) return rc;
  if (cfg->num_envs > ring->capacity) return fail(SWARM_ERR_INVALID_ARG, "num_envs exceeds the replay capacity");
  if (workspace_bytes < dqn_workspace_bytes(*cfg, hyper->graphs_per_update))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  TileParams p;
  if (int rc = fill_params(p, cfg, MODE_ROLLOUT)) return rc;
  p.weights = weights;
  p.state_in = state;
  p.state_out = state;
  p.ticks = 1;
  p.returns = returns;
  p.hits = hits;
  p.rng_seed = hyper->rng_seed;
  p.env_offset = hyper->env_offset;
  p.replay = *ring;
  p.ctl = ctl;
  if (int rc = attach_flocking(p, cfg, hyper->flocking, hyper->flocking_shaping)) return rc;
  return check_cuda(launch_tile(MODE_ROLLOUT, p, st), what);
}

static int validate_peers(const SwarmPeerExchange* peers) {
  if (!peers) return SWARM_OK;
  if (peers->world_size < 1 || peers->world_size > SWARM_MAX_PEERS || peers->rank < 0 || peers->rank >= peers->world_size)
    return fail(SWARM_ERR_INVALID_ARG, "peer exchange: bad world_size / rank");
  for (int r = 0; r < peers->world_size; ++r)
    if (!peers->data[r]) return fail(SWARM_ERR_INVALID_ARG, "peer exchange: NULL peer buffer");
  return SWARM_OK;
}

int swarm_train_tick_grad(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl, const float* weights,
                          const float* target_weights, float* state, float* returns, int32_t* hits,
                          const SwarmReplay* ring, int64_t* indices, float* grad, float* loss, void* workspace,
                          int64_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = train_tick_rollout(cfg, hyper, ctl, weights, target_weights, state, returns, hits, ring, grad, loss,
                                  workspace, workspace_bytes, st, "swarm_train_tick_grad(rollout)"))
    return rc;
  return check_cuda(launch_dqn_grad(*cfg, weights, target_weights, *ring, nullptr, hyper->graphs_per_update, hyper->gamma,
                                    hyper->loss_scale, grad, loss, nullptr, workspace, st, ctl, indices,
                                    hyper->sample_seed, cfg->num_envs),
                    "swarm_train_tick_grad(grad)");
}

int swarm_train_tick_apply(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl, float* weights,
                           float* target_weights, float* exp_avg, float* exp_avg_sq, float* grad,
                           int64_t ring_capacity, const SwarmPeerExchange* peers, void* stream) {
  if (!cfg || cfg->num_envs <= 0) return fail(SWARM_ERR_INVALID_ARG, "cfg is NULL or num_envs <= 0");
  if (int rc = validate_hyper(hyper)) return rc;
  if (!ctl || !weights || !target_weights || !exp_avg || !exp_avg_sq || !grad) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (ring_capacity < cfg->num_envs) return fail(SWARM_ERR_INVALID_ARG, "ring_capacity must be >= num_envs");
  if (int rc = validate_peers(peers)) return rc;
  return check_cuda(launch_adam_clip(weights, grad, exp_avg, exp_avg_sq, 1, hyper->lr, hyper->beta1, hyper->beta2,
                                     hyper->eps, hyper->max_norm, target_weights, nullptr, (cudaStream_t)stream, ctl,
                                     cfg->num_envs, ring_capacity, hyper->update_target_every, peers, grad),
                    "swarm_train_tick_apply");
}

int swarm_train_tick(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl, float* weights,
                     float* target_weights, float* exp_avg, float* exp_avg_sq, float* state, float* returns,
                     int32_t* hits, const SwarmReplay* ring, int64_t* indices, float* grad, void* workspace,
                     int64_t workspace_bytes, const SwarmPeerExchange* peers, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!exp_avg || !exp_avg_sq) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (int rc = validate_peers(peers)) return rc;
  if (int rc = train_tick_rollout(cfg, hyper, ctl, weights, target_weights, state, returns, hits, ring, grad,
                                  grad ? grad + SWARM_W_COUNT : nullptr, workspace, workspace_bytes, st,
                                  "swarm_train_tick(rollout)"))
    return rc;
  const int G = hyper->graphs_per_update;
  // gradient kernel on few CTAs: partial reduction (+ peer exchange) + clip + Adam as one cluster launch; a large update
  // batch keeps the reduce launch and the single-CTA clip + Adam kernel
  const bool fuse = dqn_fuse_reduce(*cfg, G);
  if (int rc = check_cuda(launch_dqn_grad(*cfg, weights, target_weights, *ring, nullptr, G, hyper->gamma, hyper->loss_scale,
                                          grad, grad + SWARM_W_COUNT, nullptr, workspace, st, ctl, indices,
                                          hyper->sample_seed, cfg->num_envs, fuse),
                          "swarm_train_tick(grad)"))
    return rc;
  return check_cuda(launch_adam_clip(weights, grad, exp_avg, exp_avg_sq, 1, hyper->lr, hyper->beta1, hyper->beta2,
                                     hyper->eps, hyper->max_norm, target_weights, nullptr, st, ctl, cfg->num_envs,
                                     ring->capacity, hyper->update_target_every, peers, grad, fuse ? cfg : nullptr,
                                     fuse ? workspace : nullptr, G, hyper->loss_scale),
                    "swarm_train_tick(apply)");
}

int swarm_reset_random(const SwarmConfig* cfg, const SwarmResetSpec* spec, const SwarmTrainCtl* ctl, int64_t episode,
                       float* centers_out, float* state, void* stream) {
  if (int rc = validate(cfg, false, true)) return rc;
  if (!spec || !state) return fail(SWARM_ERR_INVALID_ARG, "spec/state is NULL");
  if (!(spec->std_x >= 0.0f) || !(spec->std_y >= 0.0f)) return fail(SWARM_ERR_INVALID_ARG, "std must be >= 0");
  if (!ctl && episode < 0) return fail(SWARM_ERR_INVALID_ARG, "episode must be >= 0");
  const GridShape g(cfg->n_agents);
  return check_cuda(launch_reset_random(*cfg, *spec, g.cols, g.rows, ctl, episode, centers_out, state, (cudaStream_t)stream),
                    "swarm_reset_random");
}

void swarm_default_reward_spec(SwarmRewardSpec* spec, int32_t kind, int32_t num_envs, int32_t n_agents) {
  if (!spec) return;
  *spec = SwarmRewardSpec{};
  spec->kind = kind;
  spec->num_envs = num_envs;
  spec->n_agents = n_agents;
  spec->reset = 0;
  spec->env_index = -1;
  spec->goal_x = -0.8f;
  spec->goal_y = 0.8f;
  spec->goal_radius = 0.05f;
  spec->agent_radius = 0.05f;
  spec->pos_shaping = 10.0f;
  spec->dist_shaping = 10.0f;
  spec->desired_distance = 0.15f;
  spec->min_collision_distance = 0.005f;
  spec->collision_reward = -1.0f;
  spec->on_goal_bonus = 50.0f;
  spec->sigma = 0.15f;
}

namespace {
// the argument checks of the scenario rewards up to the num_envs * n_agents bound; large = false: the env-tile kernel
// (n_agents <= 128), true: the large-swarm kernel (n_agents <= 4096)
int validate_reward_spec(const SwarmRewardSpec* spec, bool large) {
  if (!spec) return fail(SWARM_ERR_INVALID_ARG, "spec is NULL");
  if (spec->kind != SWARM_REWARD_FLOCKING && spec->kind != SWARM_REWARD_COHESION)
    return fail(SWARM_ERR_INVALID_ARG, "unknown reward kind");
  if (spec->num_envs < 0) return fail(SWARM_ERR_INVALID_ARG, "num_envs must be >= 0");
  if (spec->n_agents < 2) return fail(SWARM_ERR_INVALID_ARG, "the scenario rewards need at least two agents");
  if (!large && spec->n_agents > 128)
    return fail(SWARM_ERR_UNSUPPORTED, "scenario rewards are implemented for n_agents <= 128");
  if (large && spec->n_agents > kMaxLargeAgents)
    return fail(SWARM_ERR_UNSUPPORTED, "the large-swarm scenario rewards are implemented for n_agents <= 4096");
  if (spec->env_index < -1 || spec->env_index >= spec->num_envs)
    return fail(SWARM_ERR_INVALID_ARG, "env_index out of range");
  if ((int64_t)spec->num_envs * spec->n_agents + (large ? 0 : 128 * 148 * 16) >= (1LL << 31))
    return fail(SWARM_ERR_UNSUPPORTED, "num_envs * n_agents must stay below 2^31");
  return SWARM_OK;
}
}  // namespace

int swarm_scenario_reward(const SwarmRewardSpec* spec, const float* state, float* shaping, float* reward, float* terms,
                          void* stream) {
  if (int rc = validate_reward_spec(spec, false)) return rc;
  if (spec->num_envs == 0) return SWARM_OK;
  if (!state) return fail(SWARM_ERR_INVALID_ARG, "state is NULL");
  if (int rc = validate_reward_buffers(*spec, shaping, true, reward)) return rc;
  return check_cuda(launch_scenario_reward(*spec, state, shaping, reward, terms, (cudaStream_t)stream),
                    "swarm_scenario_reward");
}

int64_t swarm_scenario_reward_large_workspace_bytes(const SwarmRewardSpec* spec) {
  if (validate_reward_spec(spec, true) != SWARM_OK) return 0;
  return scenario_reward_large_workspace_bytes(*spec);
}

int swarm_scenario_reward_large(const SwarmRewardSpec* spec, const float* state, float* shaping, float* reward,
                                float* terms, void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = validate_reward_spec(spec, true)) return rc;
  if (spec->num_envs == 0) return SWARM_OK;
  if (!state) return fail(SWARM_ERR_INVALID_ARG, "state is NULL");
  if (int rc = validate_reward_buffers(*spec, shaping, true, reward)) return rc;
  const int64_t need = scenario_reward_large_workspace_bytes(*spec);
  if (need > 0 && !workspace) return fail(SWARM_ERR_INVALID_ARG, "workspace is NULL");
  if (workspace_bytes < need) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_scenario_reward_large(*spec, state, shaping, reward, terms, nullptr, workspace,
                                                 (cudaStream_t)stream),
                    "swarm_scenario_reward_large");
}

namespace {
// large = false: the env-tile kernels (n_agents <= 128, kNN n_agents <= 16); large = true: the one-CTA-per-env kernel
// (any n_agents <= 4096; above 128 agents the kNN table comes from the partial_sort branch of swarm_graph_build)
int validate_spec(const SwarmStackSpec* spec) {
  if (!spec) return fail(SWARM_ERR_INVALID_ARG, "spec is NULL");
  if (spec->n_layers < 1 || spec->n_layers > 4) return fail(SWARM_ERR_INVALID_ARG, "n_layers must be 1 .. 4");
  if (spec->hidden < 1 || spec->hidden > 32) return fail(SWARM_ERR_UNSUPPORTED, "hidden must be 1 .. 32");
  if (spec->in_features != 7 && spec->in_features != 5) return fail(SWARM_ERR_INVALID_ARG, "in_features must be 7 or 5");
  return SWARM_OK;
}

// large = false: the env-tile kernels (n_agents <= 128, kNN n_agents <= 16); large = true: the one-CTA-per-env kernel
// (any n_agents <= 4096; above 128 agents the kNN table comes from the partial_sort branch of swarm_graph_build)
int validate_stack(const SwarmConfig* cfg, const SwarmStackSpec* spec, bool large = false) {
  if (int rc = validate(cfg, true, large)) return rc;
  if (int rc = validate_spec(spec)) return rc;
  for (int l = 0; l < spec->n_layers; ++l)
    if (spec->activation[l] != SWARM_ACT_TANH && spec->activation[l] != SWARM_ACT_RELU)
      return fail(SWARM_ERR_INVALID_ARG, "unknown activation");
  if (!large && cfg->graph_mode == SWARM_GRAPH_KNN && cfg->n_agents > 16)
    return fail(SWARM_ERR_UNSUPPORTED, "stacked networks on the kNN graph are implemented for n_agents <= 16");
  if (int rc = validate_large_knn(*cfg)) return rc;
  if (large && stack_large_smem_bytes(*cfg, *spec) > 227 * 1024)
    return fail(SWARM_ERR_UNSUPPORTED, "the large stacked forward needs more than 227 KB of shared memory for this (N, spec)");
  return SWARM_OK;
}
}  // namespace

int64_t swarm_stack_weight_count(const SwarmStackSpec* spec) {
  if (!spec || spec->n_layers < 1 || spec->n_layers > 4 || spec->hidden < 1 || spec->hidden > 32) return 0;
  return stack_weight_count_host(*spec);
}

int swarm_gatstack_forward(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, const float* state,
                           float* q, int32_t* actions, void* stream) {
  if (int rc = validate_stack(cfg, spec)) return rc;
  if (!weights || !state) return fail(SWARM_ERR_INVALID_ARG, "weights/state is NULL");
  if (!q && !actions) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  return check_cuda(launch_gatstack_forward(*cfg, *spec, weights, state, q, actions, (cudaStream_t)stream),
                    "swarm_gatstack_forward");
}

int64_t swarm_gatstack_large_workspace_bytes(const SwarmConfig* cfg, const SwarmStackSpec* spec) {
  if (validate_stack(cfg, spec, true) != SWARM_OK) return 0;
  return stack_large_workspace_bytes(*cfg, *spec);
}

int swarm_gatstack_forward_large(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights,
                                 const float* state, const int32_t* neighbours, float* q, int32_t* actions,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = validate_stack(cfg, spec, true)) return rc;
  if (!weights || !state || !workspace) return fail(SWARM_ERR_INVALID_ARG, "weights/state/workspace is NULL");
  if (cfg->graph_mode == SWARM_GRAPH_KNN && !neighbours)
    return fail(SWARM_ERR_INVALID_ARG, "the kNN graph needs the topk table (neighbours, swarm_graph_build)");
  if (!q && !actions) return fail(SWARM_ERR_INVALID_ARG, "no output requested");
  if (workspace_bytes < stack_large_workspace_bytes(*cfg, *spec)) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_gatstack_large(*cfg, *spec, weights, state, neighbours, q, actions, workspace,
                                          (cudaStream_t)stream),
                    "swarm_gatstack_forward_large");
}

namespace {
// the stacked DQN gradient tile's own limits, for a cfg and spec that validate_stack accepts
int validate_stack_grad(const SwarmConfig& c, const SwarmStackSpec& spec) {
  if (c.n_agents < 2) return fail(SWARM_ERR_UNSUPPORTED, "the stacked DQN update needs n_agents >= 2");
  if (stack_grad_smem_bytes(c, spec) > 227 * 1024)
    return fail(SWARM_ERR_UNSUPPORTED, "the stacked DQN gradient tile exceeds 227 KB of shared memory for this (N, k, spec)");
  return SWARM_OK;
}

// the checks of swarm_gatstack_forward on a batch of n_graphs transitions, then the gradient tile's
int validate_dqn_stack(const SwarmConfig* cfg, const SwarmStackSpec* spec, int32_t n_graphs) {
  if (!cfg) return fail(SWARM_ERR_INVALID_ARG, "cfg is NULL");
  if (n_graphs <= 0) return fail(SWARM_ERR_INVALID_ARG, "n_graphs must be positive");
  if (cfg->n_agents > kTileThreads)
    return fail(SWARM_ERR_UNSUPPORTED, "the stacked DQN update is implemented for n_agents <= 128");
  SwarmConfig c = *cfg;
  c.num_envs = n_graphs;
  if (int rc = validate_stack(&c, spec)) return rc;
  return validate_stack_grad(c, *spec);
}
}  // namespace

int64_t swarm_dqn_stack_workspace_bytes(const SwarmConfig* cfg, const SwarmStackSpec* spec, int32_t n_graphs) {
  if (validate_dqn_stack(cfg, spec, n_graphs) != SWARM_OK) return 0;
  return stack_grad_workspace_bytes(*cfg, *spec, n_graphs);
}

int swarm_dqn_stack_grad(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* online_weights,
                         const float* target_weights, const SwarmReplay* batch, const int64_t* indices, int32_t n_graphs,
                         float gamma, float loss_scale, float* grad, float* loss, float* td, void* workspace,
                         int64_t workspace_bytes, void* stream) {
  if (int rc = validate_dqn_stack(cfg, spec, n_graphs)) return rc;
  if (!online_weights || !target_weights || !grad || !loss || !workspace) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (int rc = validate_ring(batch, "batch", false)) return rc;
  if (workspace_bytes < stack_grad_workspace_bytes(*cfg, *spec, n_graphs))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return check_cuda(launch_stack_grad(*cfg, *spec, online_weights, target_weights, *batch, indices, n_graphs, gamma,
                                      loss_scale, grad, loss, td, workspace, (cudaStream_t)stream),
                    "swarm_dqn_stack_grad");
}

int swarm_adam_clip_stack_step(const SwarmStackSpec* spec, float* weights, const float* grad, float* exp_avg,
                               float* exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                               double max_norm, float* target_weights, float* grad_norm, void* stream) {
  if (int rc = validate_spec(spec)) return rc;
  if (!weights || !grad || !exp_avg || !exp_avg_sq) return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (step < 1) return fail(SWARM_ERR_INVALID_ARG, "step is 1-based");
  if (int rc = validate_adam(lr, beta1, beta2, eps)) return rc;
  return check_cuda(launch_stack_adam_clip(*spec, weights, grad, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, max_norm,
                                           target_weights, grad_norm, (cudaStream_t)stream),
                    "swarm_adam_clip_stack_step");
}

int64_t swarm_rollout_stack_workspace_bytes(const SwarmConfig* cfg) {
  if (!cfg || cfg->num_envs <= 0 || cfg->n_agents <= 0) return 0;
  return rollout_stack_workspace(*cfg).bytes;
}

// the Flocking / Cohesion reward of the n_agents <= 128 stacked tick (reward == NULL: the world's own): checked, and
// copied into rs as one tick over every env reads it
static int stack_reward(const SwarmConfig* cfg, const SwarmRewardSpec* reward, const float* shaping, SwarmRewardSpec& rs) {
  if (!reward) return SWARM_OK;
  rs = *reward;
  rs.reset = 0;
  rs.env_index = -1;
  if (rs.kind != SWARM_REWARD_FLOCKING && rs.kind != SWARM_REWARD_COHESION)
    return fail(SWARM_ERR_INVALID_ARG, "unknown reward kind");
  if (int rc = validate_reward_cfg(cfg, rs, true)) return rc;
  return validate_reward_buffers(rs, shaping, false, nullptr);
}

// n_agents > 128: per tick [topk table ->] the large stacked forward (argmax) -> the large world step with returns / hits;
// rs != nullptr: the world step counts the hits only, and the large scenario reward adds the tick's reward to returns
// (its per-agent terms in w.reward)
static int rollout_stack_large(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, float* state,
                               int32_t ticks, float* returns, int32_t* hits, const RolloutWorkspace& w, cudaStream_t st,
                               const SwarmRewardSpec* rs = nullptr, float* shaping = nullptr) {
  const bool knn = cfg->graph_mode == SWARM_GRAPH_KNN;
  int32_t *actions = w.actions, *nbr = w.nbr;
  // in place: one CTA owns a whole env and stages its positions first
  SimStepArgs p = step_args(*cfg, state, actions, state);
  p.returns = rs ? nullptr : returns;
  p.hits = hits;
  for (int t = 0; t < ticks; ++t) {
    if (knn)
      if (cudaError_t e = launch_graph_large(*cfg, state, nullptr, nbr, (int)swarm_edges_per_env(cfg), st); e != cudaSuccess)
        return check_cuda(e, "swarm_rollout_stack (graph)");
    if (cudaError_t e = launch_gatstack_large(*cfg, *spec, weights, state, knn ? nbr : nullptr, nullptr, actions, w.forward, st);
        e != cudaSuccess)
      return check_cuda(e, "swarm_rollout_stack (forward)");
    if (cudaError_t e = launch_sim_step_large(p, st); e != cudaSuccess) return check_cuda(e, "swarm_rollout_stack (step)");
    if (rs)
      if (cudaError_t e = launch_scenario_reward_large(*rs, state, shaping, nullptr, nullptr, returns, w.reward, st);
          e != cudaSuccess)
        return check_cuda(e, "swarm_rollout_stack_large (reward)");
  }
  return SWARM_OK;
}

int swarm_rollout_stack(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, float* state,
                        int32_t ticks, const SwarmRewardSpec* reward, float* shaping, float* returns, int32_t* hits,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = validate_stack(cfg, spec, cfg && cfg->n_agents > kTileThreads)) return rc;
  const bool large = cfg->n_agents > kTileThreads;
  if (large && reward)
    return fail(SWARM_ERR_UNSUPPORTED, "the Flocking / Cohesion rewards are implemented for n_agents <= 128 "
                                       "(larger swarms: reward = NULL, the world's own reward)");
  if (!weights || !state || !workspace) return fail(SWARM_ERR_INVALID_ARG, "weights/state/workspace is NULL");
  if (ticks < 0) return fail(SWARM_ERR_INVALID_ARG, "ticks must be >= 0");
  const RolloutWorkspace w = rollout_stack_workspace(*cfg, workspace);
  if (workspace_bytes < w.bytes) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  if (large) return rollout_stack_large(cfg, spec, weights, state, ticks, returns, hits, w, (cudaStream_t)stream);
  SwarmRewardSpec rs;
  if (int rc = stack_reward(cfg, reward, shaping, rs)) return rc;
  // the whole loop is ONE launch with the state in registers (stack_kernels.cu gatstack_kernel<HP, true>)
  return check_cuda(launch_gatstack_rollout(*cfg, *spec, weights, state, ticks, world_consts(*cfg), reward ? &rs : nullptr,
                                            shaping, returns, hits, (cudaStream_t)stream),
                    "swarm_rollout_stack");
}

int64_t swarm_rollout_stack_large_workspace_bytes(const SwarmConfig* cfg, const SwarmRewardSpec* reward) {
  if (!cfg || cfg->num_envs <= 0 || cfg->n_agents <= kTileThreads || cfg->n_agents > kMaxLargeAgents) return 0;
  return rollout_stack_large_workspace(*cfg, reward).bytes;
}

int swarm_rollout_stack_large(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, float* state,
                              int32_t ticks, const SwarmRewardSpec* reward, float* shaping, float* returns,
                              int32_t* hits, void* workspace, int64_t workspace_bytes, void* stream) {
  if (int rc = validate_stack(cfg, spec, true)) return rc;
  if (cfg->n_agents <= kTileThreads)
    return fail(SWARM_ERR_UNSUPPORTED, "swarm_rollout_stack_large runs 129 <= n_agents <= 4096 (smaller swarms: "
                                       "swarm_rollout_stack)");
  if (!weights || !state || !workspace) return fail(SWARM_ERR_INVALID_ARG, "weights/state/workspace is NULL");
  if (ticks < 0) return fail(SWARM_ERR_INVALID_ARG, "ticks must be >= 0");
  SwarmRewardSpec rs;
  if (int rc = stack_reward(cfg, reward, shaping, rs)) return rc;
  if (reward && (int64_t)cfg->num_envs * cfg->n_agents >= (1LL << 31))
    return fail(SWARM_ERR_UNSUPPORTED, "num_envs * n_agents must stay below 2^31");
  const RolloutWorkspace w = rollout_stack_large_workspace(*cfg, reward, workspace);
  if (workspace_bytes < w.bytes) return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return rollout_stack_large(cfg, spec, weights, state, ticks, returns, hits, w, (cudaStream_t)stream,
                             reward ? &rs : nullptr, shaping);
}

// the checks of swarm_train_tick_stack and of its grad phase, in swarm_train_tick_stack's order (no_moments: the apply
// phase's exp_avg / exp_avg_sq are missing, reported with the other NULL arguments), and the reward spec copied into rs
static int validate_tick_stack(const SwarmConfig* cfg, const SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                               const SwarmRewardSpec* reward, const float* shaping, const SwarmTrainCtl* ctl,
                               const float* weights, const float* target_weights, bool no_moments, const float* state,
                               const SwarmReplay* ring, const float* grad, const void* workspace, int64_t workspace_bytes,
                               SwarmRewardSpec& rs) {
  if (int rc = validate_hyper(hyper)) return rc;
  if (int rc = validate_stack(cfg, spec)) return rc;      // the caller's cfg: its own num_envs must be positive
  if (int rc = validate_stack_grad(*cfg, *spec)) return rc;
  if (hyper->flocking)
    return fail(SWARM_ERR_INVALID_ARG, "hyper->flocking must be NULL: the stacked tick takes its reward as `reward`");
  if (!ctl || !weights || !target_weights || no_moments || !state || !grad || !workspace)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (int rc = validate_ring(ring, "replay ring", true)) return rc;
  if (cfg->num_envs > ring->capacity) return fail(SWARM_ERR_INVALID_ARG, "num_envs exceeds the replay capacity");
  if (workspace_bytes < stack_grad_workspace_bytes(*cfg, *spec, hyper->graphs_per_update))
    return fail(SWARM_ERR_INVALID_ARG, "workspace too small");
  return stack_reward(cfg, reward, shaping, rs);
}

// launches 1-3 of the stacked tick (peers != NULL: the reduce launch sums grad / loss over the ranks)
static int tick_stack_grad(const SwarmConfig* cfg, const SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                           const SwarmRewardSpec* rs, float* shaping, SwarmTrainCtl* ctl, const float* weights,
                           const float* target_weights, float* state, float* returns, int32_t* hits, const SwarmReplay* ring,
                           int64_t* indices, float* grad, void* workspace, const SwarmPeerExchange* peers, cudaStream_t st,
                           const char* what_rollout, const char* what_grad) {
  float* loss = grad + stack_weight_count_host(*spec);
  if (int rc = check_cuda(launch_gatstack_train_tick(*cfg, *spec, weights, state, world_consts(*cfg), rs, shaping, returns,
                                                     hits, *ring, ctl, hyper->rng_seed, hyper->env_offset, st),
                          what_rollout))
    return rc;
  return check_cuda(launch_stack_grad(*cfg, *spec, weights, target_weights, *ring, nullptr, hyper->graphs_per_update,
                                      hyper->gamma, hyper->loss_scale, grad, loss, nullptr, workspace, st, ctl, indices,
                                      hyper->sample_seed, cfg->num_envs, peers),
                    what_grad);
}

// launch 4 of the stacked tick
static int tick_stack_apply(const SwarmConfig* cfg, const SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                            SwarmTrainCtl* ctl, float* weights, float* target_weights, float* exp_avg, float* exp_avg_sq,
                            const float* grad, int64_t ring_capacity, cudaStream_t st, const char* what) {
  return check_cuda(launch_stack_adam_clip(*spec, weights, grad, exp_avg, exp_avg_sq, 1, hyper->lr, hyper->beta1,
                                           hyper->beta2, hyper->eps, hyper->max_norm, target_weights, nullptr, st, ctl,
                                           cfg->num_envs, ring_capacity, hyper->update_target_every),
                    what);
}

int swarm_train_tick_stack(const SwarmConfig* cfg, const SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                           const SwarmRewardSpec* reward, float* shaping, SwarmTrainCtl* ctl, float* weights,
                           float* target_weights, float* exp_avg, float* exp_avg_sq, float* state, float* returns,
                           int32_t* hits, const SwarmReplay* ring, int64_t* indices, float* grad, void* workspace,
                           int64_t workspace_bytes, void* stream) {
  SwarmRewardSpec rs;
  if (int rc = validate_tick_stack(cfg, spec, hyper, reward, shaping, ctl, weights, target_weights, !exp_avg || !exp_avg_sq,
                                   state, ring, grad, workspace, workspace_bytes, rs))
    return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = tick_stack_grad(cfg, spec, hyper, reward ? &rs : nullptr, shaping, ctl, weights, target_weights, state,
                               returns, hits, ring, indices, grad, workspace, nullptr, st, "swarm_train_tick_stack(rollout)",
                               "swarm_train_tick_stack(grad)"))
    return rc;
  return tick_stack_apply(cfg, spec, hyper, ctl, weights, target_weights, exp_avg, exp_avg_sq, grad, ring->capacity, st,
                          "swarm_train_tick_stack(apply)");
}

int swarm_train_tick_stack_grad(const SwarmConfig* cfg, const SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                                const SwarmRewardSpec* reward, float* shaping, SwarmTrainCtl* ctl, const float* weights,
                                const float* target_weights, float* state, float* returns, int32_t* hits,
                                const SwarmReplay* ring, int64_t* indices, float* grad, void* workspace,
                                int64_t workspace_bytes, const SwarmPeerExchange* peers, void* stream) {
  SwarmRewardSpec rs;
  if (int rc = validate_tick_stack(cfg, spec, hyper, reward, shaping, ctl, weights, target_weights, false, state, ring,
                                   grad, workspace, workspace_bytes, rs))
    return rc;
  if (int rc = validate_peers(peers)) return rc;
  return tick_stack_grad(cfg, spec, hyper, reward ? &rs : nullptr, shaping, ctl, weights, target_weights, state, returns,
                         hits, ring, indices, grad, workspace, peers, (cudaStream_t)stream,
                         "swarm_train_tick_stack_grad(rollout)", "swarm_train_tick_stack_grad(grad)");
}

int swarm_train_tick_stack_apply(const SwarmConfig* cfg, const SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                                 SwarmTrainCtl* ctl, float* weights, float* target_weights, float* exp_avg,
                                 float* exp_avg_sq, const float* grad, int64_t ring_capacity, void* stream) {
  if (int rc = validate_hyper(hyper)) return rc;
  if (int rc = validate_stack(cfg, spec)) return rc;
  if (int rc = validate_stack_grad(*cfg, *spec)) return rc;
  if (hyper->flocking)
    return fail(SWARM_ERR_INVALID_ARG, "hyper->flocking must be NULL: the stacked tick takes its reward as `reward`");
  if (!ctl || !weights || !target_weights || !exp_avg || !exp_avg_sq || !grad)
    return fail(SWARM_ERR_INVALID_ARG, "NULL argument");
  if (cfg->num_envs > ring_capacity) return fail(SWARM_ERR_INVALID_ARG, "num_envs exceeds the replay capacity");
  return tick_stack_apply(cfg, spec, hyper, ctl, weights, target_weights, exp_avg, exp_avg_sq, grad, ring_capacity,
                          (cudaStream_t)stream, "swarm_train_tick_stack_apply");
}

int swarm_episode_end(const SwarmConfig* cfg, SwarmTrainCtl* ctl, float* returns, int32_t* hits, const float* loss,
                      float* stats, int64_t max_episodes, double epsilon0, double epsilon_decay, double min_epsilon,
                      void* stream) {
  if (int rc = validate(cfg, false, true)) return rc;
  if (!ctl || !returns) return fail(SWARM_ERR_INVALID_ARG, "ctl/returns is NULL");
  if (stats && max_episodes <= 0) return fail(SWARM_ERR_INVALID_ARG, "max_episodes must be positive when stats is given");
  return check_cuda(launch_episode_end(*cfg, ctl, returns, hits, loss, stats, max_episodes, epsilon0, epsilon_decay,
                                       min_epsilon, (cudaStream_t)stream),
                    "swarm_episode_end");
}

}  // extern "C"
