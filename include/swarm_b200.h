/*
 * swarm_b200.h -- C ABI of the B200-native swarm hot path.
 *
 * The reference (davidedomini/experiments-2025-acsos-marl-for-swarming-behaviors) has no FFI boundary:
 * it is in-process Python on top of vmas==1.4.0 and torch_geometric==2.5.3.  These entry points are
 * what a binding for its hot path would call; each one names the reference code it replaces
 * (paths relative to the reference repository root).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in `_host`;
 *     the library never allocates, frees or keeps caller memory, and has no global mutable state
 *     apart from the thread-local error string;
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it and never
 *     synchronise the host;
 *   - return value 0 = OK; negative = error (SWARM_ERR_*), message via swarm_last_error();
 *   - layouts: state   float[B*N][4] = (x, y, vx, vy) of agent i of env b at index b*N+i
 *              actions int32[B*N], rewards float[B*N]
 *              edges   int32[B][2][E] env-local node ids, row 0 = source, row 1 = target
 *              weights float[1673], packed in SWARM_W_* order (all row-major as in the state dict)
 */
#ifndef SWARM_B200_H
#define SWARM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWARM_ABI_VERSION 9

enum { SWARM_SCENARIO_GOTO = 0, SWARM_SCENARIO_OBSTACLE_AVOIDANCE = 1 };
/* SWARM_GRAPH_RADIUS is an EXTENSION (the reference has no radius graph, SURVEY.md Appendix C): the complete-graph
 * builder of train_gcn_dqn.py:94-110 filtered by distance -- for i < j with ||p_j - p_i|| <= graph_radius (float32
 * norm as in simulator.py:18) the edges (i -> j), (j -> i), in (i, j) order, then the trailing (0 -> 0).  With an
 * infinite radius it reproduces the complete graph edge for edge. */
enum { SWARM_GRAPH_COMPLETE = 0, SWARM_GRAPH_KNN = 1, SWARM_GRAPH_RADIUS = 2 };
enum {
  SWARM_OK = 0,
  SWARM_ERR_INVALID_ARG = -1,
  SWARM_ERR_UNSUPPORTED = -2,
  SWARM_ERR_CUDA = -3
};

/* packed Q-network weights: offsets (in floats) of the state-dict tensors of
 * src/training/train_gcn_dqn.py:50-57 (GATConv(7,32) + Linear(32,32) + Linear(32,9)) */
enum {
  SWARM_W_CONV_LIN = 0,       /* conv1.lin.weight [32][7]  */
  SWARM_W_ATT_SRC = 224,      /* conv1.att_src    [32]     */
  SWARM_W_ATT_DST = 256,      /* conv1.att_dst    [32]     */
  SWARM_W_CONV_BIAS = 288,    /* conv1.bias       [32]     */
  SWARM_W_LIN1 = 320,         /* lin1.weight      [32][32] */
  SWARM_W_LIN1_BIAS = 1344,   /* lin1.bias        [32]     */
  SWARM_W_LIN2 = 1376,        /* lin2.weight      [9][32]  */
  SWARM_W_LIN2_BIAS = 1664,   /* lin2.bias        [9]      */
  SWARM_W_COUNT = 1673
};
enum { SWARM_FEAT = 7, SWARM_HIDDEN = 32, SWARM_ACTIONS = 9, SWARM_OBS = 6 };

/* per-agent flag bits written by swarm_sim_step / swarm_rollout traces */
enum {
  SWARM_FLAG_OBSTACLE_CONTACT = 1, /* centre distance to the obstacle <= r_a + r_o (vmas collides()) */
  SWARM_FLAG_HIT = 2,              /* get_distance <= hit_distance (obstacle_avoidance_scenario.py:170-173) */
  SWARM_FLAG_PENALTY = 4           /* get_distance <= penalty_distance (obstacle_avoidance_scenario.py:149) */
};

/* World + scenario constants.  swarm_default_config() fills the values the reference runs with:
 * vmas World defaults (dt .1, drag .25, collision_force 100, contact_margin 1e-3, sphere radius .05)
 * and the scenario constants of src/scenarios/{go_to_position,obstacle_avoidance}_scenario.py. */
typedef struct SwarmConfig {
  double grid_spacing;     /* desired_distance (go_to:17 / oa:23); a Python double in generate_grid */
  int32_t num_envs;        /* B */
  int32_t n_agents;        /* N */
  int32_t scenario;        /* SWARM_SCENARIO_* */
  int32_t graph_mode;      /* SWARM_GRAPH_* */
  int32_t knn_k;           /* k of simulator.py:19 (10 shipped, 5 in the goldens) */
  float dt;
  float drag;
  float collision_force;
  float contact_margin;
  float agent_radius;
  float landmark_radius;
  float goal_x, goal_y;            /* go_to:86, oa:97 */
  float obstacle_x, obstacle_y;    /* oa:99 */
  float hit_distance;              /* oa:25 */
  float penalty_distance;          /* oa:24 */
  float obstacle_weight;           /* oa:136 */
  float graph_radius;              /* SWARM_GRAPH_RADIUS only */
} SwarmConfig;

/* optional per-tick traces of swarm_rollout (any pointer may be NULL); T = ticks */
typedef struct SwarmTrace {
  float* state;          /* [T][B*N][4] state AFTER each tick                              */
  int32_t* actions;      /* [T][B*N]    greedy / injected action used at each tick          */
  float* q;              /* [T][B*N][9] Q-values computed at each tick (pre-step state)     */
  float* rewards;        /* [T][B*N]                                                        */
  uint8_t* flags;        /* [T][B*N]    SWARM_FLAG_* after each tick                        */
  uint32_t* contact;     /* [T][B*N]    bit j = agent-agent contact with agent j (N <= 32)  */
  int32_t* edges;        /* [T][B][2][E] graph built at each tick                           */
  float* dist;           /* [T][B*N][2] (distance_to_goal, get_distance to the obstacle) after each tick */
} SwarmTrace;

int swarm_abi_version(void);
const char* swarm_last_error(void);
void swarm_default_config(SwarmConfig* cfg, int32_t scenario, int32_t num_envs, int32_t n_agents);
/* number of edges per env for cfg->graph_mode: N(N-1)+1 (train_gcn_dqn.py:101-108) or 2kN+1 (simulator.py:15-24);
 * for SWARM_GRAPH_RADIUS the CAPACITY N(N-1)+1 of the padded per-env edge block */
int64_t swarm_edges_per_env(const SwarmConfig* cfg);

/* generate_grid + reset_world_at (go_to:52-106, oa:63-133): agents on the row-major grid around
 * centers[b] (float[B][2]; the caller draws them -- the reference draws one torch.normal per reset),
 * velocities zero. */
int swarm_reset_grid(const SwarmConfig* cfg, const float* centers, float* state, void* stream);

/* One vmas Environment.step (call sites train_gcn_dqn.py:169, simulator.py:68): action decode,
 * contact forces (obstacle first, then agent pairs in entity order), drag + semi-implicit Euler, then
 * the scenario's reward()/observation() and the obstacle flags.  Optional outputs may be NULL:
 * rewards float[B*N], flags uint8[B*N], contact uint32[B*N] (N <= 32 only), obs float[B*N][6],
 * dist float[B*N][2] = (agent.distance_to_goal, world.get_distance(agent, obstacle)) -- the per-agent terms
 * behind average_distance_to_goal() / average_distance_to_obstacles() (oa:164-168).  state_out may alias
 * state_in. */
int swarm_sim_step(const SwarmConfig* cfg, const float* state_in, const int32_t* actions, float* state_out,
                   float* rewards, uint8_t* flags, uint32_t* contact, float* obs, float* dist, void* stream);

/* Graph builders: train_gcn_dqn.py:94-110 (complete) and simulator.py:9-26 (symmetrised kNN with
 * torch.topk tie order).  edges int32[B][2][E]; neighbours (optional, kNN only) int32[B*N][k] holds the
 * topk index row of every agent. */
int swarm_graph_build(const SwarmConfig* cfg, const float* state, int32_t* edges, int32_t* neighbours,
                      void* stream);

/* Radius graph (extension, see SWARM_GRAPH_RADIUS): edges int32[B][2][N(N-1)+1], the first counts[b] columns of env b
 * hold its edge list, the rest is -1; counts int32[B] (always odd: pairs come as (i -> j), (j -> i), plus (0 -> 0)).
 * The per-env list is compacted in shared memory: every agent counts its partners j > i in range, an exclusive
 * prefix sum over the env's agents gives its write offset.  n_agents <= 128. */
int swarm_graph_build_radius(const SwarmConfig* cfg, const float* state, int32_t* edges, int32_t* counts, void* stream);

/* Radius graph of a swarm of ANY size (n_agents <= 4096) in compact CSR form, grouped by target -- the large-swarm
 * counterpart of swarm_graph_build_radius, whose padded N(N-1)+1 block would be 8 MB per env at N = 1024.  Same edge set
 * and order as the edge list (i -> j), (j -> i) for i < j within cfg->graph_radius (rounded float32 2-norm, inclusive),
 * then (0 -> 0), after a stable sort by target: the sources of a node ascend, node 0's self loop comes last.
 * Candidates come from a uniform grid (cells one radius wide, at most 64 x 64 over the env's bounding box, agents sorted
 * by (cell, index) in shared memory; a node looks at its 3 x 3 cells), membership from the exact distance test.
 * Two passes on the same state:
 *   count: degree int32[B*N] != NULL, row_ptr = src = NULL   -> in-degree of every node
 *   fill:  degree = NULL, row_ptr int32[B*N+1] = exclusive prefix sum of the degrees (the caller's scan), src int32[E]
 *          -> GLOBAL source ids b*N + j.  (row_ptr, src) feed swarm_gatq_forward_csr / swarm_gatq_backward_csr with
 *          n_nodes = B*N directly. */
int swarm_graph_build_radius_csr(const SwarmConfig* cfg, const float* state, int32_t* degree, const int32_t* row_ptr,
                                 int32_t* src, void* stream);

/* GCN.forward (train_gcn_dqn.py:59-70) + argmax for LARGE swarms on the radius graph (sources from the uniform grid
 * above) or the complete graph (train:94-110: every other agent, node 0 also itself) without materialising an edge
 * list -- the complete graph of 1 024 agents is 1 047 553 edges per env.  One CTA per env, attention in input space
 * (GATConv's projection is linear and bias-free: softmax-weighted mean of the sources' 7 input features, then one
 * projection), 20 B of shared memory per agent (+ 4 B + 16 KB for the grid): n_agents <= 4096.  Same mathematics as
 * swarm_gatq_forward_csr on the same graph with float32-level different rounding (no fixed edge order); any n_agents
 * >= 1 is accepted.  q float[B*N][9] and actions int32[B*N] are optional. */
int swarm_gatq_forward_large(const SwarmConfig* cfg, const float* weights, const float* state, float* q,
                             int32_t* actions, void* stream);

/* GCN.forward (train_gcn_dqn.py:59-70) on the per-env graph named by cfg->graph_mode, node features
 * [pos, vel, goal, agent id] built from state (train:95-99).  q float[B*N][9] and actions int32[B*N]
 * (argmax, first maximum wins; train:167, simulator:64) are optional. */
int swarm_gatq_forward(const SwarmConfig* cfg, const float* weights, const float* state, float* q,
                       int32_t* actions, void* stream);

/* GCN.forward on an arbitrary graph: x float[n][7]; edges grouped by target in CSR form, each group in
 * edge-list order (row_ptr int32[n+1], src int32[E]).  Used by the nn.Module seam (train_gcn_dqn.py:59-70)
 * for arbitrary Data/Batch inputs and the Q-network path of large swarms (n_agents > 128).  q float[n][9] and
 * actions int32[n] (argmax) are optional.  workspace: swarm_gatq_workspace_bytes(n) bytes of device memory. */
int64_t swarm_gatq_workspace_bytes(int32_t n_nodes);
int swarm_gatq_forward_csr(int32_t n_nodes, const float* weights, const float* x, const int32_t* row_ptr,
                           const int32_t* src, float* q, int32_t* actions, void* workspace, int64_t workspace_bytes,
                           void* stream);

/* Stable grouping of an edge list by target (the order scatter-add sees): edge_src/edge_dst int64[E]
 * (torch_geometric edge_index rows) -> row_ptr int32[n+1], src int32[E], perm int32[E] (perm[p] = position
 * in the input list of grouped edge p).  workspace: swarm_csr_workspace_bytes(n, E) bytes.  An edgeless graph
 * (E = 0, e.g. a single agent) is valid: the edge arrays may then be NULL and row_ptr is all zeros. */
int64_t swarm_csr_workspace_bytes(int32_t n_nodes, int64_t n_edges);
int swarm_csr_from_edges(int32_t n_nodes, int64_t n_edges, const int64_t* edge_src, const int64_t* edge_dst,
                         int32_t* row_ptr, int32_t* src, int32_t* perm, void* workspace, int64_t workspace_bytes,
                         void* stream);

/* GCN.forward on the symmetrised kNN graph of large swarms (n_agents > 128) straight from the topk table that
 * swarm_graph_build returns in `neighbours` (int32[B][N][k]): one CTA per env builds the in-edge lists in shared memory
 * (same edge-list order as swarm_graph_build + swarm_csr_from_edges + swarm_gatq_forward_csr, same Q bit for bit) without
 * materialising the edge list.  Needs N * (144 + 4k) + 7.4 K bytes of shared memory (n_agents <= ~1 200 for k = 10); larger swarms
 * use the generic CSR path.  q float[B*N][9] and actions int32[B*N] are optional. */
int swarm_gatq_forward_knn_large(const SwarmConfig* cfg, const float* weights, const float* state,
                                 const int32_t* neighbours, float* q, int32_t* actions, void* stream);

/* (graph_mode RADIUS / COMPLETE: the per-tick sequence is swarm_gatq_forward_large + the world step -- two launches --
 * and SWARM_TC has no effect; everything else below applies.) */
/* `ticks` greedy evaluation ticks of a LARGE kNN swarm (n_agents > 128; simulator.py:59-93 with the shipped kNN graph)
 * launched back to back from the library: per tick the topk table (swarm_graph_build), the Q forward + argmax straight
 * from the table (swarm_gatq_forward_knn_large) and the world step, whose kernel also accumulates returns float[B*N] (+=)
 * and hits int32[B] (+=), both optional.  state float[B][N][4] is advanced in place.  No host work, no allocation and
 * no tensor-library op between the launches (the loop is CUDA-graph capturable).  The Q forward attends in input space
 * (GATConv's projection is linear: weighted mean of the neighbours' 7 input features, then one projection), which needs
 * 28 + 2k bytes of shared memory per agent, so envs up to 4 096 agents fit; its greedy actions equal those of
 * swarm_gatq_forward_knn_large except at float32 near-ties, and SWARM_TC=0 selects that bit-faithful forward (then the
 * env must fit its 144 + 4k bytes per agent).  64 k <= n_agents as for swarm_graph_build. */
int64_t swarm_rollout_large_workspace_bytes(const SwarmConfig* cfg);
int swarm_rollout_large(const SwarmConfig* cfg, const float* weights, float* state, int32_t ticks, float* returns,
                        int32_t* hits, void* workspace, int64_t workspace_bytes, void* stream);

/* Backward pass of GCN.forward on an arbitrary graph (loss.backward() through the nn.Module, train_gcn_dqn.py:116-124
 * when a script drives the module with torch autograd): grad_q float[n][9] -> grad_weights float[1673] (overwritten).
 * The graph is given twice, grouped by target (row_ptr / src / perm, as for the forward) and grouped by source
 * (row_ptr_s / tgt_s / perm_s = swarm_csr_from_edges with the two edge rows swapped); perm arrays map grouped
 * positions to edge-list positions.  Gathers only, fixed summation order (bit-reproducible).
 * workspace: swarm_gatq_backward_workspace_bytes(n, E). */
int64_t swarm_gatq_backward_workspace_bytes(int32_t n_nodes, int64_t n_edges);
int swarm_gatq_backward_csr(int32_t n_nodes, int64_t n_edges, const float* weights, const float* x,
                            const int32_t* row_ptr, const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                            const int32_t* tgt_s, const int32_t* perm_s, const float* grad_q, float* grad_weights,
                            void* workspace, int64_t workspace_bytes, void* stream);

/* The GATConv layer alone (torch_geometric.nn.GATConv(7, 32, heads=1, add_self_loops=False) as the reference's GCN
 * class calls it, train_gcn_dqn.py:53,61): out float[n][32] = softmax-weighted aggregate + bias, and its backward pass
 * (grad_out float[n][32] -> the conv1.* segments of grad_weights float[1673]; the other segments are zero).  Same
 * graph arguments, workspaces (swarm_gatq_workspace_bytes / swarm_gatq_backward_workspace_bytes) and determinism as
 * the whole-network calls above; only the conv1.* entries of `weights` are read. */
int swarm_gatconv_forward_csr(int32_t n_nodes, const float* weights, const float* x, const int32_t* row_ptr,
                              const int32_t* src, float* out, void* workspace, int64_t workspace_bytes, void* stream);
int swarm_gatconv_backward_csr(int32_t n_nodes, int64_t n_edges, const float* weights, const float* x,
                               const int32_t* row_ptr, const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                               const int32_t* tgt_s, const int32_t* perm_s, const float* grad_out, float* grad_weights,
                               void* workspace, int64_t workspace_bytes, void* stream);

/* One single-head GATConv layer of any small width (EXTENSION towards SURVEY.md 8f rank 4, multi-layer attention
 * networks such as the three 8-wide layers of the reference's data/models/experiment_Flocking-seed_*.pth):
 * torch_geometric.nn.GATConv(in_channels, out_channels, heads=1, add_self_loops=False, bias=True), 1 <= in_channels,
 * out_channels <= 64, on an arbitrary graph given as for swarm_gatq_forward_csr / swarm_gatq_backward_csr.
 *   forward : lin_weight float[out][in], att_src / att_dst / bias float[out], x float[n][in] -> out float[n][out]
 *   backward: grad_out float[n][out] -> grad_lin_weight, grad_att_src, grad_att_dst, grad_bias (overwritten) and,
 *             when grad_x != NULL, grad_x float[n][in] -- so layers can be stacked under torch autograd.
 * Gather-only with fixed reduction orders: results are bit-reproducible.  Workspace in bytes from
 * swarm_gat_layer_workspace_bytes(n, E, in, out, backward != 0). */
int64_t swarm_gat_layer_workspace_bytes(int32_t n_nodes, int64_t n_edges, int32_t in_channels, int32_t out_channels,
                                        int32_t backward);
int swarm_gat_layer_forward(int32_t n_nodes, int32_t in_channels, int32_t out_channels, const float* lin_weight,
                            const float* att_src, const float* att_dst, const float* bias, const float* x,
                            const int32_t* row_ptr, const int32_t* src, float* out, void* workspace,
                            int64_t workspace_bytes, void* stream);
int swarm_gat_layer_backward(int32_t n_nodes, int64_t n_edges, int32_t in_channels, int32_t out_channels,
                             const float* lin_weight, const float* att_src, const float* att_dst, const float* x,
                             const int32_t* row_ptr, const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                             const int32_t* tgt_s, const int32_t* perm_s, const float* grad_out, float* grad_lin_weight,
                             float* grad_att_src, float* grad_att_dst, float* grad_bias, float* grad_x, void* workspace,
                             int64_t workspace_bytes, void* stream);

/* Device replay ring of whole-swarm transitions (GraphReplayBuffer, train_gcn_dqn.py:25-48, capacity 1e6 at
 * train:86).  Only the world state is stored (37 B per agent and transition); node features and graphs are
 * rebuilt from it on the fly. */
typedef struct SwarmReplay {
  float* state;          /* [capacity][N][4] s                      */
  float* next_state;     /* [capacity][N][4] s'                     */
  uint8_t* actions;      /* [capacity][N]    a                      */
  float* rewards;        /* [capacity][N]    r                      */
  int64_t capacity;      /* slots (one slot = one env transition)   */
} SwarmReplay;

struct SwarmRewardSpec;          /* defined with swarm_scenario_reward below */

typedef struct SwarmRolloutOptions {
  const int32_t* forced_actions; /* optional [ticks][B*N]; entries >= 0 override the policy's action        */
  float epsilon;                 /* epsilon-greedy (train:164-167): one coin per env and tick; 0 = greedy   */
  uint64_t rng_seed;             /* counter-based device RNG stream (seed, env, tick0 + tick)               */
  int64_t rng_tick0;
  const SwarmReplay* replay;     /* optional: push (s, a, r, s') of every env and tick (train:171-172) ...  */
  int64_t replay_cursor;         /* ... at slot (cursor + tick*B + env) mod capacity                        */
  int64_t env_offset;            /* global index of env 0 (RNG streams of an env shard)                     */
  /* Flocking (flocking_scenario.py:124-171) on the fused path: with `flocking` set (kind SWARM_REWARD_FLOCKING,
   * cfg->scenario SWARM_SCENARIO_GOTO, whose world Flocking shares) every tick's reward -- returns, reward trace,
   * replay push -- is the Flocking collective reward, evaluated exactly like swarm_scenario_reward after each world
   * step; flocking_shaping float[B*N][2] is read at the start and written back at the end (initialise it with a
   * swarm_scenario_reward reset call after placing the agents). */
  const struct SwarmRewardSpec* flocking;
  float* flocking_shaping;
  /* kNN graph, n_agents <= 12, tensor-core path without an edge trace: the Q forward consumes the kNN graph as in-edge
   * multiplicities, so only the SET of each row's k neighbours is needed; it is unique unless a tie straddles the k
   * boundary, and only those rows need torch.topk's algorithm (libstdc++ introselect, emulated step for step).  Its
   * answer is a function of the row's order pattern alone, so it can be memoised: knn_memo uint64[knn_memo_entries]
   * (optional; entries a power of two; zero-initialised by the caller, then owned by the library's kernels: a lossy
   * direct-mapped table, one word per entry = 48-bit order pattern | 16-bit neighbour set) is shared by every CTA and
   * may be kept across launches.  ONE table per (n_agents, knn_k) pair.  Results do not depend on its contents. */
  uint64_t* knn_memo;
  int64_t knn_memo_entries;
} SwarmRolloutOptions;

/* Fused rollout: `ticks` iterations of [graph build -> GCN forward -> (epsilon-)greedy argmax -> env step]
 * (the inner loops of simulator.py:59-93 and train_gcn_dqn.py:153-178) with the state resident on chip.
 * state is updated in place; returns float[B*N] accumulates each agent's rewards (+=), hits int32[B]
 * accumulates obstacles_hits() per tick (+=); opts, returns, hits and trace are optional. */
int swarm_rollout(const SwarmConfig* cfg, const float* weights, float* state, int32_t ticks,
                  const SwarmRolloutOptions* opts, float* returns, int32_t* hits, const SwarmTrace* trace,
                  void* stream);

/* GraphReplayBuffer.push for B envs at once (train:32-36): slots (cursor + b) mod capacity. */
int swarm_replay_push(const SwarmConfig* cfg, const SwarmReplay* replay, int64_t cursor, const float* state,
                      const int32_t* actions, const float* rewards, const float* next_state, void* stream);

/* GraphReplayBuffer.sample materialisation (train:38-45): gathers n_graphs slots (indices int64[n_graphs])
 * into dense arrays state/next_state float[n_graphs][N][4], actions int32[n_graphs][N], rewards
 * float[n_graphs][N]. */
int swarm_replay_gather(const SwarmConfig* cfg, const SwarmReplay* replay, const int64_t* indices,
                        int32_t n_graphs, float* state, int32_t* actions, float* rewards, float* next_state,
                        void* stream);

/* One DQN loss + gradient (train_step_dqn, train_gcn_dqn.py:116-124) over n_graphs whole-swarm transitions
 * taken from `batch` (slot g, or slot indices[g] when indices != NULL): values = Q_online(s)[a], targets =
 * r + gamma * max_a Q_target(s') (no terminal mask), loss = mean((values - targets)^2) over all
 * n_graphs*N nodes, gradient w.r.t. the 1673 online weights by a hand-written backward pass (deterministic:
 * per-CTA partial sums reduced in a fixed order, no atomics).  cfg->graph_mode selects the per-env graph;
 * cfg->num_envs is ignored.  `loss_scale` multiplies the loss (1/total node count; pass the global count when
 * the batch is one shard of a distributed update).  Outputs: grad float[1673], loss float[1] (both
 * overwritten); td (optional) float[n_graphs*N] = values - targets.  workspace:
 * swarm_dqn_workspace_bytes(cfg, n_graphs). */
int64_t swarm_dqn_workspace_bytes(const SwarmConfig* cfg, int32_t n_graphs);
int swarm_dqn_grad(const SwarmConfig* cfg, const float* online_weights, const float* target_weights,
                   const SwarmReplay* batch, const int64_t* indices, int32_t n_graphs, float gamma,
                   float loss_scale, float* grad, float* loss, float* td, void* workspace,
                   int64_t workspace_bytes, void* stream);

/* clip_grad_norm_(params, max_norm) + Adam step (train:125-126; torch.optim.Adam defaults lr 1e-3,
 * betas (0.9, 0.999), eps 1e-8) on the packed weights, in place; exp_avg / exp_avg_sq float[1673];
 * `step` is the 1-based step count.  The gradient norm follows torch: per-tensor 2-norms, then the 2-norm
 * of those; clip coefficient max_norm / (norm + 1e-6), clamped to 1.  If target_weights != NULL the updated
 * weights are also copied there (target_model.load_state_dict, train:131-133).  grad_norm (optional)
 * float[1] receives the pre-clip norm.  max_norm <= 0 disables clipping. */
int swarm_adam_clip_step(float* weights, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t step,
                         double lr, double beta1, double beta2, double eps, double max_norm,
                         float* target_weights, float* grad_norm, void* stream);

/* ---- device-driven train tick -------------------------------------------------------------------------------
 * One tick of the training loop body (train_gcn_dqn.py:153-178): act (epsilon-greedy on Q_online) -> env step ->
 * replay push -> sample -> TD target / loss / backward -> clip + Adam (-> hard target sync).  Everything that
 * changes from tick to tick (tick number, ring cursor / fill, optimiser step, epsilon) lives in a small DEVICE
 * struct that the kernels read and the last kernel advances, so the host never has to know the tick number:
 * the launches of one or many ticks can be captured once in a CUDA graph and replayed.
 * The tick is split in two calls so that a data-parallel trainer can all-reduce `grad` / `loss` in between. */
typedef struct SwarmTrainCtl {   /* device memory, 48 bytes, zero-initialised by the caller */
  int64_t tick;          /* ticks completed (the tick being executed is tick + 1, like `ticks += 1` at train:155)   */
  int64_t ring_cursor;   /* next replay slot                                                                        */
  int64_t ring_size;     /* filled replay slots                                                                     */
  int64_t opt_step;      /* optimiser steps done                                                                    */
  float epsilon;         /* exploration rate of the running episode (the host rewrites it between episodes)         */
  int32_t updating;      /* set by swarm_train_tick_grad: 1 if the ring holds >= graphs_per_update slots (train:113) */
  int64_t episode;       /* episodes completed (advanced by swarm_episode_end)                                      */
} SwarmTrainCtl;

typedef struct SwarmTrainHyper {
  double lr, beta1, beta2, eps, max_norm;   /* torch.optim.Adam defaults + clip_grad_norm_ max_norm (train:85,125)  */
  uint64_t rng_seed;            /* exploration stream (same stream as swarm_rollout's)                              */
  uint64_t sample_seed;         /* replay sampling stream                                                           */
  int64_t env_offset;           /* global index of env 0 of this shard                                              */
  int32_t graphs_per_update;    /* G (reference: 32, train:175)                                                     */
  int32_t update_target_every;  /* hard target sync period in ticks (reference: 200, train:175)                     */
  float gamma;                  /* 0.99                                                                             */
  float loss_scale;             /* 1 / (global number of nodes in the update batch)                                 */
  /* optional, as in SwarmRolloutOptions: the tick's reward is the Flocking collective reward (cfg = the GoTo world) */
  const struct SwarmRewardSpec* flocking;
  float* flocking_shaping;
} SwarmTrainHyper;

/* Phase 1: rollout tick of all cfg->num_envs envs with the online weights (pushes B transitions at ctl->ring_cursor),
 * draws graphs_per_update slot indices uniformly and independently (i.e. with replacement; the reference's
 * random.sample draws without) from the filled part of the ring (counter RNG keyed by (sample_seed, tick, g);
 * exported to indices int64[G] when indices != NULL), then gradient + loss of the update
 * batch as swarm_dqn_grad.
 * workspace: swarm_dqn_workspace_bytes(cfg, G).  If the ring holds fewer than G slots, grad / loss are left
 * untouched and ctl->updating = 0 (the reference prints "Not enough samples" and skips, train:113-115). */
int swarm_train_tick_grad(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl,
                          const float* weights, const float* target_weights, float* state, float* returns,
                          int32_t* hits, const SwarmReplay* ring, int64_t* indices, float* grad, float* loss,
                          void* workspace, int64_t workspace_bytes, void* stream);

/* Optional peer exchange for swarm_train_tick_apply: a one-shot PUSH all-reduce of the gradient over NVLink / NVSwitch
 * peer memory fused into the clip + Adam kernel (replaces the separate NCCL all-reduce launch of a data-parallel tick).
 * data[r] is THIS process's mapping of rank r's symmetric receive buffer (e.g. from
 * torch.distributed._symmetric_memory): uint64[2][world_size][SWARM_XCHG_STRIDE], zero-initialised -- slot
 * [parity of tick + 1][source rank].  Every rank writes its partial gradient + loss into its slot of EVERY rank's buffer
 * as 8-byte words (epoch = tick + 1 in the high half, the float in the low half: the word is its own arrival flag), then
 * waits on its own (local) buffer and sums the world_size partials in rank order -- the same order on every rank, so the
 * weights stay bit-identical across ranks without a broadcast.  All ranks must run the same number of envs and start
 * from the same ring fill (they must agree on which ticks update). */
enum { SWARM_MAX_PEERS = 16, SWARM_XCHG_STRIDE = 1680 };
typedef struct SwarmPeerExchange {
  uint64_t* data[SWARM_MAX_PEERS];
  int32_t world_size;
  int32_t rank;
} SwarmPeerExchange;

/* Phase 2: clip_grad_norm_ + Adam on `grad` (bias corrections from ctl->opt_step + 1), target <- online when
 * (ctl->tick + 1) % update_target_every == 0, then ctl advances: tick += 1, ring_cursor / ring_size += B,
 * opt_step += updating.  `grad` is float[1674] = gradient followed by the loss (the layout swarm_train_tick_grad
 * writes when grad and loss are adjacent); with `peers` != NULL both are first summed over the ranks (see above) and
 * the reduced values are written back to `grad`. */
int swarm_train_tick_apply(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl, float* weights,
                           float* target_weights, float* exp_avg, float* exp_avg_sq, float* grad,
                           int64_t ring_capacity, const SwarmPeerExchange* peers, void* stream);

/* Both phases as one call, for trainers that need nothing between them (one GPU, or the fused peer exchange): the same
 * loop body (train_gcn_dqn.py:153-178) and the same bits as swarm_train_tick_grad followed by swarm_train_tick_apply.
 * On one GPU, when the gradient kernel ran on at most 64 CTAs (the reference's 32 graphs per update: one CTA each), the
 * two small launches at the end of the tick (sum of the gradient kernel's per-CTA partials; clip + Adam) run as ONE
 * thread-block cluster -- the partials are summed in CTA order as before, the sums are exchanged through
 * distributed shared memory, every CTA forms the clip coefficient in the same order and steps its 256 elements --
 * three launches per tick instead of four.  `grad` is float[1674] (gradient followed by the loss; written for the
 * caller's statistics, summed over the ranks with `peers`); `workspace` as for swarm_train_tick_grad; `ring->capacity`
 * is the ring_capacity of the apply phase. */
int swarm_train_tick(const SwarmConfig* cfg, const SwarmTrainHyper* hyper, SwarmTrainCtl* ctl, float* weights,
                     float* target_weights, float* exp_avg, float* exp_avg_sq, float* state, float* returns,
                     int32_t* hits, const SwarmReplay* ring, int64_t* indices, float* grad, void* workspace,
                     int64_t workspace_bytes, const SwarmPeerExchange* peers, void* stream);

/* The same device-driven tick for a stacked network (SwarmStackSpec, below), four launches and no host work, so it
 * captures into a CUDA graph like swarm_train_tick:
 *   1. rollout tick of all cfg->num_envs envs with the online weights: swarm_gatstack_forward (argmax), the exploration
 *      draws of swarm_train_tick_grad (same rng_seed / env_offset stream, epsilon and tick from ctl), the world step,
 *      the tick's reward, returns / hits accumulated, (s, a, r, s') pushed at slot (ctl->ring_cursor + env) % capacity;
 *   2. graphs_per_update slots drawn from the filled ring as swarm_train_tick_grad draws them (exported to indices
 *      int64[G] when indices != NULL), gradient + loss of that batch as swarm_dqn_stack_grad;
 *   3. the sum of the gradient kernel's per-CTA partials; sets ctl->updating;
 *   4. swarm_adam_clip_stack_step with the bias corrections from ctl->opt_step + 1, target <- online when
 *      (ctl->tick + 1) % update_target_every == 0, then ctl advances as in swarm_train_tick_apply.
 * While the ring holds fewer than G slots, grad / loss are left untouched and ctl->updating = 0.
 * reward: as for swarm_rollout_stack -- NULL gives the world's own reward (GoTo / ObstacleAvoidance), a Flocking spec
 * (shaping float[B][N][2] required, read and written back) or a Cohesion spec selects that reward on the GoTo world;
 * hyper->flocking must be NULL.  grad float[count + 1] = gradient (count = swarm_stack_weight_count(spec)), then the
 * loss.  2 <= n_agents <= 128, graphs and spec as for swarm_dqn_stack_grad.  workspace:
 * swarm_dqn_stack_workspace_bytes(cfg, spec, G).  A data-parallel trainer calls the same tick as its two phases,
 * swarm_train_tick_stack_grad (launches 1-3, with the gradient exchange) and swarm_train_tick_stack_apply (launch 4). */
struct SwarmStackSpec;
int swarm_train_tick_stack(const SwarmConfig* cfg, const struct SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                           const struct SwarmRewardSpec* reward, float* shaping, SwarmTrainCtl* ctl, float* weights,
                           float* target_weights, float* exp_avg, float* exp_avg_sq, float* state, float* returns,
                           int32_t* hits, const SwarmReplay* ring, int64_t* indices, float* grad, void* workspace,
                           int64_t workspace_bytes, void* stream);

/* swarm_train_tick_stack as two calls, for data-parallel training: swarm_train_tick_stack_grad followed by
 * swarm_train_tick_stack_apply gives the same bits as swarm_train_tick_stack.
 *
 * Phase 1 runs launches 1-3 of swarm_train_tick_stack (rollout tick, slot draw + gradient, partial-sum reduce) and takes
 * the same arguments, with the same checks, minus exp_avg / exp_avg_sq.  grad is float[count + 1] (gradient, then the
 * loss), so a trainer without peer memory all-reduces one buffer between the phases.  With peers != NULL the reduce
 * launch also sums grad and loss over the ranks: the peer exchange of swarm_train_tick_apply (word = epoch << 32 | float
 * bits, own buffer first, polls of the local buffer, rank-order sums), on a buffer of
 * uint64[2][world_size][SWARM_XCHG_STACK_STRIDE], zero-initialised; when the call returns on the stream, grad holds
 * the sum over the ranks on every rank.  Ticks that do not update exchange nothing.
 *
 * The exchange sits in the grad phase here, while the one-layer tick's sits in swarm_train_tick_apply: the stacked
 * reduce launch runs one gradient element per thread over ceil((count + 1) / 256) CTAs (2 for the Flocking
 * checkpoint's 409 weights, 20 for the largest stack), so every thread pushes one word per peer and polls world_size
 * words -- the shape of the one-layer exchange that measured fastest.  The stacked clip + Adam kernel is one CTA holding
 * up to 20 elements per thread; polling there would put 20 x world_size loads in one thread's registers.
 *
 * All ranks must run the same number of envs, start from the same ring fill and call the phases for the same ticks. */
enum { SWARM_XCHG_STACK_STRIDE = 5040 };     /* >= 5 033 weights of the largest stack + the loss, a multiple of 8 */
int swarm_train_tick_stack_grad(const SwarmConfig* cfg, const struct SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                                const struct SwarmRewardSpec* reward, float* shaping, SwarmTrainCtl* ctl,
                                const float* weights, const float* target_weights, float* state, float* returns,
                                int32_t* hits, const SwarmReplay* ring, int64_t* indices, float* grad, void* workspace,
                                int64_t workspace_bytes, const SwarmPeerExchange* peers, void* stream);

/* Phase 2: launch 4 of swarm_train_tick_stack -- clip_grad_norm_ + Adam on grad (the gradient phase's, reduced over the
 * ranks), the target sync and the cursor advance; ring_capacity as ring->capacity of phase 1.  Rejects every cfg, spec
 * and hyper that swarm_train_tick_stack rejects. */
int swarm_train_tick_stack_apply(const SwarmConfig* cfg, const struct SwarmStackSpec* spec, const SwarmTrainHyper* hyper,
                                 SwarmTrainCtl* ctl, float* weights, float* target_weights, float* exp_avg,
                                 float* exp_avg_sq, const float* grad, int64_t ring_capacity, void* stream);

/* ---- device-side episode boundary (SURVEY.md 8f rank 2) -------------------------------------------------------
 * The reference resets with one CPU torch.normal draw per episode (go_to:84-88, oa:100-102) and does its episode
 * bookkeeping in Python (train:179-199).  These two calls keep both on the device so that reset + max_steps ticks +
 * bookkeeping form one replayable CUDA graph and a whole training run needs no host synchronisation. */
typedef struct SwarmResetSpec {
  float base_x, base_y;      /* GoTo (1.5, -1.5) = -position_range (go_to:84); OA (0.6, -0.6) (oa:100)                 */
  float mean_x, mean_y;      /* GoTo (-0.6, 0.6); OA (0, 0)                                                            */
  float std_x, std_y;        /* GoTo 0.4; OA 0.1 with random=True, else 0                                              */
  uint64_t seed;             /* counter RNG keyed by (seed, global env index, episode): a documented deviation from    */
  int64_t env_offset;        /* torch's CPU mt19937 stream; parity tests pass explicit centres to swarm_reset_grid     */
  int32_t shared_center;     /* 1: every env gets env 0's draw (the reference's `env_index=None` behaviour)            */
  int32_t pad;
} SwarmResetSpec;

/* centres c_b = base + mean + std * N(0,1) drawn for episode `ctl->episode` (or `episode` when ctl == NULL), agents on
 * the start grid around them, velocities zero.  centers_out (optional) float[B][2] receives the drawn centres. */
int swarm_reset_random(const SwarmConfig* cfg, const SwarmResetSpec* spec, const SwarmTrainCtl* ctl, int64_t episode,
                       float* centers_out, float* state, void* stream);

/* End-of-episode bookkeeping (train:179-199): row ctl->episode of stats float[max_episodes][4] receives
 * (mean over envs of agent 0's return / N, mean obstacle hits per env, the last update's loss, the epsilon used);
 * returns / hits are zeroed for the next episode; epsilon <- max(min_epsilon, epsilon0 * exp(-decay * episode))
 * (train:180); ctl->episode += 1.  Rows beyond max_episodes are dropped. */
int swarm_episode_end(const SwarmConfig* cfg, SwarmTrainCtl* ctl, float* returns, int32_t* hits, const float* loss,
                      float* stats, int64_t max_episodes, double epsilon0, double epsilon_decay, double min_epsilon,
                      void* stream);

/* ---- rewards of the remaining reference scenarios (SURVEY.md 8f rank 3) -----------------------------------------
 * FlockingScenario (flocking_scenario.py:93-176) and CohesionScenario (cohesion_scenario.py:66-85) step the same world
 * as GoTo (colliding sphere agents, no colliding landmark: swarm_sim_step with SWARM_SCENARIO_GOTO); only their reward
 * differs.  swarm_scenario_reward evaluates it on the stepped state, one env = one copy of the reference's one-env
 * computation (the reference branches on tensors in Python and cannot run batched).
 *   Flocking: reward float[B] = the collective reward every agent receives (flocking:124-131); shaping float[B][N][2]
 *     carries (previous_distance_to_goal, previous_distance_to_agents) between ticks and is REQUIRED; a call with
 *     reset = 1 initialises it the way reset_world_at does (agent i sees the agents after it at the origin, where
 *     world.reset left them, flocking:93-121) and writes no reward; env_index >= 0 restricts either call to one env
 *     (reset_world_at(env_index)).  terms (optional) float[B][N][4] = (pos_rew, avoidance, dist_rew, distance_to_goal).
 *   Cohesion: reward float[B][N] per agent; shaping unused (NULL); terms (optional) float[B][N][4] =
 *     (collision_factor, cohesion_factor, min_distance, max_distance).
 * 2 <= n_agents <= 128 (with one agent the reference's torch.stack / torch.cat of an empty list raises); larger swarms:
 * swarm_scenario_reward_large. */
#define SWARM_REWARD_FLOCKING 0
#define SWARM_REWARD_COHESION 1
typedef struct SwarmRewardSpec {
  int32_t kind;                  /* SWARM_REWARD_*                                                                      */
  int32_t num_envs, n_agents;
  int32_t reset;                 /* Flocking: 1 = initialise the shaping memory, no reward                              */
  int64_t env_index;             /* -1 = every env                                                                      */
  float goal_x, goal_y;          /* (-0.8, 0.8) flocking:96                                                             */
  float goal_radius;             /* 0.05: on_goal = distance_to_goal < goal.shape.radius (flocking:134)                 */
  float agent_radius;            /* 0.05: world.get_distance subtracts both radii                                       */
  float pos_shaping;             /* pos_shaping_factor 10 (flocking:10)                                                 */
  float dist_shaping;            /* dist_shaping_factor 10 (flocking:11)                                                */
  float desired_distance;        /* 0.15 (flocking:20)                                                                  */
  float min_collision_distance;  /* 0.005 (flocking:21)                                                                 */
  float collision_reward;        /* -1 (flocking:19)                                                                    */
  float on_goal_bonus;           /* 50 (flocking:142)                                                                   */
  float sigma;                   /* Cohesion 0.15 (cohesion:23)                                                         */
  float pad;
} SwarmRewardSpec;

void swarm_default_reward_spec(SwarmRewardSpec* spec, int32_t kind, int32_t num_envs, int32_t n_agents);
int swarm_scenario_reward(const SwarmRewardSpec* spec, const float* state, float* shaping, float* reward, float* terms,
                          void* stream);

/* The same rewards, outputs and arguments for 2 <= n_agents <= 4096 (num_envs * n_agents < 2^31), equal bit for bit to
 * the reference's float32 CPU computation at every size: the spacing term's mean over the N - 1 partner distances adds
 * in the order torch's CPU row sum takes, including the cascade ATen starts at 512 floats per row.  One thread per
 * agent sweeps every partner of its env from shared memory (O(N^2) per env); Flocking's collective reward is then added
 * in agent order by a second launch.  workspace: swarm_scenario_reward_large_workspace_bytes(spec) bytes (Flocking:
 * float[B][N] of per-agent terms; Cohesion: 0, workspace may be NULL; 0 as well for arguments the call rejects). */
int64_t swarm_scenario_reward_large_workspace_bytes(const SwarmRewardSpec* spec);
int swarm_scenario_reward_large(const SwarmRewardSpec* spec, const float* state, float* shaping, float* reward,
                                float* terms, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- multi-layer GAT Q-networks (SURVEY.md 8f rank 4) -------------------------------------------------------------
 * The reference's GCN class carries conv2 / conv3 in comments (train_gcn_dqn.py:54-55, 64-67) and ships checkpoints of
 * that form: data/models/experiment_Flocking-seed_*.pth = conv1 (7 -> 8), conv2, conv3 (8 -> 8), lin1 (8 -> 8), lin2
 * (8 -> 9).  A stack is n_layers single-head GATConv layers (add_self_loops = False, bias) of one width, each followed
 * by an activation, then lin1 -> ReLU -> lin2 as in GCN.forward (train:59-70).
 * weights: state-dict order, float32 -- per layer att_src[H], att_dst[H], bias[H], lin.weight[H][Cin] (Cin = in_features
 * for conv1, H above), then lin1.weight[H][H], lin1.bias[H], lin2.weight[9][H], lin2.bias[9];
 * swarm_stack_weight_count(spec) floats. */
#define SWARM_ACT_TANH 0
#define SWARM_ACT_RELU 1
typedef struct SwarmStackSpec {
  int32_t n_layers;        /* 1 .. 4                                                                                  */
  int32_t hidden;          /* H: 1 .. 32                                                                              */
  int32_t in_features;     /* 7: [pos, vel, goal, agent id] (train:95-99); 5: [pos, vel, agent id] for scenarios whose
                              observation() is cat[pos, vel] (cohesion_scenario.py:87-94)                            */
  int32_t activation[4];   /* SWARM_ACT_* after conv l (train:62,65,67: tanh, relu, relu)                             */
  int32_t pad;
} SwarmStackSpec;
int64_t swarm_stack_weight_count(const SwarmStackSpec* spec);

/* The whole forward of a stack on the per-env graph named by cfg->graph_mode (complete; radius; kNN for n_agents <= 16)
 * in ONE launch: in-edge lists built once in shared memory, layer outputs never leave the chip.  n_agents <= 128
 * (larger swarms: swarm_gatstack_forward_large).  q float[B*N][9] and actions int32[B*N] (argmax, first maximum wins)
 * are optional. */
int swarm_gatstack_forward(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, const float* state,
                           float* q, int32_t* actions, void* stream);

/* The same forward for large swarms, ONE launch with one CTA per env: any spec, 1 <= n_agents <= 4096, on the radius
 * and complete graphs and on the kNN graph from the caller's topk table (neighbours int32[B][N][k] of swarm_graph_build;
 * above 128 agents 64 k <= n_agents, its partial_sort branch).  The attention runs in input space per layer
 * (sum alpha h_src = W sum alpha x_src, <h, att> = <x, W^T att>): float32-level different rounding from
 * swarm_gatstack_forward.  The complete graph costs O(N log N) per layer (sources sorted by alpha_src, prefix / suffix
 * scans).  The layer rows live in the workspace (double-buffered, [2][B][N][8 | 16 | 32] floats).  q / actions as
 * swarm_gatstack_forward.  workspace: swarm_gatstack_large_workspace_bytes(cfg, spec) bytes (0 for rejected
 * arguments). */
int64_t swarm_gatstack_large_workspace_bytes(const SwarmConfig* cfg, const SwarmStackSpec* spec);
int swarm_gatstack_forward_large(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights,
                                 const float* state, const int32_t* neighbours, float* q, int32_t* actions,
                                 void* workspace, int64_t workspace_bytes, void* stream);

/* `ticks` greedy evaluation ticks (simulator.py:59-93) of a stacked network: per tick swarm_gatstack_forward (argmax)
 * -> swarm_sim_step in place -> the tick's reward -> returns float[B*N] (+=), hits int32[B] (+=, obstacles_hits()).
 * reward == NULL: the world's own reward (GoTo / ObstacleAvoidance); a SwarmRewardSpec selects the Flocking collective
 * reward (shaping float[B][N][2] required, initialised by a reset call of swarm_scenario_reward) or Cohesion's per-agent
 * reward on the GoTo world, evaluated by the swarm_scenario_reward arithmetic after every step.  n_agents <= 128: the
 * whole loop is ONE launch (state, running return and Flocking memory in registers across the ticks, same tick as
 * swarm_rollout) that leaves the workspace untouched.  n_agents > 128 (up to 4096): per tick [kNN: the topk table of
 * swarm_graph_build ->] swarm_gatstack_forward_large (argmax) -> swarm_sim_step in place, returns / hits accumulated by
 * the world step; reward must be NULL there (with a Flocking / Cohesion reward above 128 agents:
 * swarm_rollout_stack_large).
 * No host work or allocation inside (graph capturable).  workspace: swarm_rollout_stack_workspace_bytes(cfg). */
int64_t swarm_rollout_stack_workspace_bytes(const SwarmConfig* cfg);
int swarm_rollout_stack(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, float* state,
                        int32_t ticks, const SwarmRewardSpec* reward, float* shaping, float* returns, int32_t* hits,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* swarm_rollout_stack for 129 <= n_agents <= 4096 with any reward: per tick [kNN: the topk table ->]
 * swarm_gatstack_forward_large (argmax) -> swarm_sim_step in place (hits += as in swarm_rollout_stack) -> with a
 * SwarmRewardSpec, swarm_scenario_reward_large on the stepped state and returns[b][i] += the tick's reward (Flocking:
 * the env's collective reward for every agent, shaping required and initialised by a reset call; Cohesion: the agent's
 * own).  reward == NULL gives exactly what swarm_rollout_stack gives (the world's own reward).  No host work or
 * allocation inside (graph capturable).  workspace: swarm_rollout_stack_large_workspace_bytes(cfg, reward) bytes, which
 * is swarm_rollout_stack_workspace_bytes(cfg) for reward == NULL (0 outside 129 <= n_agents <= 4096). */
int64_t swarm_rollout_stack_large_workspace_bytes(const SwarmConfig* cfg, const SwarmRewardSpec* reward);
int swarm_rollout_stack_large(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* weights, float* state,
                              int32_t ticks, const SwarmRewardSpec* reward, float* shaping, float* returns,
                              int32_t* hits, void* workspace, int64_t workspace_bytes, void* stream);

/* One DQN loss + gradient of a stacked network (train_step_dqn, train_gcn_dqn.py:116-124, for the conv1 .. convL form):
 * the contract of swarm_dqn_grad for the network described by `spec`.  Transitions come from `batch` (slot g, or slot
 * indices[g] when indices != NULL); values = Q_online(s)[a], targets = r + gamma * max_a Q_target(s') (no terminal
 * mask), loss = loss_scale * sum over the n_graphs*N nodes of (values - targets)^2 (loss_scale = 1 / (n_graphs*N) gives
 * nn.MSELoss).  Each graph is built per env from cfg->graph_mode, on s for the online network and on s' for the target;
 * node features as swarm_gatstack_forward, whose Q values the kernel reproduces bit for bit.  Hand-written backward
 * pass through the layer stack; per-CTA partial sums reduced in a fixed order, no atomics (bit-reproducible).
 * cfg->num_envs is ignored; 2 <= n_agents <= 128, graphs and spec as for swarm_gatstack_forward.  Outputs:
 * grad float[swarm_stack_weight_count(spec)] (packed stack order), loss float[1] (both overwritten); td (optional)
 * float[n_graphs*N] = values - targets, formed with separately rounded ops (gamma * next, + r, values -).
 * workspace: swarm_dqn_stack_workspace_bytes(cfg, spec, n_graphs) bytes (0 for arguments the call would reject). */
int64_t swarm_dqn_stack_workspace_bytes(const SwarmConfig* cfg, const SwarmStackSpec* spec, int32_t n_graphs);
int swarm_dqn_stack_grad(const SwarmConfig* cfg, const SwarmStackSpec* spec, const float* online_weights,
                         const float* target_weights, const SwarmReplay* batch, const int64_t* indices, int32_t n_graphs,
                         float gamma, float loss_scale, float* grad, float* loss, float* td, void* workspace,
                         int64_t workspace_bytes, void* stream);

/* clip_grad_norm_(model.parameters(), max_norm) + one torch.optim.Adam step (train:125-126) on the packed weights of a
 * stack, in place: swarm_adam_clip_step for swarm_stack_weight_count(spec) floats.  The per-tensor 2-norms are taken over
 * the state-dict tensors in packed order (per layer att_src, att_dst, bias, lin.weight; then lin1.weight, lin1.bias,
 * lin2.weight, lin2.bias -- the order of StackedGCN.parameters()), then the 2-norm of those; clip coefficient
 * max_norm / (norm + 1e-6), clamped to 1; max_norm <= 0 disables clipping.  `step` is the 1-based step count;
 * target_weights (optional) receives a copy of the updated weights, grad_norm (optional) float[1] the pre-clip norm. */
int swarm_adam_clip_stack_step(const SwarmStackSpec* spec, float* weights, const float* grad, float* exp_avg,
                               float* exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                               double max_norm, float* target_weights, float* grad_norm, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SWARM_B200_H */
