// launchers.h -- host-side functions that one csrc/*.cu file defines and another calls: kernel launchers and the
// workspace, shared-memory and fit functions the entry points of api.cu check before a launch. Every file that defines
// or calls one includes this header, so the compiler checks each call and each definition against one declaration.
// Default arguments live here only.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/swarm_b200.h"

namespace swarm {

struct DqnParams;
struct SimStepArgs;
struct TileParams;
struct WorldConsts;

// env-tile kernels (n_agents <= 128), world step, resets, replay ring
cudaError_t launch_tile(int mode, const TileParams& p, cudaStream_t stream);
cudaError_t launch_sim_step(SimStepArgs p, cudaStream_t stream);
cudaError_t launch_reset_grid(const SwarmConfig& c, int cols, int rows, const float* centers, float* state,
                              cudaStream_t stream);
cudaError_t launch_reset_random(const SwarmConfig& c, const SwarmResetSpec& sp, int cols, int rows, const SwarmTrainCtl* ctl,
                                long long episode, float* centers_out, float* state, cudaStream_t stream);
cudaError_t launch_episode_end(const SwarmConfig& c, SwarmTrainCtl* ctl, float* returns, int32_t* hits, const float* loss,
                               float* stats, long long max_episodes, double eps0, double decay, double min_eps,
                               cudaStream_t stream);
cudaError_t launch_replay_push(const SwarmReplay& r, long long cursor, int B, int N, const float* state,
                               const int32_t* actions, const float* rewards, const float* next_state,
                               cudaStream_t stream);
cudaError_t launch_replay_gather(const SwarmReplay& r, const int64_t* indices, int G, int N, float* state,
                                 int32_t* actions, float* rewards, float* next_state, cudaStream_t stream);

// large swarms (one CTA per env, up to 4 096 agents)
cudaError_t launch_sim_step_large(const SimStepArgs& p, cudaStream_t stream);
bool sim_step_grid_enabled(int n_agents);
cudaError_t launch_sim_step_grid(const SimStepArgs& p, cudaStream_t stream);
cudaError_t launch_graph_large(const SwarmConfig& c, const float* state, int32_t* edges, int32_t* nbr, int edges_per_env,
                               cudaStream_t stream);
cudaError_t launch_radius_csr(const SwarmConfig& c, const float* state, int32_t* degree, const int32_t* row_ptr,
                              int32_t* src, cudaStream_t stream);
bool gatq_knn_large_fits(int N, int K);
cudaError_t launch_gatq_knn_large(const SwarmConfig& c, const float* weights, const float* state, const int32_t* nbr,
                                  float* q, int32_t* actions, cudaStream_t stream);
bool gatq_knn_large_x_fits(int N, int K);
cudaError_t launch_gatq_knn_large_x(const SwarmConfig& c, const float* weights, const float* state, const int32_t* nbr,
                                    float* q, int32_t* actions, cudaStream_t stream);
bool gatq_large_x_fits(int N, bool radius);
cudaError_t launch_gatq_large_x(const SwarmConfig& c, const float* weights, const float* state, float* q, int32_t* actions,
                                cudaStream_t stream);

// generic graphs (CSR)
long long csr_workspace_bytes(int n, long long E);
cudaError_t launch_csr_from_edges(int n, long long E, const int64_t* edge_src, const int64_t* edge_dst, int32_t* row_ptr,
                                  int32_t* src, int32_t* perm, void* workspace, long long workspace_bytes,
                                  cudaStream_t stream);
long long gatq_workspace_bytes(int n);
cudaError_t launch_csr_project(int n, const float* weights, const float* x, float* rows, cudaStream_t stream);
cudaError_t launch_gatq_csr(int n, const float* weights, const float* x, const int32_t* row_ptr, const int32_t* src,
                            float* q, int32_t* actions, float* rows, cudaStream_t stream, bool conv_only = false);
long long gatq_backward_workspace_bytes(int n, long long E);
cudaError_t launch_gatq_backward_csr(int n, long long E, const float* weights, const float* x, const int32_t* row_ptr,
                                     const int32_t* src, const int32_t* perm, const int32_t* row_ptr_s,
                                     const int32_t* tgt_s, const int32_t* perm_s, const float* grad_q, float* grad_w,
                                     void* workspace, cudaStream_t stream, bool conv_only = false);
long long gat_layer_workspace_bytes(int n, long long E, int ci, int co, bool backward);
cudaError_t launch_gat_layer_forward(int n, int ci, int co, const float* W, const float* a_src, const float* a_dst,
                                     const float* bias, const float* x, const int32_t* row_ptr, const int32_t* src,
                                     float* out, void* workspace, cudaStream_t stream);
cudaError_t launch_gat_layer_backward(int n, long long E, int ci, int co, const float* W, const float* a_src,
                                      const float* a_dst, const float* x, const int32_t* row_ptr, const int32_t* src,
                                      const int32_t* perm, const int32_t* row_ptr_s, const int32_t* tgt_s,
                                      const int32_t* perm_s, const float* grad_out, float* gW, float* gas, float* gad,
                                      float* gb, float* grad_x, void* workspace, cudaStream_t stream);

// Flocking / Cohesion rewards
cudaError_t launch_scenario_reward(const SwarmRewardSpec& sp, const float* state, float* shaping, float* reward,
                                   float* terms, cudaStream_t stream);
long long scenario_reward_large_workspace_bytes(const SwarmRewardSpec& sp);
cudaError_t launch_scenario_reward_large(const SwarmRewardSpec& sp, const float* state, float* shaping, float* reward,
                                         float* terms, float* returns, void* workspace, cudaStream_t stream);

// one-layer DQN update
long long dqn_workspace_bytes(const SwarmConfig& c, int n_graphs);
int dqn_smem_bytes(const SwarmConfig& c);
bool dqn_fuse_reduce(const SwarmConfig& c, int n_graphs);
cudaError_t launch_dqn_grad_tc(DqnParams& p, cudaStream_t stream);
cudaError_t launch_dqn_grad(const SwarmConfig& c, const float* w_online, const float* w_target, const SwarmReplay& batch,
                            const int64_t* indices, int n_graphs, float gamma, float loss_scale, float* grad, float* loss,
                            float* td, void* workspace, cudaStream_t stream, SwarmTrainCtl* ctl = nullptr,
                            int64_t* indices_out = nullptr, unsigned long long sample_seed = 0, int pushed_envs = 0,
                            bool skip_reduce = false);
cudaError_t launch_adam_clip(float* w, const float* grad, float* m, float* v, long long step, double lr, double beta1,
                             double beta2, double eps, double max_norm, float* target, float* grad_norm,
                             cudaStream_t stream, SwarmTrainCtl* ctl = nullptr, int num_envs = 0,
                             long long ring_capacity = 1, int update_target_every = 1,
                             const SwarmPeerExchange* peers = nullptr, float* grad_rw = nullptr,
                             const SwarmConfig* reduce_cfg = nullptr, const void* reduce_workspace = nullptr,
                             int reduce_graphs = 0, float loss_scale = 0.0f);

// stacked GAT Q-networks
int stack_weight_count_host(const SwarmStackSpec& s);
cudaError_t launch_gatstack_forward(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, const float* state,
                                    float* q, int32_t* actions, cudaStream_t stream);
cudaError_t launch_gatstack_rollout(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, float* state,
                                    int ticks, const WorldConsts& step, const SwarmRewardSpec* flock, float* shaping,
                                    float* returns, int32_t* hits, cudaStream_t stream);
cudaError_t launch_gatstack_train_tick(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, float* state,
                                       const WorldConsts& step, const SwarmRewardSpec* flock, float* shaping,
                                       float* returns, int32_t* hits, const SwarmReplay& ring, const SwarmTrainCtl* ctl,
                                       unsigned long long rng_seed, long long env_offset, cudaStream_t stream);
int stack_large_smem_bytes(const SwarmConfig& c, const SwarmStackSpec& s);
long long stack_large_workspace_bytes(const SwarmConfig& c, int hp);
long long stack_large_workspace_bytes(const SwarmConfig& c, const SwarmStackSpec& s);
cudaError_t launch_gatstack_large(const SwarmConfig& c, const SwarmStackSpec& spec, const float* weights, const float* state,
                                  const int32_t* nbr, float* q, int32_t* actions, void* workspace, cudaStream_t stream);
int stack_grad_smem_bytes(const SwarmConfig& c, const SwarmStackSpec& s);
long long stack_grad_workspace_bytes(const SwarmConfig& c, const SwarmStackSpec& s, int n_graphs);
cudaError_t launch_stack_grad(const SwarmConfig& c, const SwarmStackSpec& spec, const float* w_online, const float* w_target,
                              const SwarmReplay& batch, const int64_t* indices, int n_graphs, float gamma, float loss_scale,
                              float* grad, float* loss, float* td, void* workspace, cudaStream_t stream,
                              SwarmTrainCtl* ctl = nullptr, int64_t* indices_out = nullptr,
                              unsigned long long sample_seed = 0, int pushed_envs = 0,
                              const SwarmPeerExchange* peers = nullptr);
cudaError_t launch_stack_adam_clip(const SwarmStackSpec& spec, float* w, const float* grad, float* m, float* v,
                                   long long step, double lr, double beta1, double beta2, double eps, double max_norm,
                                   float* target, float* grad_norm, cudaStream_t stream, SwarmTrainCtl* ctl = nullptr,
                                   int num_envs = 0, long long ring_capacity = 1, int update_target_every = 1);

}  // namespace swarm
