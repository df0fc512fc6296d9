// ppo_kernels.h -- internal launcher interface between ppo_api.cu and ppo_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PPO_H 64
#define PPO_A 4
#define PPO_DPAD 32
#define PPO_FWD_THREADS 128

cudaError_t ppok_forward(const float* params, int d, const float* obs_raw, const double* stats, float clip, int n,
                         uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev, int deterministic,
                         float* obs_norm, float* act_env, float* act_raw, float* logp, float* value, int want_policy,
                         cudaStream_t st, const uint8_t* boot_flags = nullptr, float boot_gamma = 0.0f,
                         float* boot_rew = nullptr, int a = PPO_A);
cudaError_t ppok_counter_add(uint32_t* ctr, uint32_t inc, cudaStream_t st);
cudaError_t ppok_eval_ledger(const float* rew, const uint8_t* flags, const uint8_t* tidx, int n, double* ret, int* len, int* count,
                             const int* quota, const int* offset, uint32_t step, const uint32_t* step_dev, int step_limit,
                             int* remaining, double* ep_ret, int* ep_len, uint8_t* ep_tr, uint8_t* ep_flags, int* ep_step,
                             cudaStream_t st);
cudaError_t ppok_permutation(long long* out, long long n, uint64_t seed, uint64_t epoch, cudaStream_t st);
cudaError_t ppok_permutation_window(long long* out, long long n, uint64_t seed, uint32_t* ctr, long long window_len, cudaStream_t st);
cudaError_t ppok_moments(const float* x, int n, int d, double* stats, double* scratch, double* accum, cudaStream_t st);
cudaError_t ppok_moments_finalize(double* acc, int slots, int n, int d, double* stats, double* accum, cudaStream_t st);
cudaError_t ppok_reward_normalize(const float* rew, const uint8_t* flags, int n, float gamma, float clip, float* ret,
                                  double* ret_stats, double* scratch, double* accum, float* rew_norm, float* done_out,
                                  cudaStream_t st);
cudaError_t ppok_bootstrap(const float* params, int d, const float* term_obs, const double* stats, float clip,
                           const uint8_t* flags, int n, float gamma, float* rew, float* value_scratch, cudaStream_t st,
                           int a = PPO_A);
cudaError_t ppok_gae(const float* rewards, const float* values, const float* dones, const float* last_values, int T, int n,
                     float gamma, float lam, float* adv, float* ret, cudaStream_t st);
// tensor-core forward: one instantiation per action width (ppo_tc.cu compiled for 4, ppo_tc_a6.cu for 6)
#define PPOK_DECLARE_FORWARD_TC(ns)                                                                                      \
    namespace ns {                                                                                                        \
    cudaError_t ppok_forward_tc(const float* params, int d, const float* obs_raw, const double* stats, float clip, int n, \
                                uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev,                \
                                int deterministic, float* obs_norm, float* act_env, float* act_raw, float* logp,         \
                                float* value, cudaStream_t st);                                                          \
    }
PPOK_DECLARE_FORWARD_TC(ppo_a4)
PPOK_DECLARE_FORWARD_TC(ppo_a6)
PPOK_DECLARE_FORWARD_TC(ppo_a4d64)
int ppok_update_grid(int batch);
// clip + Adam folded into the partial-gradient reduction (single process: nothing sits between gradient and optimizer)
// world > 1: the last block of the reduction all-reduces the gradient through peer memory first (ppo_update_tc.cu, ppo_peer_*)
struct PpokAdam { float lr, beta1, beta2, eps, max_norm; float* params; float* m; float* v; int* step_ctr; float* norm_out; unsigned* arrivals;
                  int world = 1, rank = 0; unsigned* seq = nullptr; float* peer[8] = {}; };
size_t ppok_peer_bytes();
void ppok_launch_adv_stats(const float* adv, const long long* idx, int batch, int nmb, double* scratch, float* adv_stats, cudaStream_t st);
// fused minibatch gradient: one instantiation per (action width, observation slab): ppo_update_tc.cu = (4, 32),
// ppo_update_tc_a6.cu = (6, 32), ppo_update_tc_d64.cu = (4, 64)
#define PPOK_DECLARE_MINIBATCH_GRAD(ns)                                                                                    \
    namespace ns {                                                                                                          \
    cudaError_t ppok_minibatch_grad(const float* params, int d, const float* obs, const float* act, const float* logp_old, \
                                    const float* adv, const float* ret, const long long* idx, int batch, float clip_range, \
                                    float ent_coef, float vf_coef, double* scratch, float* adv_stats, float* partial,      \
                                    float* stats_partial, float* grad, float* stats, cudaStream_t st,                      \
                                    const PpokAdam* adam = nullptr, int have_adv_stats = 0);                               \
    cudaError_t ppok_minibatch_steps(float* params, int d, const float* obs, const float* act, const float* logp_old,       \
                                     const float* adv, const float* ret, const long long* idx, int batch, int steps,       \
                                     float clip_range, float ent_coef, float vf_coef, float* m, float* v, float lr,        \
                                     float beta1, float beta2, float eps, float max_norm, int* step_ctr, float* norm_out,  \
                                     float* grad, float* stats, cudaStream_t st, int world = 1, int rank = 0,              \
                                     void* const* peers = nullptr, unsigned* seq = nullptr);                               \
    }
PPOK_DECLARE_MINIBATCH_GRAD(ppo_a4)
PPOK_DECLARE_MINIBATCH_GRAD(ppo_a6)
PPOK_DECLARE_MINIBATCH_GRAD(ppo_a4d64)
cudaError_t ppok_adam(float* params, const float* grad, float* m, float* v, int P, float lr, float beta1, float beta2, float eps,
                      float max_norm, float grad_scale, int* step_ctr, float* norm_out, cudaStream_t st);
