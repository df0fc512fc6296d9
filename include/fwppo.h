/*
 * fwppo.h -- C ABI of the PPO rollout kernels in libfwsim.so.
 *
 * These replace, for the whole env batch at once and without leaving HBM, what the reference obtains from
 * stable_baselines3 around its env (train/train_Fixedwing_Waypoints_v3.py:260,293-337):
 *   VecNormalize (obs / reward running moments, normalise + clip)   -> ppo_moments_update, ppo_reward_normalize
 *   MlpPolicy forward (separate pi / vf towers 64-64 tanh, diagonal Gaussian, action clip)
 *                                                                     -> ppo_policy_forward, ppo_value_forward
 *   time-limit bootstrap r += gamma * V(terminal_obs)               -> ppo_timeout_bootstrap
 *   RolloutBuffer.compute_returns_and_advantage (GAE)                -> ppo_gae
 * Same conventions as fwsim.h: 0 = OK, negative = error, fw_last_error() for the message; all pointers are
 * DEVICE pointers owned by the caller (torch tensors); work is enqueued on the caller's stream.
 *
 * Parameter vector layout (fp32, contiguous), H = 64 hidden units, D = obs_dim, A = 4 actions:
 *   pi.W1[H,D] pi.b1[H] pi.W2[H,H] pi.b2[H] pi.W3[A,H] pi.b3[A]
 *   vf.W1[H,D] vf.b1[H] vf.W2[H,H] vf.b2[H] vf.W3[1,H] vf.b3[1]  log_std[A]
 * (row-major [out,in], i.e. torch.nn.Linear.weight), 12,361 floats for D = 28.
 */
#ifndef FWPPO_H
#define FWPPO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPO_HIDDEN 64
#define PPO_ACT 4
#define PPO_MAX_OBS 64      /* CUDA-core forward, value, bootstrap, running moments */
#define PPO_TC_MAX_OBS 32   /* tcgen05 forward (ppo_policy_forward_tc*) and fused minibatch gradient with a = 6.  With a = 4
                             * both also take d up to PPO_MAX_OBS (64-wide builds, csrc/ppo_tc_d64.cu, ppo_update_tc_d64.cu) */

/* number of floats in the parameter vector for observation width d */
int ppo_param_count(int32_t d);

/* RunningMeanStd.update (batch-parallel Chan merge): x [n,d] fp32; stats = double[2*d+1] = mean[d], var[d], count.
 * scratch: device doubles, at least 2*d+2, zero on first use (the call leaves it zeroed).
 * accum (may be NULL): double[2*d+1] receiving += column sums, sums of squares and n -- the raw batch moments a
 * multi-GPU run all-reduces once per rollout to reconcile the per-rank running statistics exactly. */
int ppo_moments_update(const float* x, int32_t n, int32_t d, double* stats, double* scratch, double* accum,
                       void* stream);
/* The same update from batch sums the env-step kernels accumulated in their epilogue (fw_set_obs_accumulator, fwsim.h):
 * acc = slots x double[2*d] (column sums | sums of squares per slot), n = rows the sums cover.  Folds them into stats
 * (and accum) and zeroes acc: one 64-thread block instead of a pass over the observation batch. */
int ppo_moments_finalize(double* acc, int32_t slots, int32_t n, int32_t d, double* stats, double* accum, void* stream);

/* Policy + value forward for n rows.  obs_raw [n,d]; obs_stats as above (NULL = no normalisation);
 * writes obs_norm [n,d] (what the policy saw; may be NULL), act_env [n,4] (clipped to [-1,1], what the env
 * gets), act_raw [n,4] (unclipped sample, what the rollout buffer stores), logp [n], value [n].
 * Noise: Philox keyed (seed, env_id0 + row, step + *step_dev); step_dev (may be NULL) is a device counter so
 * that a captured CUDA graph of a whole rollout draws fresh noise on every replay.
 * deterministic != 0 -> action = mean. */
int ppo_policy_forward(const float* params, int32_t d, const float* obs_raw, const double* obs_stats, float clip_obs,
                       int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev,
                       int32_t deterministic, float* obs_norm, float* act_env, float* act_raw, float* logp,
                       float* value, void* stream);

/* Same contract as ppo_policy_forward, computed on the tcgen05 tensor cores (TF32 inputs, fp32 accumulate in
 * TMEM; csrc/ppo_tc.cu): the hidden layers of both towers are 128x32x64 and 128x64x64 UMMA tiles per 128 envs. */
int ppo_policy_forward_tc(const float* params, int32_t d, const float* obs_raw, const double* obs_stats, float clip_obs,
                          int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev,
                          int32_t deterministic, float* obs_norm, float* act_env, float* act_raw, float* logp,
                          float* value, void* stream);

/* Wide-action variants: action width a = 4 or 6.  a = 6 is the low-level env's MlpPolicy
 * (train/train_lowlevel_cmd.py: FixedwingLowLevelEnv, Box(6) actions); the parameter vector has the layout above with
 * A = a, the action buffers are [n, a]. */
int ppo_param_count_a(int32_t d, int32_t a);
int ppo_policy_forward_a(const float* params, int32_t d, int32_t a, const float* obs_raw, const double* obs_stats,
                         float clip_obs, int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev,
                         int32_t deterministic, float* obs_norm, float* act_env, float* act_raw, float* logp, float* value,
                         void* stream);
int ppo_policy_forward_tc_a(const float* params, int32_t d, int32_t a, const float* obs_raw, const double* obs_stats,
                            float clip_obs, int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step,
                            const uint32_t* step_dev, int32_t deterministic, float* obs_norm, float* act_env, float* act_raw,
                            float* logp, float* value, void* stream);     /* tcgen05 forward, a = 4 or 6 */
int ppo_value_forward_a(const float* params, int32_t d, int32_t a, const float* obs_raw, const double* obs_stats,
                        float clip_obs, int32_t n, float* value, void* stream);
int ppo_timeout_bootstrap_a(const float* params, int32_t d, int32_t a, const float* term_obs_raw, const double* obs_stats,
                            float clip_obs, const uint8_t* flags, int32_t n, float gamma, float* rew_inout, void* stream);

/* counter[0] += inc on the device (one node of the rollout graph). */
int ppo_counter_add(uint32_t* counter, uint32_t inc, void* stream);

/* Per-episode bookkeeping of stable_baselines3 evaluate_policy on the device, one thread per env, one launch per agent
 * step (after the step that produced rew / flags).  The eval step index is step + *step_dev (the ppo_policy_forward
 * convention, so a captured chunk of steps replays with ppo_counter_add advancing step_dev); steps at or after
 * step_limit record and accumulate nothing.
 *   rew [n], flags [n]      the step's rewards and flag bytes
 *   targets_reached [n]     the pre-reset num_targets_reached plane (fw_targets_reached); NULL = task without targets
 *   ret [n] (double), len [n], count [n]   running return (ret += (double)rew), length, episodes recorded so far
 *   quota [n], offset [n]   episodes env i records (SB3: (n_eval_episodes + i) // n) and its first slot in the table
 *   remaining               envs with count < quota; decremented (atomically) when an env fills its quota
 * An env whose episode ends (flags & 3) while count < quota writes slot offset + count of the episode table:
 * ep_return (return), ep_length (length), ep_targets (targets reached, 0 without a plane), ep_flags (the terminal step's
 * flag byte), ep_step (eval step index of the episode's last step).  Every ended episode then zeroes ret and len.  The
 * slot depends only on the env and its episode number: the table is bit-reproducible. */
int ppo_eval_ledger(const float* rew, const uint8_t* flags, const uint8_t* targets_reached, int32_t n, double* ret,
                    int32_t* len, int32_t* count, const int32_t* quota, const int32_t* offset, uint32_t step,
                    const uint32_t* step_dev, int32_t step_limit, int32_t* remaining, double* ep_return, int32_t* ep_length,
                    uint8_t* ep_targets, uint8_t* ep_flags, int32_t* ep_step, void* stream);

/* Value tower only (last_values of a rollout). */
int ppo_value_forward(const float* params, int32_t d, const float* obs_raw, const double* obs_stats, float clip_obs,
                      int32_t n, float* value, void* stream);

/* VecNormalize reward path: ret = ret*gamma + r; ret_rms.update(ret); r_norm = clip(r / sqrt(var + eps), +-clip);
 * ret[done] = 0.  flags are the env's flag bytes; done_out [n] receives 1.0/0.0.  ret_stats = double[3]
 * (mean, var, count); scratch = double[3] zero on first use; accum (may be NULL) = double[3] raw sums as above. */
int ppo_reward_normalize(const float* rew, const uint8_t* flags, int32_t n, float gamma, float clip_rew,
                         float* ret, double* ret_stats, double* scratch, double* accum, float* rew_norm,
                         float* done_out, void* stream);

/* SB3 collect_rollouts: for envs that were truncated but not terminated, rew += gamma * V(terminal_obs).
 * value_scratch: n floats (the value tower is evaluated for every row, the add is masked by the flags). */
int ppo_timeout_bootstrap(const float* params, int32_t d, const float* term_obs_raw, const double* obs_stats,
                          float clip_obs, const uint8_t* flags, int32_t n, float gamma, float* rew_inout,
                          float* value_scratch, void* stream);

/* GAE over a [T,n] rollout: rewards, values, dones (done after step t), last_values [n] -> advantages, returns. */
int ppo_gae(const float* rewards, const float* values, const float* dones, const float* last_values, int32_t T,
            int32_t n, float gamma, float lam, float* advantages, float* returns, void* stream);

/* Minibatch order of one epoch: out[0..n) = a keyed pseudo-random permutation of 0..n-1 (device int64), a fresh one per
 * (seed, epoch).  Replaces the np.random.permutation of RolloutBuffer.get (a Feistel bijection with cycle walking
 * instead of a sort). */
int ppo_random_permutation(int64_t* out, int64_t n, uint64_t seed, uint64_t epoch, void* stream);
/* One window of that permutation with the position kept on the device: counters = uint32[2] {epoch, window};
 * out[t] = permutation_epoch(window * window_len + t) for t < window_len (indices past n are not written), then the
 * window advances (wrapping to the next epoch after the last one).  The launch arguments never change, which is what lets
 * a CUDA graph of "indices of the next window -> its minibatch updates" serve every window of every epoch. */
int ppo_random_permutation_window(int64_t* out, int64_t n, uint64_t seed, uint32_t* counters, int64_t window_len, void* stream);

/* ---- PPO minibatch update (stable_baselines3 PPO.train for one minibatch), csrc/ppo_update_tc.cu ----
 * ppo_minibatch_grad: gradient of
 *     -mean(min(A r, A clip(r, 1 +- clip_range))) - ent_coef * mean(entropy) + vf_coef * mean((ret - V)^2)
 * over the `batch` samples idx[0..batch) (int64 row indices into the flattened rollout buffers), with the
 * per-minibatch advantage normalisation (A - mean) / (std + 1e-8), r = exp(logp - logp_old).  Forward and backward
 * of both towers run on the tcgen05 tensor cores (TF32 forward, bf16 backward operands, fp32 accumulation; for
 * d > 32 layer 2 of the forward is a bf16 hi/lo split instead of TF32).  grad receives all ppo_param_count(d) entries;
 * stats[8] (may be NULL) = sums over the minibatch of {policy loss, squared value error, approx KL, clipped,
 * ratio, samples, 0, 0}.  workspace: ppo_update_workspace_floats(d) floats, 16-byte aligned, zero on first use. */
int ppo_update_workspace_floats(int32_t d);
/* action width a = 4 or 6 (the six-channel MlpPolicy of train/train_lowlevel_cmd.py:97-110): parameter vector, action
 * rows and gradient in the layout above with A = a */
int ppo_update_workspace_floats_a(int32_t d, int32_t a);
int ppo_minibatch_grad_a(const float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                         const float* logp_old, const float* adv, const float* ret, const int64_t* idx, int32_t batch,
                         float clip_range, float ent_coef, float vf_coef, float* workspace, float* grad, float* stats,
                         void* stream);
int ppo_minibatch_grad(const float* params, int32_t d, const float* obs_norm, const float* act, const float* logp_old,
                       const float* adv, const float* ret, const int64_t* idx, int32_t batch, float clip_range,
                       float ent_coef, float vf_coef, float* workspace, float* grad, float* stats, void* stream);

/* `steps` consecutive optimizer steps of a single process in ONE launch of one thread block: for s = 0..steps-1 the minibatch
 * idx[s*batch .. (s+1)*batch) goes through its advantage statistics, the gradient above, clip_grad_norm_ and Adam.step
 * (the arithmetic of ppo_minibatch_grad + ppo_adam_step, grad_scale 1), the parameters staying in global memory between
 * steps.  For stable_baselines3-sized minibatches (batch_size 128 = one tile): an optimizer step is then bounded by the
 * tile's latency instead of four kernel launches.  grad / stats / grad_norm_out hold the last step's values. */
#define PPO_FUSED_MAX_BATCH 4096
int ppo_minibatch_steps_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act, const float* logp_old,
                          const float* adv, const float* ret, const int64_t* idx, int32_t batch, int32_t steps, float clip_range,
                          float ent_coef, float vf_coef, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2,
                          float eps, float max_grad_norm, int32_t* step_counter, float* grad_norm_out, float* grad, float* stats,
                          void* stream);

/* A window of n_minibatches (<= PPO_MAX_WINDOW) consecutive optimizer steps of a single process at ANY minibatch size:
 * idx[k*batch .. (k+1)*batch) is minibatch k.  One launch computes the advantage statistics of all of them, then per
 * minibatch the gradient kernel and the partial-gradient reduction whose last block applies clip_grad_norm_ + Adam.step
 * (2 n + 1 launches instead of 4 n; results bit-identical to ppo_minibatch_grad_a + ppo_adam_step with grad_scale 1).
 * workspace as for ppo_minibatch_grad_a. */
#define PPO_MAX_WINDOW 16
int ppo_window_update_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act, const float* logp_old,
                        const float* adv, const float* ret, const int64_t* idx, int32_t batch, int32_t n_minibatches,
                        float clip_range, float ent_coef, float vf_coef, float* exp_avg, float* exp_avg_sq, float lr, float beta1,
                        float beta2, float eps, float max_grad_norm, int32_t* step_counter, float* grad_norm_out, float* workspace,
                        float* grad, float* stats, void* stream);

/* The same window for `world` processes (one per GPU of an NVLink node, world <= 8) WITHOUT a collective library between the
 * gradient and the optimizer: the last block of each rank's gradient reduction pushes the gradient into every rank's
 * exchange buffer with remote stores over NVLink peer memory, raises a sequence-numbered flag, waits for the world's flags,
 * sums the slots in rank order (the same bits on every rank) and applies clip + Adam with grad_scale 1/world -- what
 * all_reduce(sum) + ppo_adam_step do, in the launch that produced the gradient.  peer_buffers[j] = rank j's exchange
 * buffer as mapped into THIS process (own buffer at index `rank`); sequence = a zero-initialised device uint32 of this
 * rank; every rank must make the same calls in the same order.  A rank whose peers do not arrive traps (CUDA error)
 * after about a second instead of hanging.
 *   ppo_peer_alloc / ppo_peer_free        one zeroed exchange buffer (ppo_peer_bytes() bytes, cudaMalloc)
 *   ppo_peer_export / ppo_peer_import     its 64-byte CUDA IPC handle / the peer's buffer mapped here (ppo_peer_close) */
int64_t ppo_peer_bytes(void);
int ppo_peer_alloc(void** buffer);
int ppo_peer_free(void* buffer);
int ppo_peer_export(void* buffer, uint8_t handle[64]);
int ppo_peer_import(const uint8_t handle[64], void** buffer);
int ppo_peer_close(void* buffer);
/* ppo_minibatch_steps_a for `world` processes: every rank's thread block exchanges the step's gradient with the same
 * peer-memory protocol (peer_buffers / sequence as above) before its clip + Adam, `steps` times per launch. */
int ppo_minibatch_steps_p2p_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act, const float* logp_old,
                              const float* adv, const float* ret, const int64_t* idx, int32_t batch, int32_t steps,
                              float clip_range, float ent_coef, float vf_coef, float* exp_avg, float* exp_avg_sq, float lr,
                              float beta1, float beta2, float eps, float max_grad_norm, int32_t* step_counter, float* grad_norm_out,
                              float* grad, float* stats, int32_t world, int32_t rank, void* const* peer_buffers,
                              uint32_t* sequence, void* stream);
int ppo_window_update_p2p_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act, const float* logp_old,
                            const float* adv, const float* ret, const int64_t* idx, int32_t batch, int32_t n_minibatches,
                            float clip_range, float ent_coef, float vf_coef, float* exp_avg, float* exp_avg_sq, float lr,
                            float beta1, float beta2, float eps, float max_grad_norm, int32_t* step_counter, float* grad_norm_out,
                            float* workspace, float* grad, float* stats, int32_t world, int32_t rank, void* const* peer_buffers,
                            uint32_t* sequence, void* stream);

/* torch.nn.utils.clip_grad_norm_(max_grad_norm) followed by torch.optim.Adam.step (no weight decay / amsgrad) on the
 * flat parameter vector; grad is pre-multiplied by grad_scale (1 / world_size after the NCCL sum).
 * step_counter: device int32 incremented by the call (bias correction). */
int ppo_adam_step(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t n_params, float lr,
                  float beta1, float beta2, float eps, float max_grad_norm, float grad_scale, int32_t* step_counter,
                  float* grad_norm_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif
