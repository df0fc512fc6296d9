// ppo_api.cu -- C ABI of the PPO rollout kernels (include/fwppo.h).  Thin argument checking over ppo_kernels.cu.
#include "../../include/fwppo.h"
#include "../../include/fwsim.h"
#include "ppo_kernels.h"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>

// error string shared with fw_api.cu through fw_last_error(): set via this hook
extern "C" void fw_set_last_error_(const char* msg);

static int pfail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    fw_set_last_error_(buf);
    return code;
}

#define PCU(call)                                                                               \
    do {                                                                                        \
        cudaError_t _e = (call);                                                                \
        if (_e != cudaSuccess) return pfail(FW_ECUDA, "%s: %s", #call, cudaGetErrorString(_e)); \
    } while (0)

static int check_d(int d) {
    if (d < 1 || d > PPO_MAX_OBS) return pfail(FW_EINVAL, "obs width %d out of range [1,%d]", d, PPO_MAX_OBS);
    return FW_OK;
}
// the tcgen05 kernels (K4 forward, K6 minibatch gradient) stage one 32-wide K slab of observations per tile
static int check_d_tc(int d) {
    if (d < 1 || d > PPO_TC_MAX_OBS)
        return pfail(FW_EINVAL, "obs width %d out of range [1,%d] for the tensor-core kernels (use the CUDA-core forward / "
                                "the torch update)", d, PPO_TC_MAX_OBS);
    return FW_OK;
}

static int check_a(int a) {
    if (a != 4 && a != 6) return pfail(FW_EINVAL, "action width %d not supported (4 or 6)", a);
    return 0;
}

extern "C" int ppo_param_count_a(int32_t d, int32_t a) {
    const int H = PPO_HIDDEN;
    return (H * d + H + H * H + H + a * H + a) + (H * d + H + H * H + H + H + 1) + a;
}
extern "C" int ppo_param_count(int32_t d) { return ppo_param_count_a(d, PPO_ACT); }

extern "C" int ppo_policy_forward_a(const float* params, int32_t d, int32_t a, const float* obs_raw, const double* obs_stats,
                                    float clip_obs, int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step,
                                    const uint32_t* step_dev, int32_t deterministic, float* obs_norm, float* act_env,
                                    float* act_raw, float* logp, float* value, void* stream) {
    if (!params || !obs_raw || !act_env || !value) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    if ((reinterpret_cast<uintptr_t>(act_env) & 15u) || (act_raw && (reinterpret_cast<uintptr_t>(act_raw) & 15u)))
        return pfail(FW_EINVAL, "action buffers must be 16-byte aligned");
    PCU(ppok_forward(params, d, obs_raw, obs_stats, clip_obs, n, seed, env_id0, step, step_dev, deterministic, obs_norm,
                     act_env, act_raw, logp, value, 1, (cudaStream_t)stream, nullptr, 0.0f, nullptr, a));
    return FW_OK;
}

extern "C" int ppo_value_forward_a(const float* params, int32_t d, int32_t a, const float* obs_raw, const double* obs_stats,
                                   float clip_obs, int32_t n, float* value, void* stream) {
    if (!params || !obs_raw || !value) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    PCU(ppok_forward(params, d, obs_raw, obs_stats, clip_obs, n, 0, 0, 0, nullptr, 1, nullptr, nullptr, nullptr, nullptr,
                     value, 0, (cudaStream_t)stream, nullptr, 0.0f, nullptr, a));
    return FW_OK;
}

extern "C" int ppo_timeout_bootstrap_a(const float* params, int32_t d, int32_t a, const float* term_obs_raw,
                                       const double* obs_stats, float clip_obs, const uint8_t* flags, int32_t n, float gamma,
                                       float* rew_inout, void* stream) {
    if (!params || !term_obs_raw || !flags || !rew_inout) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    PCU(ppok_bootstrap(params, d, term_obs_raw, obs_stats, clip_obs, flags, n, gamma, rew_inout, nullptr,
                       (cudaStream_t)stream, a));
    return FW_OK;
}

extern "C" int ppo_moments_update(const float* x, int32_t n, int32_t d, double* stats, double* scratch, double* accum,
                                  void* stream) {
    if (!x || !stats || !scratch) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    PCU(ppok_moments(x, n, d, stats, scratch, accum, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_moments_finalize(double* acc, int32_t slots, int32_t n, int32_t d, double* stats, double* accum, void* stream) {
    if (!acc || !stats) return pfail(FW_EINVAL, "null argument");
    if (n <= 0 || slots <= 0) return pfail(FW_EINVAL, "n and slots must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    PCU(ppok_moments_finalize(acc, slots, n, d, stats, accum, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_policy_forward(const float* params, int32_t d, const float* obs_raw, const double* obs_stats,
                                  float clip_obs, int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step,
                                  const uint32_t* step_dev, int32_t deterministic, float* obs_norm, float* act_env,
                                  float* act_raw, float* logp, float* value, void* stream) {
    if (!params || !obs_raw || !act_env || !value) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    if ((reinterpret_cast<uintptr_t>(act_env) & 15u) || (act_raw && (reinterpret_cast<uintptr_t>(act_raw) & 15u)))
        return pfail(FW_EINVAL, "action buffers must be 16-byte aligned");
    PCU(ppok_forward(params, d, obs_raw, obs_stats, clip_obs, n, seed, env_id0, step, step_dev, deterministic, obs_norm,
                     act_env, act_raw, logp, value, 1, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_policy_forward_tc_a(const float* params, int32_t d, int32_t a, const float* obs_raw,
                                       const double* obs_stats, float clip_obs, int32_t n, uint64_t seed, uint32_t env_id0,
                                       uint32_t step, const uint32_t* step_dev, int32_t deterministic, float* obs_norm,
                                       float* act_env, float* act_raw, float* logp, float* value, void* stream) {
    if (!params || !obs_raw || !act_env || !value) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = (a == 4) ? check_d(d) : check_d_tc(d);        // 64-wide build for four-channel policies (ppo_tc_d64.cu)
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    if ((reinterpret_cast<uintptr_t>(act_env) & 15u) || (act_raw && (reinterpret_cast<uintptr_t>(act_raw) & 15u)))
        return pfail(FW_EINVAL, "action buffers must be 16-byte aligned");
    if (a == 4 && d > PPO_TC_MAX_OBS)
        PCU(ppo_a4d64::ppok_forward_tc(params, d, obs_raw, obs_stats, clip_obs, n, seed, env_id0, step, step_dev, deterministic,
                                       obs_norm, act_env, act_raw, logp, value, (cudaStream_t)stream));
    else if (a == 4)
        PCU(ppo_a4::ppok_forward_tc(params, d, obs_raw, obs_stats, clip_obs, n, seed, env_id0, step, step_dev, deterministic,
                                    obs_norm, act_env, act_raw, logp, value, (cudaStream_t)stream));
    else
        PCU(ppo_a6::ppok_forward_tc(params, d, obs_raw, obs_stats, clip_obs, n, seed, env_id0, step, step_dev, deterministic,
                                    obs_norm, act_env, act_raw, logp, value, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_policy_forward_tc(const float* params, int32_t d, const float* obs_raw, const double* obs_stats,
                                     float clip_obs, int32_t n, uint64_t seed, uint32_t env_id0, uint32_t step,
                                     const uint32_t* step_dev, int32_t deterministic, float* obs_norm, float* act_env,
                                     float* act_raw, float* logp, float* value, void* stream) {
    return ppo_policy_forward_tc_a(params, d, PPO_ACT, obs_raw, obs_stats, clip_obs, n, seed, env_id0, step, step_dev,
                                   deterministic, obs_norm, act_env, act_raw, logp, value, stream);
}

extern "C" int ppo_value_forward(const float* params, int32_t d, const float* obs_raw, const double* obs_stats,
                                 float clip_obs, int32_t n, float* value, void* stream) {
    if (!params || !obs_raw || !value) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    PCU(ppok_forward(params, d, obs_raw, obs_stats, clip_obs, n, 0, 0, 0, nullptr, 1, nullptr, nullptr, nullptr, nullptr,
                     value, 0, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_reward_normalize(const float* rew, const uint8_t* flags, int32_t n, float gamma, float clip_rew,
                                    float* ret, double* ret_stats, double* scratch, double* accum, float* rew_norm,
                                    float* done_out, void* stream) {
    if (!rew || !flags || !ret || !ret_stats || !scratch || !rew_norm) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    PCU(ppok_reward_normalize(rew, flags, n, gamma, clip_rew, ret, ret_stats, scratch, accum, rew_norm, done_out,
                              (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_timeout_bootstrap(const float* params, int32_t d, const float* term_obs_raw, const double* obs_stats,
                                     float clip_obs, const uint8_t* flags, int32_t n, float gamma, float* rew_inout,
                                     float* value_scratch, void* stream) {
    if (!params || !term_obs_raw || !flags || !rew_inout || !value_scratch) return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    int rc = check_d(d);
    if (rc) return rc;
    PCU(ppok_bootstrap(params, d, term_obs_raw, obs_stats, clip_obs, flags, n, gamma, rew_inout, value_scratch,
                       (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_gae(const float* rewards, const float* values, const float* dones, const float* last_values, int32_t T,
                       int32_t n, float gamma, float lam, float* advantages, float* returns, void* stream) {
    if (!rewards || !values || !dones || !last_values || !advantages || !returns) return pfail(FW_EINVAL, "null argument");
    if (T <= 0 || n <= 0) return pfail(FW_EINVAL, "T and n must be positive");
    PCU(ppok_gae(rewards, values, dones, last_values, T, n, gamma, lam, advantages, returns, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_random_permutation(int64_t* out, int64_t n, uint64_t seed, uint64_t epoch, void* stream) {
    if (!out || n < 0) return pfail(FW_EINVAL, "ppo_random_permutation: null output or negative length");
    if (n >= (1ll << 62)) return pfail(FW_EINVAL, "ppo_random_permutation: n too large");
    PCU(ppok_permutation(reinterpret_cast<long long*>(out), (long long)n, seed, epoch, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_random_permutation_window(int64_t* out, int64_t n, uint64_t seed, uint32_t* counters, int64_t window_len,
                                             void* stream) {
    if (!out || !counters || n < 0 || window_len <= 0)
        return pfail(FW_EINVAL, "ppo_random_permutation_window: null argument, negative length or empty window");
    if (n >= (1ll << 62)) return pfail(FW_EINVAL, "ppo_random_permutation_window: n too large");
    PCU(ppok_permutation_window(reinterpret_cast<long long*>(out), (long long)n, seed, counters, (long long)window_len,
                                (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_counter_add(uint32_t* counter, uint32_t inc, void* stream) {
    if (!counter) return pfail(FW_EINVAL, "null argument");
    PCU(ppok_counter_add(counter, inc, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int ppo_eval_ledger(const float* rew, const uint8_t* flags, const uint8_t* targets_reached, int32_t n, double* ret,
                               int32_t* len, int32_t* count, const int32_t* quota, const int32_t* offset, uint32_t step,
                               const uint32_t* step_dev, int32_t step_limit, int32_t* remaining, double* ep_return,
                               int32_t* ep_length, uint8_t* ep_targets, uint8_t* ep_flags, int32_t* ep_step, void* stream) {
    if (!rew || !flags || !ret || !len || !count || !quota || !offset || !step_dev || !remaining || !ep_return || !ep_length ||
        !ep_targets || !ep_flags || !ep_step)
        return pfail(FW_EINVAL, "null argument");
    if (n <= 0) return pfail(FW_EINVAL, "n must be positive");
    if (step_limit < 0) return pfail(FW_EINVAL, "step_limit must not be negative");
    PCU(ppok_eval_ledger(rew, flags, targets_reached, n, ret, len, count, quota, offset, step, step_dev, step_limit, remaining,
                         ep_return, ep_length, ep_targets, ep_flags, ep_step, (cudaStream_t)stream));
    return FW_OK;
}

// workspace layout (floats): [0,8) arrival counter of the reduce+Adam kernel (unsigned, starts zeroed) + pad | [8,16) adv stats
// of a single-minibatch call | [16, 16 + 160*P) per-CTA gradient partials | 160*8 per-CTA loss statistics | PPO_MAX_WINDOW
// scratch slices of PPO_ADV_SCRATCH floats (doubles: arrival counter + 592 block partials; the counters start zeroed and
// the kernel leaves them zeroed) | 2 * PPO_MAX_WINDOW floats: advantage statistics of a window's minibatches
#define PPO_ADV_SCRATCH (2 * (2 + 2 * 592))
extern "C" int ppo_update_workspace_floats_a(int32_t d, int32_t a) {
    return 16 + 160 * ppo_param_count_a(d, a) + 160 * 8 + PPO_MAX_WINDOW * PPO_ADV_SCRATCH + 2 * PPO_MAX_WINDOW;
}
extern "C" int ppo_update_workspace_floats(int32_t d) { return ppo_update_workspace_floats_a(d, PPO_ACT); }

extern "C" int ppo_minibatch_grad_a(const float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                                    const float* logp_old, const float* adv, const float* ret, const int64_t* idx,
                                    int32_t batch, float clip_range, float ent_coef, float vf_coef, float* workspace,
                                    float* grad, float* stats, void* stream) {
    if (!params || !obs_norm || !act || !logp_old || !adv || !ret || !idx || !workspace || !grad)
        return pfail(FW_EINVAL, "null argument");
    if (batch <= 0) return pfail(FW_EINVAL, "batch must be positive");
    // one 32-wide observation slab for both action widths; a 64-wide one (bf16-split layer 2) for four-channel policies
    int rc = (a == 4) ? check_d(d) : check_d_tc(d);
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    if ((reinterpret_cast<uintptr_t>(workspace) & 15u) || (reinterpret_cast<uintptr_t>(act) & 15u))
        return pfail(FW_EINVAL, "workspace and action buffer must be 16-byte aligned");
    const int P = ppo_param_count_a(d, a);
    if (ppok_update_grid(batch) > 160) return pfail(FW_ESTATE, "more SMs than the workspace was sized for");
    float* adv_stats = workspace + 8;
    float* partial = workspace + 16;
    float* stats_partial = partial + (size_t)160 * P;
    // 8-byte aligned: the workspace is 16-byte aligned and 16 + 160 * (P + 8) is even
    double* scratch = reinterpret_cast<double*>(stats_partial + 160 * 8);
    if (a == 4 && d > PPO_TC_MAX_OBS)
        PCU(ppo_a4d64::ppok_minibatch_grad(params, d, obs_norm, act, logp_old, adv, ret, reinterpret_cast<const long long*>(idx), batch,
                                           clip_range, ent_coef, vf_coef, scratch, adv_stats, partial, stats_partial, grad, stats,
                                           (cudaStream_t)stream));
    else if (a == 4)
        PCU(ppo_a4::ppok_minibatch_grad(params, d, obs_norm, act, logp_old, adv, ret, reinterpret_cast<const long long*>(idx), batch,
                                        clip_range, ent_coef, vf_coef, scratch, adv_stats, partial, stats_partial, grad, stats,
                                        (cudaStream_t)stream));
    else
        PCU(ppo_a6::ppok_minibatch_grad(params, d, obs_norm, act, logp_old, adv, ret, reinterpret_cast<const long long*>(idx), batch,
                                        clip_range, ent_coef, vf_coef, scratch, adv_stats, partial, stats_partial, grad, stats,
                                        (cudaStream_t)stream));
    return FW_OK;
}

static int minibatch_steps_impl(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                                     const float* logp_old, const float* adv, const float* ret, const int64_t* idx,
                                     int32_t batch, int32_t steps, float clip_range, float ent_coef, float vf_coef,
                                     float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                     float max_grad_norm, int32_t* step_counter, float* grad_norm_out, float* grad, float* stats,
                                     void* stream, int world, int rank, void* const* peers, uint32_t* seq) {
    if (!params || !obs_norm || !act || !logp_old || !adv || !ret || !idx || !exp_avg || !exp_avg_sq || !step_counter || !grad ||
        !stats)
        return pfail(FW_EINVAL, "null argument");
    if (batch <= 0 || batch > PPO_FUSED_MAX_BATCH)
        return pfail(FW_EINVAL, "batch %d out of range [1,%d] for the single-CTA optimizer steps", batch, PPO_FUSED_MAX_BATCH);
    if (steps <= 0) return pfail(FW_EINVAL, "steps must be positive");
    int rc = (a == 4) ? check_d(d) : check_d_tc(d);
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    if (reinterpret_cast<uintptr_t>(act) & 15u) return pfail(FW_EINVAL, "action buffer must be 16-byte aligned");
    if (ppo_param_count_a(d, a) > 16384) return pfail(FW_EINVAL, "parameter vector too long");
    const long long* ix = reinterpret_cast<const long long*>(idx);
    cudaStream_t st = (cudaStream_t)stream;
#define STEPS_ARGS params, d, obs_norm, act, logp_old, adv, ret, ix, batch, steps, clip_range, ent_coef, vf_coef, exp_avg, exp_avg_sq, \
                   lr, beta1, beta2, eps, max_grad_norm, step_counter, grad_norm_out, grad, stats, st, world, rank, peers, seq
    if (a == 4 && d > PPO_TC_MAX_OBS) PCU(ppo_a4d64::ppok_minibatch_steps(STEPS_ARGS));
    else if (a == 4) PCU(ppo_a4::ppok_minibatch_steps(STEPS_ARGS));
    else PCU(ppo_a6::ppok_minibatch_steps(STEPS_ARGS));
#undef STEPS_ARGS
    return FW_OK;
}

extern "C" int ppo_minibatch_steps_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                                     const float* logp_old, const float* adv, const float* ret, const int64_t* idx,
                                     int32_t batch, int32_t steps, float clip_range, float ent_coef, float vf_coef,
                                     float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                     float max_grad_norm, int32_t* step_counter, float* grad_norm_out, float* grad, float* stats,
                                     void* stream) {
    return minibatch_steps_impl(params, d, a, obs_norm, act, logp_old, adv, ret, idx, batch, steps, clip_range, ent_coef, vf_coef, exp_avg,
                                exp_avg_sq, lr, beta1, beta2, eps, max_grad_norm, step_counter, grad_norm_out, grad, stats, stream, 1, 0,
                                nullptr, nullptr);
}

extern "C" int ppo_minibatch_steps_p2p_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                                         const float* logp_old, const float* adv, const float* ret, const int64_t* idx,
                                         int32_t batch, int32_t steps, float clip_range, float ent_coef, float vf_coef,
                                         float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                         float max_grad_norm, int32_t* step_counter, float* grad_norm_out, float* grad,
                                         float* stats, int32_t world, int32_t rank, void* const* peer_buffers, uint32_t* sequence,
                                         void* stream) {
    if (world < 1 || world > 8 || rank < 0 || rank >= world) return pfail(FW_EINVAL, "world must be in [1,8] and rank inside it");
    if (world > 1) {
        if (!peer_buffers || !sequence) return pfail(FW_EINVAL, "null peer buffers or sequence counter");
        for (int j = 0; j < world; ++j)
            if (!peer_buffers[j]) return pfail(FW_EINVAL, "peer buffer %d is null", j);
    }
    return minibatch_steps_impl(params, d, a, obs_norm, act, logp_old, adv, ret, idx, batch, steps, clip_range, ent_coef, vf_coef, exp_avg,
                                exp_avg_sq, lr, beta1, beta2, eps, max_grad_norm, step_counter, grad_norm_out, grad, stats, stream, world,
                                rank, peer_buffers, sequence);
}

static int window_update_impl(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                              const float* logp_old, const float* adv, const float* ret, const int64_t* idx, int32_t batch,
                              int32_t n_minibatches, float clip_range, float ent_coef, float vf_coef, float* exp_avg,
                              float* exp_avg_sq, float lr, float beta1, float beta2, float eps, float max_grad_norm,
                              int32_t* step_counter, float* grad_norm_out, float* workspace, float* grad, float* stats,
                              void* stream, int world, int rank, void* const* peers, uint32_t* seq) {
    if (!params || !obs_norm || !act || !logp_old || !adv || !ret || !idx || !exp_avg || !exp_avg_sq || !step_counter || !workspace ||
        !grad)
        return pfail(FW_EINVAL, "null argument");
    if (batch <= 0) return pfail(FW_EINVAL, "batch must be positive");
    if (n_minibatches <= 0 || n_minibatches > PPO_MAX_WINDOW)
        return pfail(FW_EINVAL, "n_minibatches %d out of range [1,%d]", n_minibatches, PPO_MAX_WINDOW);
    int rc = (a == 4) ? check_d(d) : check_d_tc(d);
    if (rc) return rc;
    if ((rc = check_a(a)) != 0) return rc;
    if ((reinterpret_cast<uintptr_t>(workspace) & 15u) || (reinterpret_cast<uintptr_t>(act) & 15u))
        return pfail(FW_EINVAL, "workspace and action buffer must be 16-byte aligned");
    const int P = ppo_param_count_a(d, a);
    if (P > 16384) return pfail(FW_EINVAL, "parameter vector too long");
    if (ppok_update_grid(batch) > 160) return pfail(FW_ESTATE, "more SMs than the workspace was sized for");
    float* partial = workspace + 16;
    float* stats_partial = partial + (size_t)160 * P;
    double* scratch = reinterpret_cast<double*>(stats_partial + 160 * 8);
    float* win_stats = stats_partial + 160 * 8 + (size_t)PPO_MAX_WINDOW * PPO_ADV_SCRATCH;
    cudaStream_t st = (cudaStream_t)stream;
    const long long* ix = reinterpret_cast<const long long*>(idx);
    // one launch for the advantage statistics of every minibatch of the window, then per minibatch the gradient kernel and
    // the reduction whose last block applies clip + Adam
    ppok_launch_adv_stats(adv, ix, batch, n_minibatches, scratch, win_stats, st);
    PCU(cudaGetLastError());
    PpokAdam adam{lr, beta1, beta2, eps, max_grad_norm, params, exp_avg, exp_avg_sq, step_counter, grad_norm_out,
                  reinterpret_cast<unsigned*>(workspace)};
    if (world > 1) {
        adam.world = world; adam.rank = rank; adam.seq = seq;
        for (int j = 0; j < world; ++j) adam.peer[j] = static_cast<float*>(peers[j]);
    }
    for (int k = 0; k < n_minibatches; ++k) {
        const long long* ik = ix + (size_t)k * batch;
        float* as = win_stats + 2 * k;
        if (a == 4 && d > PPO_TC_MAX_OBS)
            PCU(ppo_a4d64::ppok_minibatch_grad(params, d, obs_norm, act, logp_old, adv, ret, ik, batch, clip_range, ent_coef, vf_coef,
                                               scratch, as, partial, stats_partial, grad, stats, st, &adam, 1));
        else if (a == 4)
            PCU(ppo_a4::ppok_minibatch_grad(params, d, obs_norm, act, logp_old, adv, ret, ik, batch, clip_range, ent_coef, vf_coef,
                                            scratch, as, partial, stats_partial, grad, stats, st, &adam, 1));
        else
            PCU(ppo_a6::ppok_minibatch_grad(params, d, obs_norm, act, logp_old, adv, ret, ik, batch, clip_range, ent_coef, vf_coef,
                                            scratch, as, partial, stats_partial, grad, stats, st, &adam, 1));
    }
    return FW_OK;
}

extern "C" int ppo_window_update_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                                   const float* logp_old, const float* adv, const float* ret, const int64_t* idx, int32_t batch,
                                   int32_t n_minibatches, float clip_range, float ent_coef, float vf_coef, float* exp_avg,
                                   float* exp_avg_sq, float lr, float beta1, float beta2, float eps, float max_grad_norm,
                                   int32_t* step_counter, float* grad_norm_out, float* workspace, float* grad, float* stats,
                                   void* stream) {
    return window_update_impl(params, d, a, obs_norm, act, logp_old, adv, ret, idx, batch, n_minibatches, clip_range, ent_coef, vf_coef,
                              exp_avg, exp_avg_sq, lr, beta1, beta2, eps, max_grad_norm, step_counter, grad_norm_out, workspace, grad,
                              stats, stream, 1, 0, nullptr, nullptr);
}

extern "C" int ppo_window_update_p2p_a(float* params, int32_t d, int32_t a, const float* obs_norm, const float* act,
                                       const float* logp_old, const float* adv, const float* ret, const int64_t* idx,
                                       int32_t batch, int32_t n_minibatches, float clip_range, float ent_coef, float vf_coef,
                                       float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                       float max_grad_norm, int32_t* step_counter, float* grad_norm_out, float* workspace,
                                       float* grad, float* stats, int32_t world, int32_t rank, void* const* peer_buffers,
                                       uint32_t* sequence, void* stream) {
    if (world < 1 || world > 8 || rank < 0 || rank >= world) return pfail(FW_EINVAL, "world must be in [1,8] and rank inside it");
    if (world > 1) {
        if (!peer_buffers || !sequence) return pfail(FW_EINVAL, "null peer buffers or sequence counter");
        for (int j = 0; j < world; ++j)
            if (!peer_buffers[j]) return pfail(FW_EINVAL, "peer buffer %d is null", j);
    }
    return window_update_impl(params, d, a, obs_norm, act, logp_old, adv, ret, idx, batch, n_minibatches, clip_range, ent_coef, vf_coef,
                              exp_avg, exp_avg_sq, lr, beta1, beta2, eps, max_grad_norm, step_counter, grad_norm_out, workspace, grad,
                              stats, stream, world, rank, peer_buffers, sequence);
}

// ---- peer memory for the in-kernel gradient all-reduce: one cudaMalloc'ed exchange buffer per rank, shared through CUDA IPC
extern "C" int64_t ppo_peer_bytes(void) { return (int64_t)ppok_peer_bytes(); }
extern "C" int ppo_peer_alloc(void** out) {
    if (!out) return pfail(FW_EINVAL, "null argument");
    PCU(cudaMalloc(out, ppok_peer_bytes()));
    PCU(cudaMemset(*out, 0, ppok_peer_bytes()));
    PCU(cudaDeviceSynchronize());
    return FW_OK;
}
extern "C" int ppo_peer_free(void* p) { if (p) PCU(cudaFree(p)); return FW_OK; }
extern "C" int ppo_peer_export(void* p, uint8_t handle[64]) {
    if (!p || !handle) return pfail(FW_EINVAL, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    cudaIpcMemHandle_t h;
    PCU(cudaIpcGetMemHandle(&h, p));
    memcpy(handle, &h, 64);
    return FW_OK;
}
extern "C" int ppo_peer_import(const uint8_t handle[64], void** out) {
    if (!handle || !out) return pfail(FW_EINVAL, "null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    PCU(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return FW_OK;
}
extern "C" int ppo_peer_close(void* p) { if (p) PCU(cudaIpcCloseMemHandle(p)); return FW_OK; }

extern "C" int ppo_minibatch_grad(const float* params, int32_t d, const float* obs_norm, const float* act,
                                  const float* logp_old, const float* adv, const float* ret, const int64_t* idx,
                                  int32_t batch, float clip_range, float ent_coef, float vf_coef, float* workspace,
                                  float* grad, float* stats, void* stream) {
    return ppo_minibatch_grad_a(params, d, PPO_ACT, obs_norm, act, logp_old, adv, ret, idx, batch, clip_range, ent_coef, vf_coef,
                                workspace, grad, stats, stream);
}

extern "C" int ppo_adam_step(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t n_params, float lr,
                             float beta1, float beta2, float eps, float max_grad_norm, float grad_scale, int32_t* step_counter,
                             float* grad_norm_out, void* stream) {
    if (!params || !grad || !exp_avg || !exp_avg_sq || !step_counter) return pfail(FW_EINVAL, "null argument");
    if (n_params <= 0) return pfail(FW_EINVAL, "n_params must be positive");
    PCU(ppok_adam(params, grad, exp_avg, exp_avg_sq, n_params, lr, beta1, beta2, eps, max_grad_norm, grad_scale, step_counter,
                  grad_norm_out, (cudaStream_t)stream));
    return FW_OK;
}
