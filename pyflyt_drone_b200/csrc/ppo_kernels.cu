// ppo_kernels.cu -- sm_100a kernels for the PPO rollout path around the env step (include/fwppo.h).
//
// Replaces what the reference obtains from stable_baselines3 (train/train_Fixedwing_Waypoints_v3.py:260,293-337):
// VecNormalize running moments + normalisation, the MlpPolicy forward (pi and vf towers 64-64 tanh, diagonal
// Gaussian head), the time-limit bootstrap and the GAE scan.  All of it runs on device tensors; the host never
// sees an observation during a rollout.
#include "ppo_kernels.h"
#include "ppo_tower.cuh"

#include <cuda_runtime.h>
#include <math_constants.h>

#define H PPO_H
#define A PPO_A
// DP (template parameter below) = observation width padded to 32 or 64 for float4 weight rows: 32 covers the
// 28/29-float Waypoints observations and the 21-float low-level one, 64 the 56-float duck-only ObjLock observation

// ------------------------------------------------------------------ shared helpers
__device__ __forceinline__ uint4 ppo_philox(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float ppo_u01(uint32_t x) { return ((float)(x >> 9) + 0.5f) * (1.0f / 8388608.0f); }

// ------------------------------------------------------------------ K4: policy + value forward, one thread per env
// AO = action width: 4 (roll, pitch, yaw, thrust) or 6 (the low-level env's surface / thrust channels)
// POP: population launch, blockIdx.y = member (see PpokPop): every per-member pointer, the seed and the bootstrap's gamma
// move to the member before the body runs over its `n` rows
template <int AO, int DP, bool POP = false>
__global__ void __launch_bounds__(PPO_FWD_THREADS)
ppo_forward_kernel(const float* __restrict__ params, int d, const float* __restrict__ obs_raw,
                   const double* __restrict__ stats, float clip, int n, uint32_t seed_lo, uint32_t seed_hi,
                   uint32_t env_id0, uint32_t step, const uint32_t* __restrict__ step_dev, int deterministic,
                   float* __restrict__ obs_norm,
                   float* __restrict__ act_env, float* __restrict__ act_raw, float* __restrict__ logp,
                   float* __restrict__ value, int want_policy, const uint8_t* __restrict__ boot_flags, float boot_gamma,
                   float* __restrict__ boot_rew, PpokPop pop) {
    extern __shared__ __align__(16) float smem[];
    if constexpr (POP) {
        const int m = blockIdx.y;
        const size_t r0 = (size_t)m * n;
        params += (size_t)m * pop.param_stride;
        obs_raw += r0 * d;
        if (stats != nullptr) stats += (size_t)m * (2 * d + 1);
        const uint64_t seed = pop.seeds != nullptr ? pop.seeds[m] : 0ull;      // value and bootstrap launches draw no noise
        seed_lo = (uint32_t)(seed & 0xffffffffu); seed_hi = (uint32_t)(seed >> 32);
        env_id0 += (uint32_t)r0;
        if (obs_norm != nullptr) obs_norm += r0 * d;
        if (act_env != nullptr) act_env += r0 * AO;
        if (act_raw != nullptr) act_raw += r0 * AO;
        if (logp != nullptr) logp += r0;
        if (value != nullptr) value += r0;
        if (boot_flags != nullptr) { boot_flags += r0; boot_rew += r0; boot_gamma = pop.hp[m * PPO_POP_HP + PPO_POP_GAMMA]; }
    }
    // time-limit bootstrap mode: only blocks holding a truncated-but-not-terminated row do any work (truncations
    // arrive in bursts -- every env of a synchronised batch hits the step limit together -- and are absent otherwise)
    bool boot_need = false;
    if (boot_flags != nullptr) {
        const int r0 = blockIdx.x * blockDim.x + threadIdx.x;
        if (r0 < n) { const uint32_t f = boot_flags[r0]; boot_need = (f & 2u) != 0 && (f & 1u) == 0; }
        if (!__syncthreads_or(boot_need ? 1 : 0)) return;
    }
    float* s_pi = smem;
    float* s_vf = s_pi + TowerOff<AO, DP>::SIZE;
    float* s_mean = s_vf + TowerOff<1, DP>::SIZE;
    float* s_istd = s_mean + DP;
    float* s_logstd = s_istd + DP;
    float* hbuf = s_logstd + 8;
    const int pi_count = H * d + H + H * H + H + AO * H + AO;
    const int vf_count = H * d + H + H * H + H + H + 1;
    if (want_policy) load_tower<AO, DP>(s_pi, params, d);
    load_tower<1, DP>(s_vf, params + pi_count, d);
    stage_stats<DP>(stats, d, s_mean, s_istd);
    if (threadIdx.x < AO) s_logstd[threadIdx.x] = params[pi_count + vf_count + threadIdx.x];
    __syncthreads();

    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    float x[DP];
    load_obs<DP>(obs_raw, stats ? s_mean : nullptr, s_istd, clip, d, row, x, obs_norm);
    float v[1];
    tower_forward<1, DP>(s_vf, x, hbuf, v);
    if (boot_flags != nullptr) {
        if (boot_need) boot_rew[row] = fmaf(boot_gamma, v[0], boot_rew[row]);    // TimeLimit.truncated
        return;
    }
    value[row] = v[0];
    if (!want_policy) return;
    float mean[AO];
    tower_forward<AO, DP>(s_pi, x, hbuf, mean);
    // diagonal Gaussian: a = mu + sigma * eps ; log pi(a) = sum -0.5 eps^2 - log sigma - 0.5 log 2pi
    const uint32_t step_eff = step + (step_dev != nullptr ? step_dev[0] : 0u);   // device counter: graph-replayable
    float eps[AO];
#pragma unroll
    for (int g = 0; g < (AO + 3) / 4; ++g) {          // four normals per Philox call; channels 4.. use counter word 2 = 1
        uint4 r = ppo_philox(seed_lo, seed_hi, env_id0 + (uint32_t)row, step_eff, (uint32_t)g, 7u);
        float ra = sqrtf(-2.0f * __logf(ppo_u01(r.x))), rb = sqrtf(-2.0f * __logf(ppo_u01(r.z)));
        float s0, c0, s1, c1;
        sincospif(2.0f * ppo_u01(r.y), &s0, &c0);
        sincospif(2.0f * ppo_u01(r.w), &s1, &c1);
        const float e4[4] = {ra * c0, ra * s0, rb * c1, rb * s1};
#pragma unroll
        for (int k = 0; k < 4; ++k) if (4 * g + k < AO) eps[4 * g + k] = e4[k];
    }
    float lp = 0.0f;
    float av[AO], ac[AO];
#pragma unroll
    for (int a = 0; a < AO; ++a) {
        float ls = s_logstd[a];
        float e = deterministic ? 0.0f : eps[a];
        av[a] = fmaf(__expf(ls), e, mean[a]);
        ac[a] = ppo_clip_action(av[a]);
        lp += -0.5f * e * e - ls - 0.91893853320467274178f;
    }
    // rows are AO floats wide: 8-byte aligned for the even widths supported
#pragma unroll
    for (int a = 0; a < AO; a += 2) {
        reinterpret_cast<float2*>(act_env + (size_t)row * AO)[a / 2] = make_float2(ac[a], ac[a + 1]);
        if (act_raw != nullptr) reinterpret_cast<float2*>(act_raw + (size_t)row * AO)[a / 2] = make_float2(av[a], av[a + 1]);
    }
    if (logp != nullptr) logp[row] = lp;
}

template <int AO, int DP>
static size_t ppo_forward_smem_t() {
    return (size_t)(TowerOff<AO, DP>::SIZE + TowerOff<1, DP>::SIZE + 2 * DP + 8 + H * PPO_FWD_THREADS) * sizeof(float);
}
size_t ppo_forward_smem() { return ppo_forward_smem_t<A, 32>(); }

template <int AO, int DP, bool POP = false>
static cudaError_t ppok_forward_t(const float* params, int d, const float* obs_raw, const double* stats, float clip, int n,
                                  uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev, int deterministic,
                                  float* obs_norm, float* act_env, float* act_raw, float* logp, float* value, int want_policy,
                                  cudaStream_t st, const uint8_t* boot_flags, float boot_gamma, float* boot_rew,
                                  const PpokPop& pop = PpokPop{}) {
    static bool attr_set = false;
    const size_t sm = ppo_forward_smem_t<AO, DP>();
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(ppo_forward_kernel<AO, DP, POP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    const dim3 grid((n + PPO_FWD_THREADS - 1) / PPO_FWD_THREADS, POP ? pop.members : 1);
    ppo_forward_kernel<AO, DP, POP><<<grid, PPO_FWD_THREADS, sm, st>>>(params, d, obs_raw, stats, clip, n, (uint32_t)(seed & 0xffffffffu),
                                                                   (uint32_t)(seed >> 32), env_id0, step, step_dev, deterministic,
                                                                   obs_norm, act_env, act_raw, logp, value, want_policy, boot_flags,
                                                                   boot_gamma, boot_rew, pop);
    return cudaGetLastError();
}

cudaError_t ppok_forward(const float* params, int d, const float* obs_raw, const double* stats, float clip, int n,
                         uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev, int deterministic,
                         float* obs_norm, float* act_env, float* act_raw, float* logp, float* value, int want_policy,
                         cudaStream_t st, const uint8_t* boot_flags, float boot_gamma, float* boot_rew, int a) {
    if (d > 64) return cudaErrorInvalidValue;
#define FWD_DISPATCH(AO_, DP_)                                                                                             \
    return ppok_forward_t<AO_, DP_>(params, d, obs_raw, stats, clip, n, seed, env_id0, step, step_dev, deterministic, obs_norm, \
                                    act_env, act_raw, logp, value, want_policy, st, boot_flags, boot_gamma, boot_rew)
    if (a == 4 && d <= 32) FWD_DISPATCH(4, 32);
    if (a == 6 && d <= 32) FWD_DISPATCH(6, 32);
    if (a == 4) FWD_DISPATCH(4, 64);                 // the 56-float duck-only ObjLock observation
#undef FWD_DISPATCH
    return cudaErrorInvalidValue;
}

cudaError_t ppok_pop_forward(const PpokPop& pop, const float* params, int d, const float* obs_raw, const double* stats, float clip,
                             int n, uint32_t env_id0, uint32_t step, const uint32_t* step_dev, int deterministic, float* obs_norm,
                             float* act_env, float* act_raw, float* logp, float* value, int want_policy, cudaStream_t st,
                             const uint8_t* boot_flags, float* boot_rew, int a) {
    if (d > 64) return cudaErrorInvalidValue;
#define FWD_DISPATCH(AO_, DP_)                                                                                               \
    return ppok_forward_t<AO_, DP_, true>(params, d, obs_raw, stats, clip, n, 0, env_id0, step, step_dev, deterministic, obs_norm, \
                                          act_env, act_raw, logp, value, want_policy, st, boot_flags, 0.0f, boot_rew, pop)
    if (a == 4 && d <= 32) FWD_DISPATCH(4, 32);
    if (a == 6 && d <= 32) FWD_DISPATCH(6, 32);
    if (a == 4) FWD_DISPATCH(4, 64);
#undef FWD_DISPATCH
    return cudaErrorInvalidValue;
}

// ------------------------------------------------------------------ K7: running moments (RunningMeanStd.update)
// scratch = double[2*d + 2]: column sums, column sums of squares, block-arrival counter (as double), spare.
#define MOM_ROWS 128          // rows per block: 512 blocks at 65,536 envs, every load of a thread in flight at once
// POP: blockIdx.y = member, n = rows per member; the member's rows, statistics, scratch and accumulator
template <bool POP = false>
__global__ void __launch_bounds__(256)
ppo_moments_kernel(const float* __restrict__ x, int n, int d, double* __restrict__ stats, double* __restrict__ scratch,
                   double* __restrict__ accum, int rows_per_block) {
    __shared__ float s_sum[8][32], s_sq[8][32];
    __shared__ bool is_last;
    if constexpr (POP) {
        const int m = blockIdx.y;
        x += (size_t)m * n * d;
        stats += (size_t)m * (2 * d + 1);
        scratch += (size_t)m * (2 * d + 2);
        if (accum != nullptr) accum += (size_t)m * (2 * d + 1);
    }
    // thread layout: 32 columns x 8 row-lanes; a warp reads 32 consecutive floats of one row when d == 32, and
    // d/32 of a 128-byte line otherwise (rows are contiguous, so the block still streams whole lines)
    const int lane_row = threadIdx.x >> 5;
    const int r0 = blockIdx.x * rows_per_block, r1 = min(n, r0 + rows_per_block);
    for (int c0 = 0; c0 < d; c0 += 32) {             // observations wider than 32 floats: one pass per 32-column chunk
        const int col = c0 + (threadIdx.x & 31);
        float sum = 0.0f, sq = 0.0f;
        if (col < d) {
            // all of this thread's loads are issued before the first add (MOM_ROWS / 8 = 16 independent requests)
            float v[MOM_ROWS / 8];
#pragma unroll
            for (int k = 0; k < MOM_ROWS / 8; ++k) {
                const int r = r0 + lane_row + 8 * k;
                v[k] = r < r1 ? x[(size_t)r * d + col] : 0.0f;
            }
#pragma unroll
            for (int k = 0; k < MOM_ROWS / 8; ++k) { sum += v[k]; sq = fmaf(v[k], v[k], sq); }
        }
        if (c0) __syncthreads();                     // the previous chunk's partials have been consumed
        s_sum[lane_row][threadIdx.x & 31] = sum; s_sq[lane_row][threadIdx.x & 31] = sq;
        __syncthreads();
        if (lane_row == 0 && col < d) {
            double a = 0.0, b = 0.0;
            for (int k = 0; k < 8; ++k) { a += (double)s_sum[k][threadIdx.x & 31]; b += (double)s_sq[k][threadIdx.x & 31]; }
            atomicAdd(&scratch[col], a);
            atomicAdd(&scratch[d + col], b);
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        double prev = atomicAdd(&scratch[2 * d], 1.0);
        is_last = (prev == (double)(gridDim.x - 1));
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // the last block folds the batch moments into the running ones (Chan et al., as SB3's update_from_moments)
    if (threadIdx.x < d) {
        const int k = threadIdx.x;
        volatile double* sc = scratch;
        if (accum != nullptr) { accum[k] += sc[k]; accum[d + k] += sc[d + k]; }   // raw sums for cross-rank merges
        double bmean = sc[k] / n;
        double bvar = sc[d + k] / n - bmean * bmean;
        if (bvar < 0.0) bvar = 0.0;
        double count = stats[2 * d], mean = stats[k], var = stats[d + k];
        double tot = count + (double)n, delta = bmean - mean;
        double m2 = var * count + bvar * (double)n + delta * delta * count * (double)n / tot;
        stats[k] = mean + delta * (double)n / tot;
        stats[d + k] = m2 / tot;
    }
    __syncthreads();
    if (threadIdx.x == 0) { stats[2 * d] += (double)n; if (accum != nullptr) accum[2 * d] += (double)n; }
    // leave the scratch zeroed for the next call
    for (int k = threadIdx.x; k < 2 * d + 2; k += blockDim.x) scratch[k] = 0.0;
}

// The same merge for batch sums the env-step kernels accumulated in their epilogue (fw_set_obs_accumulator): acc =
// slots x double[2 d]; summed in slot order, folded into the running statistics, zeroed for the next step.
#define MOMF_GROUPS 4          // slot groups: 256 threads = 4 groups x 64 columns, every load of a thread issued before its first add
__global__ void __launch_bounds__(64 * MOMF_GROUPS)
ppo_moments_finalize_kernel(double* __restrict__ acc, int slots, int n, int d, double* __restrict__ stats, double* __restrict__ accum) {
    __shared__ double s_a[MOMF_GROUPS][64], s_b[MOMF_GROUPS][64];
    const int k = threadIdx.x & 63, g = threadIdx.x >> 6;
    constexpr int PER = 16;                              // slots per thread: slots <= MOMF_GROUPS * PER
    double a = 0.0, b = 0.0;
    if (k < d) {
        double va[PER], vb[PER];
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int s = g * PER + i;
            va[i] = s < slots ? acc[(size_t)s * 2 * d + k] : 0.0;
            vb[i] = s < slots ? acc[(size_t)s * 2 * d + d + k] : 0.0;
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int s = g * PER + i;
            a += va[i]; b += vb[i];
            if (s < slots) { acc[(size_t)s * 2 * d + k] = 0.0; acc[(size_t)s * 2 * d + d + k] = 0.0; }
        }
    }
    s_a[g][k] = a; s_b[g][k] = b;
    __syncthreads();
    if (g == 0 && k < d) {
        a = 0.0; b = 0.0;
#pragma unroll
        for (int i = 0; i < MOMF_GROUPS; ++i) { a += s_a[i][k]; b += s_b[i][k]; }      // slot order: deterministic
        if (accum != nullptr) { accum[k] += a; accum[d + k] += b; }
        double bmean = a / n;
        double bvar = b / n - bmean * bmean;
        if (bvar < 0.0) bvar = 0.0;
        double count = stats[2 * d], mean = stats[k], var = stats[d + k];
        double tot = count + (double)n, delta = bmean - mean;
        double m2 = var * count + bvar * (double)n + delta * delta * count * (double)n / tot;
        stats[k] = mean + delta * (double)n / tot;
        stats[d + k] = m2 / tot;
    }
    __syncthreads();
    if (threadIdx.x == 0) { stats[2 * d] += (double)n; if (accum != nullptr) accum[2 * d] += (double)n; }
}

cudaError_t ppok_moments_finalize(double* acc, int slots, int n, int d, double* stats, double* accum, cudaStream_t st) {
    if (d > 64 || slots > MOMF_GROUPS * 16) return cudaErrorInvalidValue;
    ppo_moments_finalize_kernel<<<1, 64 * MOMF_GROUPS, 0, st>>>(acc, slots, n, d, stats, accum);
    return cudaGetLastError();
}

cudaError_t ppok_moments(const float* x, int n, int d, double* stats, double* scratch, double* accum, cudaStream_t st) {
    const int rows_per_block = MOM_ROWS;
    const int grid = (n + rows_per_block - 1) / rows_per_block;
    ppo_moments_kernel<<<grid, 256, 0, st>>>(x, n, d, stats, scratch, accum, rows_per_block);
    return cudaGetLastError();
}

cudaError_t ppok_pop_moments(const PpokPop& pop, const float* x, int n, int d, double* stats, double* scratch, double* accum,
                             cudaStream_t st) {
    const dim3 grid((n + MOM_ROWS - 1) / MOM_ROWS, pop.members);
    ppo_moments_kernel<true><<<grid, 256, 0, st>>>(x, n, d, stats, scratch, accum, MOM_ROWS);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ VecNormalize reward path (two launches: the
// normalisation needs the variance that includes this very batch of returns)
// POP (both kernels): blockIdx.y = member, n = rows per member; the member's rows, return statistics, scratch (4 doubles per
// member) and accumulator, and its gamma
template <bool POP = false>
__global__ void __launch_bounds__(256)
ppo_ret_kernel(const float* __restrict__ rew, int n, float gamma, float* __restrict__ ret, double* __restrict__ ret_stats,
               double* __restrict__ scratch, double* __restrict__ accum, const float* __restrict__ pop_hp = nullptr) {
    __shared__ double s_a[8], s_b[8];
    __shared__ bool is_last;
    if constexpr (POP) {
        const int m = blockIdx.y;
        rew += (size_t)m * n; ret += (size_t)m * n; ret_stats += 3 * m; scratch += 4 * m;
        if (accum != nullptr) accum += 3 * m;
        gamma = pop_hp[m * PPO_POP_HP + PPO_POP_GAMMA];
    }
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float v = 0.0f;
    if (i < n) { v = fmaf(ret[i], gamma, rew[i]); ret[i] = v; }
    double a = (i < n) ? (double)v : 0.0, b = a * a;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    if ((threadIdx.x & 31) == 0) { s_a[threadIdx.x >> 5] = a; s_b[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ta = 0, tb = 0;
        for (int k = 0; k < 8; ++k) { ta += s_a[k]; tb += s_b[k]; }
        atomicAdd(&scratch[0], ta); atomicAdd(&scratch[1], tb);
        __threadfence();
        double prev = atomicAdd(&scratch[2], 1.0);
        is_last = (prev == (double)(gridDim.x - 1));
    }
    __syncthreads();
    if (!is_last || threadIdx.x != 0) return;
    __threadfence();
    volatile double* sc = scratch;
    if (accum != nullptr) { accum[0] += sc[0]; accum[1] += sc[1]; accum[2] += (double)n; }
    double bmean = sc[0] / n, bvar = sc[1] / n - bmean * bmean;
    if (bvar < 0.0) bvar = 0.0;
    double mean = ret_stats[0], var = ret_stats[1], count = ret_stats[2];
    double tot = count + (double)n, delta = bmean - mean;
    double m2 = var * count + bvar * (double)n + delta * delta * count * (double)n / tot;
    ret_stats[0] = mean + delta * (double)n / tot;
    ret_stats[1] = m2 / tot;
    ret_stats[2] = tot;
    scratch[0] = 0.0; scratch[1] = 0.0; scratch[2] = 0.0;
}

template <bool POP = false>
__global__ void __launch_bounds__(256)
ppo_rew_finalize_kernel(const float* __restrict__ rew, const uint8_t* __restrict__ flags, int n, float clip,
                        float* __restrict__ ret, const double* __restrict__ ret_stats, float* __restrict__ rew_norm,
                        float* __restrict__ done_out) {
    if constexpr (POP) {
        const size_t r0 = (size_t)blockIdx.y * n;
        rew += r0; flags += r0; ret += r0; ret_stats += 3 * blockIdx.y; rew_norm += r0;
        if (done_out != nullptr) done_out += r0;
    }
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float istd = (float)(1.0 / sqrt(ret_stats[1] + 1e-8));
    const bool done = (flags[i] & 3u) != 0;
    rew_norm[i] = fminf(fmaxf(rew[i] * istd, -clip), clip);
    if (done) ret[i] = 0.0f;
    if (done_out != nullptr) done_out[i] = done ? 1.0f : 0.0f;
}

cudaError_t ppok_reward_normalize(const float* rew, const uint8_t* flags, int n, float gamma, float clip, float* ret,
                                  double* ret_stats, double* scratch, double* accum, float* rew_norm, float* done_out,
                                  cudaStream_t st) {
    const int grid = (n + 255) / 256;
    ppo_ret_kernel<<<grid, 256, 0, st>>>(rew, n, gamma, ret, ret_stats, scratch, accum);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ppo_rew_finalize_kernel<<<grid, 256, 0, st>>>(rew, flags, n, clip, ret, ret_stats, rew_norm, done_out);
    return cudaGetLastError();
}

cudaError_t ppok_pop_reward_normalize(const PpokPop& pop, const float* rew, const uint8_t* flags, int n, float clip, float* ret,
                                      double* ret_stats, double* scratch, double* accum, float* rew_norm, float* done_out,
                                      cudaStream_t st) {
    const dim3 grid((n + 255) / 256, pop.members);
    ppo_ret_kernel<true><<<grid, 256, 0, st>>>(rew, n, 0.0f, ret, ret_stats, scratch, accum, pop.hp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ppo_rew_finalize_kernel<true><<<grid, 256, 0, st>>>(rew, flags, n, clip, ret, ret_stats, rew_norm, done_out);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ time-limit bootstrap
// r += gamma * V(terminal_obs) for rows that were truncated but not terminated: the batched value forward in its
// bootstrap mode (blocks without such a row exit before staging the weights; a masked per-row MLP reading weights
// from global memory measured 100+ us per step during a truncation burst, the unmasked forward 80 us on every step).
cudaError_t ppok_bootstrap(const float* params, int d, const float* term_obs, const double* stats, float clip,
                           const uint8_t* flags, int n, float gamma, float* rew, float* value_scratch, cudaStream_t st, int a) {
    (void)value_scratch;
    return ppok_forward(params, d, term_obs, stats, clip, n, 0, 0, 0, nullptr, 1, nullptr, nullptr, nullptr, nullptr,
                        nullptr, 0, st, flags, gamma, rew, a);
}

// ------------------------------------------------------------------ minibatch permutation
// A keyed pseudo-random permutation of [0, n): 4-round Feistel network on 2*hb bits (2^(2 hb) >= n) with cycle walking.
// Replaces torch.randperm (a 4 M-key radix sort, ~0.4 ms per epoch at 65,536 envs x 64 steps) by one ~20 us pass;
// every epoch gets a fresh key.  stable_baselines3 draws np.random.permutation here (RolloutBuffer.get).
__device__ __forceinline__ uint32_t ppo_mix32(uint32_t x, uint32_t k) {
    x ^= k; x *= 0x9E3779B1u; x ^= x >> 15; x *= 0x85EBCA77u; x ^= x >> 13; x *= 0xC2B2AE3Du; x ^= x >> 16;
    return x;
}
__host__ __device__ __forceinline__ void ppo_perm_keys(uint64_t seed, uint64_t epoch, uint32_t& k0, uint32_t& k1) {
    k0 = (uint32_t)(seed ^ (epoch * 0x9E3779B97F4A7C15ull));
    k1 = (uint32_t)((seed >> 32) ^ ((epoch * 0xC2B2AE3D27D4EB4Full) >> 32) ^ 0xA5A5A5A5u);
}

// POP: blockIdx.y = member; its permutation of [0, n) (n = its sample count) with its own seed, written to out[m * n ..] as
// population rows (k / rows) * members * rows + m * rows + k % rows of the time-major [T, members * rows] rollout buffers
template <bool POP = false>
__global__ void __launch_bounds__(256)
ppo_permutation_kernel(long long* __restrict__ out, long long n, int hb, uint32_t k0, uint32_t k1, PpokPop pop) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if constexpr (POP) {
        out += (size_t)blockIdx.y * n;
        ppo_perm_keys(pop.seeds[blockIdx.y], pop.epoch, k0, k1);
    }
    const uint32_t mask = (1u << hb) - 1u;
    unsigned long long x = (unsigned long long)i;
    do {                                     // cycle walking: re-encrypt until the value falls inside [0, n)
        uint32_t L = (uint32_t)(x >> hb) & mask, R = (uint32_t)x & mask;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const uint32_t t = L ^ (ppo_mix32(R, k0 + 0x9E3779B9u * (uint32_t)r) ^ ppo_mix32(R ^ k1, (uint32_t)r)) & mask;
            L = R; R = t & mask;
        }
        x = ((unsigned long long)L << hb) | R;
    } while (x >= (unsigned long long)n);
    if constexpr (POP) {
        const long long rows = pop.rows, k = (long long)x;
        x = (unsigned long long)((k / rows) * pop.members * rows + (long long)blockIdx.y * rows + k % rows);
    }
    out[i] = (long long)x;
}

__device__ __forceinline__ long long ppo_perm_at(long long i, long long n, int hb, uint32_t k0, uint32_t k1) {
    const uint32_t mask = (1u << hb) - 1u;
    unsigned long long x = (unsigned long long)i;
    do {
        uint32_t L = (uint32_t)(x >> hb) & mask, R = (uint32_t)x & mask;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const uint32_t t = L ^ (ppo_mix32(R, k0 + 0x9E3779B9u * (uint32_t)r) ^ ppo_mix32(R ^ k1, (uint32_t)r)) & mask;
            L = R; R = t & mask;
        }
        x = ((unsigned long long)L << hb) | R;
    } while (x >= (unsigned long long)n);
    return (long long)x;
}

// The same permutation, one window at a time, with (epoch, window) read from device memory: the launch arguments never
// change, so a CUDA graph of "window of indices -> its minibatch updates" can be replayed for every window of every epoch.
// out[t] = perm_epoch(window * window_len + t)
__global__ void __launch_bounds__(256)
ppo_permutation_window_kernel(long long* __restrict__ out, long long n, int hb, uint64_t seed, const uint32_t* __restrict__ ctr,
                              long long window_len) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i = (long long)ctr[1] * window_len + t;
    if (t >= window_len || i >= n) return;
    uint32_t k0, k1;
    ppo_perm_keys(seed, (uint64_t)ctr[0], k0, k1);
    out[t] = ppo_perm_at(i, n, hb, k0, k1);
}
__global__ void ppo_permutation_advance_kernel(uint32_t* ctr, long long n, long long window_len) {
    const uint32_t w = ctr[1] + 1u;
    if ((long long)w * window_len >= n) { ctr[1] = 0u; ctr[0] += 1u; } else ctr[1] = w;
}

static int perm_half_bits(long long n) {
    int hb = 1;
    while (hb < 31 && (1ull << (2 * hb)) < (unsigned long long)n) ++hb;
    return hb;
}

cudaError_t ppok_permutation(long long* out, long long n, uint64_t seed, uint64_t epoch, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    uint32_t k0, k1;
    ppo_perm_keys(seed, epoch, k0, k1);
    ppo_permutation_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(out, n, perm_half_bits(n), k0, k1, PpokPop{});
    return cudaGetLastError();
}

cudaError_t ppok_pop_permutation(const PpokPop& pop, long long* out, long long n, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const dim3 grid((unsigned)((n + 255) / 256), pop.members);
    ppo_permutation_kernel<true><<<grid, 256, 0, st>>>(out, n, perm_half_bits(n), 0u, 0u, pop);
    return cudaGetLastError();
}

cudaError_t ppok_permutation_window(long long* out, long long n, uint64_t seed, uint32_t* ctr, long long window_len, cudaStream_t st) {
    if (n <= 0 || window_len <= 0) return cudaSuccess;
    ppo_permutation_window_kernel<<<(unsigned)((window_len + 255) / 256), 256, 0, st>>>(out, n, perm_half_bits(n), seed, ctr, window_len);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ppo_permutation_advance_kernel<<<1, 1, 0, st>>>(ctr, n, window_len);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ K5: GAE, one thread per env, coalesced over envs
// POP: gamma and lambda of member i / pop.rows (n = every column of the population)
template <bool POP = false>
__global__ void __launch_bounds__(256)
ppo_gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values, const float* __restrict__ dones,
               const float* __restrict__ last_values, int T, int n, float gamma, float lam,
               float* __restrict__ adv, float* __restrict__ ret, const float* __restrict__ pop_hp = nullptr, int pop_rows = 0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if constexpr (POP) {
        const float* h = pop_hp + (size_t)(i / pop_rows) * PPO_POP_HP;
        gamma = h[PPO_POP_GAMMA]; lam = h[PPO_POP_GAE_LAMBDA];
    }
    float next_value = last_values[i], gae = 0.0f;
    for (int t = T - 1; t >= 0; --t) {
        const size_t o = (size_t)t * n + i;
        const float nnt = 1.0f - dones[o];
        const float v = values[o];
        const float delta = rewards[o] + gamma * next_value * nnt - v;
        gae = delta + gamma * lam * nnt * gae;
        adv[o] = gae;
        ret[o] = gae + v;
        next_value = v;
    }
}

cudaError_t ppok_gae(const float* rewards, const float* values, const float* dones, const float* last_values, int T, int n,
                     float gamma, float lam, float* adv, float* ret, cudaStream_t st) {
    ppo_gae_kernel<<<(n + 255) / 256, 256, 0, st>>>(rewards, values, dones, last_values, T, n, gamma, lam, adv, ret);
    return cudaGetLastError();
}

cudaError_t ppok_pop_gae(const PpokPop& pop, const float* rewards, const float* values, const float* dones, const float* last_values,
                         int T, int n, float* adv, float* ret, cudaStream_t st) {
    const int cols = n * pop.members;
    ppo_gae_kernel<true><<<(cols + 255) / 256, 256, 0, st>>>(rewards, values, dones, last_values, T, cols, 0.0f, 0.0f, adv, ret,
                                                            pop.hp, n);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ device-side step counter (CUDA-graph replay)
__global__ void ppo_counter_add_kernel(uint32_t* ctr, uint32_t inc) { if (threadIdx.x == 0 && blockIdx.x == 0) ctr[0] += inc; }

cudaError_t ppok_counter_add(uint32_t* ctr, uint32_t inc, cudaStream_t st) {
    ppo_counter_add_kernel<<<1, 32, 0, st>>>(ctr, inc);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ evaluation ledger (evaluate_policy's bookkeeping)
// One thread per env.  The return is summed in double in step order, as the host loop of PPO.evaluate_policy does
// (ret += rew.double()), so recorded returns are bit-identical to it.  The table slot of an episode is fixed by its env and
// episode number; the only atomic is the count of envs still below quota, which the host polls once per chunk of steps.
__global__ void __launch_bounds__(256)
ppo_eval_ledger_kernel(const float* __restrict__ rew, const uint8_t* __restrict__ flags, const uint8_t* __restrict__ tidx, int n,
                       double* __restrict__ ret, int* __restrict__ len, int* __restrict__ count, const int* __restrict__ quota,
                       const int* __restrict__ offset, uint32_t step, const uint32_t* __restrict__ step_dev, int step_limit,
                       int* __restrict__ remaining, double* __restrict__ ep_ret, int* __restrict__ ep_len,
                       uint8_t* __restrict__ ep_tr, uint8_t* __restrict__ ep_flags, int* __restrict__ ep_step) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = step + step_dev[0];
    if (s >= (uint32_t)step_limit) return;
    double r = ret[i] + (double)rew[i];
    int l = len[i] + 1;
    const uint8_t f = flags[i];
    if (f & 3u) {
        const int c = count[i], q = quota[i];
        if (c < q) {
            const size_t slot = (size_t)offset[i] + (size_t)c;
            ep_ret[slot] = r;
            ep_len[slot] = l;
            ep_tr[slot] = tidx != nullptr ? tidx[i] : (uint8_t)0;
            ep_flags[slot] = f;
            ep_step[slot] = (int)s;
            count[i] = c + 1;
            if (c + 1 == q) atomicSub(remaining, 1);
        }
        r = 0.0;
        l = 0;
    }
    ret[i] = r;
    len[i] = l;
}

cudaError_t ppok_eval_ledger(const float* rew, const uint8_t* flags, const uint8_t* tidx, int n, double* ret, int* len, int* count,
                             const int* quota, const int* offset, uint32_t step, const uint32_t* step_dev, int step_limit,
                             int* remaining, double* ep_ret, int* ep_len, uint8_t* ep_tr, uint8_t* ep_flags, int* ep_step,
                             cudaStream_t st) {
    ppo_eval_ledger_kernel<<<(n + 255) / 256, 256, 0, st>>>(rew, flags, tidx, n, ret, len, count, quota, offset, step, step_dev,
                                                            step_limit, remaining, ep_ret, ep_len, ep_tr, ep_flags, ep_step);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ training episode ledger (population episode statistics)
// One thread per env, one launch per rollout step, on the raw rewards and flags of the step.  Each env keeps its running return
// (double, summed in step order) and length, and adds every finished episode to its own sums acc[k * n + i] for the eight
// quantities of fw_episode_stats: episodes, return, length, targets reached, collisions, out-of-bounds, completed, strikes.  No
// atomics: a member's statistics are reduced afterwards over its envs in env order.
__global__ void __launch_bounds__(256)
ppo_pop_episode_ledger_kernel(const float* __restrict__ rew, const uint8_t* __restrict__ flags, const uint8_t* __restrict__ tidx,
                              int n, double* __restrict__ ret, int* __restrict__ len, double* __restrict__ acc) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r = ret[i] + (double)rew[i];
    int l = len[i] + 1;
    const uint8_t f = flags[i];
    if (f & 3u) {
        const size_t s = (size_t)n;
        acc[i] += 1.0;
        acc[s + i] += r;
        acc[2 * s + i] += (double)l;
        if (tidx != nullptr) acc[3 * s + i] += (double)tidx[i];
        if (f & 4u) acc[4 * s + i] += 1.0;          // FLAG_COLLISION
        if (f & 8u) acc[5 * s + i] += 1.0;          // FLAG_OOB
        if (f & 16u) acc[6 * s + i] += 1.0;         // FLAG_COMPLETE
        if (f & 32u) acc[7 * s + i] += 1.0;         // FLAG_STRIKE
        r = 0.0;
        l = 0;
    }
    ret[i] = r;
    len[i] = l;
}

cudaError_t ppok_pop_episode_ledger(const float* rew, const uint8_t* flags, const uint8_t* tidx, int n, double* ret, int* len,
                                    double* acc, cudaStream_t st) {
    ppo_pop_episode_ledger_kernel<<<(n + 255) / 256, 256, 0, st>>>(rew, flags, tidx, n, ret, len, acc);
    return cudaGetLastError();
}
