// ppo_tower.cuh -- the CUDA-core MlpPolicy tower, one thread per row: shared by the PPO forward (ppo_kernels.cu, K4) and by
// the high-level waypoint step (fw_kernels.cu, task 5), which evaluates a frozen low-level tracker with it.  One copy of the
// arithmetic is what makes the tracker's action inside the step bit-identical to PPO.predict(obs, deterministic=True).
#pragma once
#include "ppo_kernels.h"

// tanh(x) = 1 - 2/(exp(2x)+1): relative error ~2e-7 with the SFU exp2/rcp, saturates cleanly at +-1
__device__ __forceinline__ float ppo_tanh(float x) {
    float e = __expf(2.0f * x);
    return 1.0f - __fdividef(2.0f, e + 1.0f);
}

// smem layout of one tower: W1[H][DP] b1[H] W2[H][H] b2[H] W3[OUT][H] b3[OUT]
template <int OUT, int DP>
struct TowerOff {
    static constexpr int W1 = 0, B1 = W1 + PPO_H * DP, W2 = B1 + PPO_H, B2 = W2 + PPO_H * PPO_H, W3 = B2 + PPO_H,
                         B3 = W3 + OUT * PPO_H, SIZE = ((B3 + OUT + 3) / 4) * 4;
};

// copy one tower from the packed global parameter vector ([out,in] rows of width d) into padded smem
template <int OUT, int DP>
__device__ void load_tower(float* s, const float* __restrict__ g, int d) {
    using O = TowerOff<OUT, DP>;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < PPO_H * DP; i += nt) { int j = i / DP, k = i % DP; s[O::W1 + i] = k < d ? g[j * d + k] : 0.0f; }
    const float* gb1 = g + PPO_H * d;
    for (int i = tid; i < PPO_H; i += nt) s[O::B1 + i] = gb1[i];
    const float* gw2 = gb1 + PPO_H;
    for (int i = tid; i < PPO_H * PPO_H; i += nt) s[O::W2 + i] = gw2[i];
    const float* gb2 = gw2 + PPO_H * PPO_H;
    for (int i = tid; i < PPO_H; i += nt) s[O::B2 + i] = gb2[i];
    const float* gw3 = gb2 + PPO_H;
    for (int i = tid; i < OUT * PPO_H; i += nt) s[O::W3 + i] = gw3[i];
    const float* gb3 = gw3 + OUT * PPO_H;
    for (int i = tid; i < OUT; i += nt) s[O::B3 + i] = gb3[i];
}

// One tower for the calling thread's row.  x: normalised observation in registers (DP wide, zero padded);
// hbuf: this block's [H][blockDim.x] activation scratch (column = thread, conflict-free).  out[OUT].
template <int OUT, int DP>
__device__ __forceinline__ void tower_forward(const float* __restrict__ s, const float (&x)[DP], float* hbuf, float (&out)[OUT]) {
    using O = TowerOff<OUT, DP>;
    const int tid = threadIdx.x, nt = blockDim.x;
    // layer 1: weights broadcast from smem (every thread reads the same address), inputs in registers
    for (int j = 0; j < PPO_H; ++j) {
        const float4* w = reinterpret_cast<const float4*>(s + O::W1 + j * DP);
        float acc = s[O::B1 + j];
#pragma unroll
        for (int k4 = 0; k4 < DP / 4; ++k4) {
            float4 ww = w[k4];
            acc = fmaf(ww.x, x[4 * k4 + 0], acc); acc = fmaf(ww.y, x[4 * k4 + 1], acc);
            acc = fmaf(ww.z, x[4 * k4 + 2], acc); acc = fmaf(ww.w, x[4 * k4 + 3], acc);
        }
        hbuf[j * nt + tid] = ppo_tanh(acc);
    }
    float h1[PPO_H];
#pragma unroll
    for (int k = 0; k < PPO_H; ++k) h1[k] = hbuf[k * nt + tid];
#pragma unroll
    for (int a = 0; a < OUT; ++a) out[a] = s[O::B3 + a];
    // layer 2 fused with the head: each hidden unit is consumed as soon as it is produced
    for (int j = 0; j < PPO_H; ++j) {
        const float4* w = reinterpret_cast<const float4*>(s + O::W2 + j * PPO_H);
        float acc0 = s[O::B2 + j], acc1 = 0.0f;
#pragma unroll
        for (int k4 = 0; k4 < PPO_H / 4; k4 += 2) {
            float4 wa = w[k4], wb = w[k4 + 1];
            acc0 = fmaf(wa.x, h1[4 * k4 + 0], acc0); acc0 = fmaf(wa.y, h1[4 * k4 + 1], acc0);
            acc0 = fmaf(wa.z, h1[4 * k4 + 2], acc0); acc0 = fmaf(wa.w, h1[4 * k4 + 3], acc0);
            acc1 = fmaf(wb.x, h1[4 * k4 + 4], acc1); acc1 = fmaf(wb.y, h1[4 * k4 + 5], acc1);
            acc1 = fmaf(wb.z, h1[4 * k4 + 6], acc1); acc1 = fmaf(wb.w, h1[4 * k4 + 7], acc1);
        }
        float h2 = ppo_tanh(acc0 + acc1);
#pragma unroll
        for (int a = 0; a < OUT; ++a) out[a] = fmaf(s[O::W3 + a * PPO_H + j], h2, out[a]);
    }
}

// normalise one observation row into registers (VecNormalize.normalize_obs) and optionally store it
template <int DP>
__device__ __forceinline__ void load_obs(const float* __restrict__ obs_raw, const float* s_mean, const float* s_istd,
                                         float clip, int d, int row, float (&x)[DP], float* __restrict__ obs_norm) {
#pragma unroll
    for (int k = 0; k < DP; ++k) {
        float v = 0.0f;
        if (k < d) {
            v = obs_raw[(size_t)row * d + k];
            if (s_mean != nullptr) v = fminf(fmaxf((v - s_mean[k]) * s_istd[k], -clip), clip);
            if (obs_norm != nullptr) obs_norm[(size_t)row * d + k] = v;
        }
        x[k] = v;
    }
}

template <int DP>
__device__ __forceinline__ void stage_stats(const double* __restrict__ stats, int d, float* s_mean, float* s_istd) {
    for (int k = threadIdx.x; k < DP; k += blockDim.x) {
        if (stats != nullptr && k < d) {
            s_mean[k] = (float)stats[k];
            s_istd[k] = (float)(1.0 / sqrt(stats[d + k] + 1e-8));     // VecNormalize epsilon
        } else { s_mean[k] = 0.0f; s_istd[k] = 1.0f; }
    }
}

// the action the env receives: the Gaussian sample (the mean, when deterministic) clipped to the action box
__device__ __forceinline__ float ppo_clip_action(float a) { return fminf(fmaxf(a, -1.f), 1.f); }
