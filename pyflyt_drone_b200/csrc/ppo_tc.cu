// ppo_tc.cu -- K4 on the 5th-generation tensor cores: the policy/value MLP forward over the whole env batch.
//
// One persistent CTA per SM walks 128-row tiles (128 envs).  Per tile and tower:
//   X[128x32] (tf32, K-major canonical smem layout) x W1^T[32x64]  -> tcgen05.mma kind::tf32, accumulator in TMEM
//   epilogue: tcgen05.ld (each thread owns one row = one env), + bias, tanh, write H1 back to smem as the next A
//   H1[128x64] x W2^T[64x64] -> TMEM -> tcgen05.ld, + bias, tanh, 4-wide / 1-wide heads on CUDA cores
// Both towers' GEMMs of a layer are issued back to back by one elected thread and complete on one mbarrier
// (tcgen05.commit); their accumulators live side by side in 128 TMEM columns.  Weights stay resident in
// shared memory for the CTA's lifetime.  Replaces stable_baselines3 ActorCriticPolicy.forward as called from
// collect_rollouts (reference wiring: train/train_Fixedwing_Waypoints_v3.py:293-310).
//
// TF32 inputs (10-bit mantissa), fp32 accumulate: the rollout log-probabilities differ from the fp32 update
// path by ~1e-3 absolute, far inside PPO's clip range; tests/test_ppo_gpu.py states the tolerance.
#include "ppo_kernels.h"

#include <cuda_runtime.h>

// The file is compiled once per supported (action width, observation slab): ppo_tc_a6.cu includes it with PPO_A_BUILD = 6,
// ppo_tc_d64.cu with PPO_D_BUILD = 64 (observations of 33..64 floats: two 32-column slabs per row); everything lives in a
// namespace named after the build.
#ifndef PPO_A_BUILD
#define PPO_A_BUILD 4
#endif
#ifndef PPO_D_BUILD
#define PPO_D_BUILD 32
#endif
#if PPO_A_BUILD == 4 && PPO_D_BUILD == 32
namespace ppo_a4 {
#elif PPO_A_BUILD == 6 && PPO_D_BUILD == 32
namespace ppo_a6 {
#elif PPO_A_BUILD == 4 && PPO_D_BUILD == 64
namespace ppo_a4d64 {
#else
#error "supported builds: action width 4 or 6 with a 32-wide observation slab, action width 4 with a 64-wide one"
#endif

#define H PPO_H
#define A PPO_A_BUILD
#define AP ((A + 3) / 4 * 4)      // action width padded to whole float4s: the head weights are read as float4 rows
#define DP PPO_D_BUILD
#define NSLAB (DP / 32)
#define TC_ROWS 128
#define TC_THREADS 512
#define TC_TMEM_COLS 128

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// K-major, no-swizzle UMMA canonical layout of an [R x K] fp32 matrix: 8-row x 16-byte core matrices,
// core matrices of one 8-row group contiguous along K (LBO = 128 B), groups K*32 B apart (SBO).
__device__ __forceinline__ uint32_t tc_off(int r, int c, int K) {
    return (uint32_t)((r >> 3) * (K * 32) + (c >> 2) * 128 + (r & 7) * 16 + (c & 3) * 4);
}

__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;        // descriptor version 1 (Blackwell); layout_type 0 = no swizzle
    return d;
}

// instruction descriptor: D = F32, A = B = TF32, both K-major, N = 64, M = 128
#define TC_IDESC ((1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(H >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24))

#define TC_IDESC128 ((1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(2 * H >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24))

__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}

// D[128 x 64] (TMEM) = A[128 x K] (smem) * B[64 x K]^T (smem), K in steps of 8 (32 bytes of tf32 per instruction)
__device__ __forceinline__ void tc_gemm(uint32_t tmem_d, uint32_t a_base, uint32_t b_base, int K, uint32_t idesc = TC_IDESC) {
    uint64_t da = tc_desc(a_base, 128, K * 32), db = tc_desc(b_base, 128, K * 32);
#pragma unroll 1
    for (int k8 = 0; k8 < K / 8; ++k8) {
        tc_mma(tmem_d, da, db, idesc, k8 > 0 ? 1u : 0u);
        da += 16; db += 16;            // 256 bytes further along K: only the start-address field changes
    }
}

__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}

// Wait for the mbarrier phase.  try_wait suspends in hardware for a bounded time; the iteration cap turns a
// malformed-descriptor hang into a trap (an error the host sees) instead of a wedged GPU.
__device__ __forceinline__ void tc_wait(uint32_t bar, uint32_t parity) {
    for (uint32_t it = 0;; ++it) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
        if (it > (1u << 22)) __trap();
    }
}

__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t* u = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32"
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
          "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
          "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
          "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// MUFU.TANH (max relative error 2^-11, the order of the TF32 operand rounding); ppo_update_tc.cu uses the same
// instruction so that the update's log-probabilities reproduce the rollout's.
__device__ __forceinline__ float tc_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ uint4 tc_philox(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
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
__device__ __forceinline__ float tc_u01(uint32_t x) { return ((float)(x >> 9) + 0.5f) * (1.0f / 8388608.0f); }

// shared-memory plan (bytes); every MMA operand is 128-byte aligned
struct TcSmem {
    static constexpr int AX = 0;                          // X      [128 x 32]  16 KB
    static constexpr int AH_PI = AX + TC_ROWS * DP * 4;   // H1 pi  [128 x 64]  32 KB
    static constexpr int AH_VF = AH_PI + TC_ROWS * H * 4; // H1 vf  [128 x 64]  32 KB
    static constexpr int W1_PI = AH_VF + TC_ROWS * H * 4; // W1 pi  [64 x 32]    8 KB
    static constexpr int W1_VF = W1_PI + H * DP * 4;
    static constexpr int W2_PI = W1_VF + H * DP * 4;      // W2 pi  [64 x 64]   16 KB
    static constexpr int W2_VF = W2_PI + H * H * 4;
    static constexpr int SMALL = W2_VF + H * H * 4;       // biases, heads, stats, barrier, tmem pointer
    // floats inside SMALL
    static constexpr int B1_PI = 0, B1_VF = 64, B2_PI = 128, B2_VF = 192, W3_PI = 256 /* [64][AP] */, W3_VF = W3_PI + H * AP,
                         B3_PI = W3_VF + H, B3_VF = B3_PI + 8, LOGSTD = B3_VF + 4, MEAN = LOGSTD + 8, ISTD = MEAN + DP,
                         BAR = ISTD + DP /* 8-byte aligned */, TPTR = BAR + 4, NSMALL = TPTR + 4;
    static_assert((BAR % 2) == 0 && (NSMALL % 4) == 0 && (W3_PI % 4) == 0 && (W3_VF % 4) == 0, "alignment of the small area");
    static constexpr int HP = SMALL + NSMALL * 4;          // head partial sums [4 warpgroups][128 rows][AP] floats
    static constexpr int TOTAL = HP + 4 * TC_ROWS * AP * 4;
};

// every load of the thread (H * K / 512 = 4 or 8) is issued before its first store: the staging is latency-bound
template <int K>
__device__ __forceinline__ void tc_load_weight(char* smem, int off, const float* __restrict__ g, int d) {
    constexpr int N = H * K / TC_THREADS;
    float v[N];
#pragma unroll
    for (int n = 0; n < N; ++n) {
        const int i = threadIdx.x + n * TC_THREADS, j = i / K, k = i % K;
        v[n] = k < d ? g[j * d + k] : 0.0f;
    }
#pragma unroll
    for (int n = 0; n < N; ++n) {
        const int i = threadIdx.x + n * TC_THREADS, j = i / K, k = i % K;
        *reinterpret_cast<float*>(smem + off + tc_off(j, k, K)) = v[n];
    }
}

// load + normalise (VecNormalize.normalize_obs) 8 consecutive columns [8*part, 8*part+8) of observation row `grow_g`;
// optionally store the normalised values (what the rollout buffer keeps).  Rows of a tile are contiguous in memory,
// so the four threads of a row and the eight rows of a warp read one 896-byte span.
__device__ __forceinline__ void tc_load8(const float* __restrict__ obs_raw, float* __restrict__ obs_norm, int d, int grow_g,
                                         bool live, int part, bool have_stats, const float* s_mean, const float* s_istd,
                                         float clip, float (&x)[8]) {
    float raw[8];
    const bool vec = (d & 3) == 0;
    if (vec) {
        const float4* src = reinterpret_cast<const float4*>(obs_raw + (size_t)grow_g * d);
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        if (live && 8 * part < d) a = src[2 * part];
        if (live && 8 * part + 4 < d) b = src[2 * part + 1];
        raw[0] = a.x; raw[1] = a.y; raw[2] = a.z; raw[3] = a.w; raw[4] = b.x; raw[5] = b.y; raw[6] = b.z; raw[7] = b.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) { const int k = 8 * part + i; raw[i] = (live && k < d) ? obs_raw[(size_t)grow_g * d + k] : 0.0f; }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int k = 8 * part + i;
        float v = raw[i];
        if (have_stats) v = fminf(fmaxf((v - s_mean[k]) * s_istd[k], -clip), clip);
        x[i] = (live && k < d) ? v : 0.0f;
    }
    if (obs_norm != nullptr && live) {
        if (vec) {
            float4* dst = reinterpret_cast<float4*>(obs_norm + (size_t)grow_g * d);
            if (8 * part < d) dst[2 * part] = make_float4(x[0], x[1], x[2], x[3]);
            if (8 * part + 4 < d) dst[2 * part + 1] = make_float4(x[4], x[5], x[6], x[7]);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) { const int k = 8 * part + i; if (k < d) obs_norm[(size_t)grow_g * d + k] = x[i]; }
        }
    }
}

// 512 threads = 4 warpgroups: TMEM lane (= env row of the tile) = tid & 127; warpgroup q = tid >> 7 owns hidden units
// [32q, 32q+32) of the stacked pi|vf layers in both epilogues (q 0,1 = policy tower, 2,3 = value tower).
// POP: population launch, grid (CTAs per member, members): blockIdx.y = member, whose weights, statistics, seed and rows the
// CTA takes before it walks that member's tiles only (a member's tail tile is masked at its own n, as in a standalone launch)
template <bool POP = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
ppo_forward_tc_kernel(const float* __restrict__ params, int d, const float* __restrict__ obs_raw,
                      const double* __restrict__ stats, float clip, int n, uint32_t seed_lo, uint32_t seed_hi,
                      uint32_t env_id0, uint32_t step, const uint32_t* __restrict__ step_dev, int deterministic,
                      float* __restrict__ obs_norm, float* __restrict__ act_env, float* __restrict__ act_raw,
                      float* __restrict__ logp, float* __restrict__ value, PpokPop pop) {
    extern __shared__ __align__(1024) char smem[];
    if constexpr (POP) {
        const int m = blockIdx.y;
        const size_t r0 = (size_t)m * n;
        params += (size_t)m * pop.param_stride;
        obs_raw += r0 * d;
        if (stats != nullptr) stats += (size_t)m * (2 * d + 1);
        const uint64_t seed = pop.seeds[m];
        seed_lo = (uint32_t)(seed & 0xffffffffu); seed_hi = (uint32_t)(seed >> 32);
        env_id0 += (uint32_t)r0;
        if (obs_norm != nullptr) obs_norm += r0 * d;
        act_env += r0 * A;
        if (act_raw != nullptr) act_raw += r0 * A;
        if (logp != nullptr) logp += r0;
        value += r0;
    }
    float* small = reinterpret_cast<float*>(smem + TcSmem::SMALL);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int q = tid >> 7, lrow = tid & (TC_ROWS - 1);
    const int grow = tid >> 2, gpart = tid & 3;
    const int pi_count = H * d + H + H * H + H + A * H + A;
    const float* g_pi = params;
    const float* g_vf = params + pi_count;
    const int vf_count = H * d + H + H * H + H + H + 1;

    // ---- one-time: weights into the canonical operand layout, small vectors, barrier, TMEM
    tc_load_weight<DP>(smem, TcSmem::W1_PI, g_pi, d);
    tc_load_weight<DP>(smem, TcSmem::W1_VF, g_vf, d);
    tc_load_weight<H>(smem, TcSmem::W2_PI, g_pi + H * d + H, H);
    tc_load_weight<H>(smem, TcSmem::W2_VF, g_vf + H * d + H, H);
    if (tid < H) {
        small[TcSmem::B1_PI + tid] = g_pi[H * d + tid];
        small[TcSmem::B1_VF + tid] = g_vf[H * d + tid];
        small[TcSmem::B2_PI + tid] = g_pi[H * d + H + H * H + tid];
        small[TcSmem::B2_VF + tid] = g_vf[H * d + H + H * H + tid];
        small[TcSmem::W3_VF + tid] = g_vf[H * d + H + H * H + H + tid];
    }
    for (int i = tid; i < H * AP; i += blockDim.x) {                               // [j][a], zero padded to AP
        const int j = i / AP, a = i % AP;
        small[TcSmem::W3_PI + i] = a < A ? g_pi[H * d + H + H * H + H + a * H + j] : 0.0f;
    }
    if (tid < A) {
        small[TcSmem::B3_PI + tid] = g_pi[H * d + H + H * H + H + A * H + tid];
        small[TcSmem::LOGSTD + tid] = params[pi_count + vf_count + tid];
    }
    if (tid == 0) small[TcSmem::B3_VF] = g_vf[H * d + H + H * H + H + H];
    if (tid < DP) {
        if (stats != nullptr && tid < d) {
            small[TcSmem::MEAN + tid] = (float)stats[tid];
            small[TcSmem::ISTD + tid] = (float)(1.0 / sqrt(stats[d + tid] + 1e-8));
        } else { small[TcSmem::MEAN + tid] = 0.0f; small[TcSmem::ISTD + tid] = 1.0f; }
    }
    const uint32_t bar = tc_smem_u32(&small[TcSmem::BAR]);
    uint32_t* tptr = reinterpret_cast<uint32_t*>(&small[TcSmem::TPTR]);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(tc_smem_u32(tptr)), "r"((uint32_t)TC_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tptr;
    const uint32_t t_pi = tmem, t_vf = tmem + H;                       // column offsets 0 and 64
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;      // a warp may touch TMEM lanes 32*(warp%4)..+31
    const uint32_t s_base = tc_smem_u32(smem);
    const uint32_t step_eff = step + (step_dev != nullptr ? step_dev[0] : 0u);
    const bool have_stats = stats != nullptr;
    uint32_t phase = 0;
    // this warpgroup's slice: tower, first hidden unit inside the tower, TMEM columns, H1 buffer, parameter vectors
    const bool is_pi = q < 2;
    const int j0 = (q & 1) * 32;
    const uint32_t tcol = (is_pi ? t_pi : t_vf) + j0;
    const int ah = is_pi ? TcSmem::AH_PI : TcSmem::AH_VF;
    const float* b1 = small + (is_pi ? TcSmem::B1_PI : TcSmem::B1_VF) + j0;
    const float* b2 = small + (is_pi ? TcSmem::B2_PI : TcSmem::B2_VF) + j0;

    const int ntiles = (n + TC_ROWS - 1) / TC_ROWS;
    float xcur[NSLAB][8];
    if ((int)blockIdx.x < ntiles) {
        const int gr = blockIdx.x * TC_ROWS + grow;
#pragma unroll
        for (int sl = 0; sl < NSLAB; ++sl)
            tc_load8(obs_raw, obs_norm, d, gr, gr < n, gpart + 4 * sl, have_stats, small + TcSmem::MEAN, small + TcSmem::ISTD, clip,
                     xcur[sl]);
    }
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // ---- stage the normalised observation slice as the A operand of layer 1
#pragma unroll
        for (int sl = 0; sl < NSLAB; ++sl) {
            const int k = 8 * (gpart + 4 * sl);
            *reinterpret_cast<float4*>(smem + TcSmem::AX + tc_off(grow, k, DP)) = make_float4(xcur[sl][0], xcur[sl][1], xcur[sl][2], xcur[sl][3]);
            *reinterpret_cast<float4*>(smem + TcSmem::AX + tc_off(grow, k + 4, DP)) = make_float4(xcur[sl][4], xcur[sl][5], xcur[sl][6], xcur[sl][7]);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> tensor-core reads
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tc_gemm(t_pi, s_base + TcSmem::AX, s_base + TcSmem::W1_PI, DP, TC_IDESC128);   // W1_pi|W1_vf: one N = 128 B operand
            tc_commit(bar);
        }
        // the next tile's observations are requested now and land while this tile is processed
        {
            const int nt = tile + gridDim.x;
            const int gr = nt * TC_ROWS + grow;
#pragma unroll
            for (int sl = 0; sl < NSLAB; ++sl)
                tc_load8(obs_raw, obs_norm, d, gr, nt < ntiles && gr < n, gpart + 4 * sl, have_stats, small + TcSmem::MEAN,
                         small + TcSmem::ISTD, clip, xcur[sl]);
        }
        tc_wait(bar, phase); phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- layer-1 epilogue: bias + tanh, H1 becomes the A operand of layer 2 (this thread's row, 32 hidden units)
        {
            float v[32];
            tc_ld32(tcol + lane_base, v);
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4) {
                const float4 b = *reinterpret_cast<const float4*>(b1 + 4 * c4);
                float4 o = make_float4(tc_tanh(v[4 * c4 + 0] + b.x), tc_tanh(v[4 * c4 + 1] + b.y),
                                       tc_tanh(v[4 * c4 + 2] + b.z), tc_tanh(v[4 * c4 + 3] + b.w));
                *reinterpret_cast<float4*>(smem + ah + tc_off(lrow, j0 + 4 * c4, H)) = o;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tc_gemm(t_pi, s_base + TcSmem::AH_PI, s_base + TcSmem::W2_PI, H);
            tc_gemm(t_vf, s_base + TcSmem::AH_VF, s_base + TcSmem::W2_VF, H);
            tc_commit(bar);
        }
        // Gaussian noise for this row (warpgroup 0), drawn while the layer-2 MMAs run
        const int row = tile * TC_ROWS + lrow;
        const bool live = row < n;
        float eps[A];
#pragma unroll
        for (int a = 0; a < A; ++a) eps[a] = 0.0f;
        if (q == 0 && live && !deterministic) {
#pragma unroll
            for (int g = 0; g < AP / 4; ++g) {          // four normals per Philox call; channels 4.. use counter word 2 = 1
                uint4 r = tc_philox(seed_lo, seed_hi, env_id0 + (uint32_t)row, step_eff, (uint32_t)g, 7u);
                float ra = sqrtf(-2.0f * __logf(tc_u01(r.x))), rb = sqrtf(-2.0f * __logf(tc_u01(r.z)));
                float s0, c0, s1, c1;
                sincospif(2.0f * tc_u01(r.y), &s0, &c0);
                sincospif(2.0f * tc_u01(r.w), &s1, &c1);
                const float e4[4] = {ra * c0, ra * s0, rb * c1, rb * s1};
#pragma unroll
                for (int k = 0; k < 4; ++k) if (4 * g + k < A) eps[4 * g + k] = e4[k];
            }
        }
        tc_wait(bar, phase); phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- layer-2 epilogue: partial head sums over this warpgroup's 32 hidden units
        {
            float v[32];
            tc_ld32(tcol + lane_base, v);
            float ps[AP];
#pragma unroll
            for (int a = 0; a < AP; ++a) ps[a] = 0.0f;
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4) {
                const float4 b = *reinterpret_cast<const float4*>(b2 + 4 * c4);
                const float h2[4] = {tc_tanh(v[4 * c4 + 0] + b.x), tc_tanh(v[4 * c4 + 1] + b.y), tc_tanh(v[4 * c4 + 2] + b.z),
                                     tc_tanh(v[4 * c4 + 3] + b.w)};
                if (is_pi) {
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
#pragma unroll
                        for (int g = 0; g < AP / 4; ++g) {
                            const float4 w = *reinterpret_cast<const float4*>(small + TcSmem::W3_PI + (j0 + 4 * c4 + r) * AP + 4 * g);
                            ps[4 * g + 0] = fmaf(w.x, h2[r], ps[4 * g + 0]); ps[4 * g + 1] = fmaf(w.y, h2[r], ps[4 * g + 1]);
                            ps[4 * g + 2] = fmaf(w.z, h2[r], ps[4 * g + 2]); ps[4 * g + 3] = fmaf(w.w, h2[r], ps[4 * g + 3]);
                        }
                    }
                } else {
                    const float4 w = *reinterpret_cast<const float4*>(small + TcSmem::W3_VF + j0 + 4 * c4);
                    ps[0] = fmaf(w.x, h2[0], ps[0]); ps[0] = fmaf(w.y, h2[1], ps[0]);
                    ps[0] = fmaf(w.z, h2[2], ps[0]); ps[0] = fmaf(w.w, h2[3], ps[0]);
                }
            }
#pragma unroll
            for (int g = 0; g < AP / 4; ++g)
                *reinterpret_cast<float4*>(smem + TcSmem::HP + ((q * TC_ROWS + lrow) * AP + 4 * g) * 4) =
                    make_float4(ps[4 * g + 0], ps[4 * g + 1], ps[4 * g + 2], ps[4 * g + 3]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ---- heads, diagonal-Gaussian sample and log-probability: one thread per env
        if (q == 0 && live) {
            const float* hp0 = reinterpret_cast<const float*>(smem + TcSmem::HP) + (0 * TC_ROWS + lrow) * AP;
            const float* hp1 = reinterpret_cast<const float*>(smem + TcSmem::HP) + (1 * TC_ROWS + lrow) * AP;
            const float pv0 = *(reinterpret_cast<const float*>(smem + TcSmem::HP) + (2 * TC_ROWS + lrow) * AP);
            const float pv1 = *(reinterpret_cast<const float*>(smem + TcSmem::HP) + (3 * TC_ROWS + lrow) * AP);
            value[row] = small[TcSmem::B3_VF] + pv0 + pv1;
            float lp = 0.0f, av[A], ac[A];
#pragma unroll
            for (int a = 0; a < A; ++a) {
                const float mean = small[TcSmem::B3_PI + a] + hp0[a] + hp1[a];
                const float ls = small[TcSmem::LOGSTD + a];
                av[a] = fmaf(__expf(ls), eps[a], mean);
                ac[a] = fminf(fmaxf(av[a], -1.f), 1.f);
                lp += -0.5f * eps[a] * eps[a] - ls - 0.91893853320467274178f;
            }
#pragma unroll
            for (int a = 0; a < A; a += 2) {             // rows are A floats wide (8-byte aligned for the even widths)
                reinterpret_cast<float2*>(act_env + (size_t)row * A)[a / 2] = make_float2(ac[a], ac[a + 1]);
                if (act_raw != nullptr) reinterpret_cast<float2*>(act_raw + (size_t)row * A)[a / 2] = make_float2(av[a], av[a + 1]);
            }
            if (logp != nullptr) logp[row] = lp;
        }
        // no trailing barrier: the partials live outside the operand buffers, and the two block-wide syncs of the next
        // tile separate these reads from the next writes
    }
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"((uint32_t)TC_TMEM_COLS) : "memory");
}

static int g_tc_sm_count = 0;
static cudaError_t tc_setup() {
    if (g_tc_sm_count != 0) return cudaSuccess;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ppo_forward_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ppo_forward_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem::TOTAL);
    if (e != cudaSuccess) return e;
    g_tc_sm_count = sms;
    return cudaSuccess;
}

cudaError_t ppok_forward_tc(const float* params, int d, const float* obs_raw, const double* stats, float clip, int n,
                            uint64_t seed, uint32_t env_id0, uint32_t step, const uint32_t* step_dev, int deterministic,
                            float* obs_norm, float* act_env, float* act_raw, float* logp, float* value, cudaStream_t st) {
    if (d > DP) return cudaErrorInvalidValue;
    cudaError_t e = tc_setup();
    if (e != cudaSuccess) return e;
    const int sm_count = g_tc_sm_count;
    const int ntiles = (n + TC_ROWS - 1) / TC_ROWS;
    const int grid = ntiles < sm_count ? ntiles : sm_count;          // persistent: one CTA per SM walks the tiles
    ppo_forward_tc_kernel<<<grid, TC_THREADS, TcSmem::TOTAL, st>>>(params, d, obs_raw, stats, clip, n, (uint32_t)(seed & 0xffffffffu),
                                                               (uint32_t)(seed >> 32), env_id0, step, step_dev, deterministic,
                                                               obs_norm, act_env, act_raw, logp, value, PpokPop{});
    return cudaGetLastError();
}

// n = rows per member.  Each member gets an equal share of the SMs (at least one CTA, at most one per tile); a CTA walks
// only its member's tiles, so it stages one member's weights once, and every row sees the arithmetic of a standalone launch.
cudaError_t ppok_pop_forward_tc(const PpokPop& pop, const float* params, int d, const float* obs_raw, const double* stats, float clip,
                                int n, uint32_t env_id0, uint32_t step, const uint32_t* step_dev, int deterministic, float* obs_norm,
                                float* act_env, float* act_raw, float* logp, float* value, cudaStream_t st) {
    if (d > DP) return cudaErrorInvalidValue;
    cudaError_t e = tc_setup();
    if (e != cudaSuccess) return e;
    const int ntiles = (n + TC_ROWS - 1) / TC_ROWS;
    int per = g_tc_sm_count / pop.members;
    if (per < 1) per = 1;
    if (per > ntiles) per = ntiles;
    ppo_forward_tc_kernel<true><<<dim3(per, pop.members), TC_THREADS, TcSmem::TOTAL, st>>>(
        params, d, obs_raw, stats, clip, n, 0u, 0u, env_id0, step, step_dev, deterministic, obs_norm, act_env, act_raw, logp, value, pop);
    return cudaGetLastError();
}

}  // namespace ppo_a4 / ppo_a6 / ppo_a4d64
