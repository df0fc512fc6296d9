// ppo_update_tc.cu -- K6: the PPO minibatch gradient (forward + backward of both MLP towers and the clipped
// surrogate / value / entropy losses) fused into ONE kernel on the tcgen05 tensor cores, plus the partial-sum
// reduction and the clipped Adam step.  Replaces stable_baselines3 PPO.train()'s per-minibatch
// evaluate_actions -> loss -> backward -> clip_grad_norm_ -> Adam.step
// (reference wiring: /root/reference/train/train_Fixedwing_Waypoints_v3.py:293-337).
//
// Work decomposition: a persistent CTA (128 threads = 128 samples per tile, thread == sample == TMEM lane) walks
// tiles of the minibatch.  All matrix products are tcgen05.mma with fp32 accumulators in TMEM:
//   forward   X[128x32] W1^T, H1[128x64] W2^T        kind::tf32, A and B K-major (the log-probability ratio needs
//                                                     the forward pass to agree with the rollout to ~1e-3)
//   dgrad     dZ2[128x64] W2                          kind::f16 (bf16), B read MN-major from the forward-layout copy
//   wgrad     [dZ2_pi|dZ2_vf]^T H1, [dZ1_pi|dZ1_vf]^T X, [H2_pi|H2_vf]^T dOut, bias sums against a ones column
//             kind::f16 (bf16), A and B read MN-major: the activation rows each thread writes for its own sample ARE
//             the transposed operands the weight gradients need -- no transposes, no extra copies.
//             (Measured on B200: kind::tf32 returns zeros for MN-major operands in the no-swizzle layout, bf16
//             handles all four major combinations -- scripts/tc_probe.cu -- hence bf16 for the backward products;
//             tanh' is recomputed from the fp32 pre-activations kept in TMEM, not from rounded activations.)
// Both towers are stacked along M (= 128 output neurons) for the weight gradients, which accumulate in TMEM
// across all tiles of the CTA and are read out once at the end into a per-CTA partial gradient.
// The file is compiled once per supported action width (ppo_update_tc_a6.cu includes it with PPO_A_BUILD = 6: the
// six-channel MlpPolicy of train/train_lowlevel_cmd.py:97-110); the gradient kernel and its launcher live in a namespace
// named after the width, the width-independent kernels (advantage statistics, partial reduction, Adam) in the first build.
#include "ppo_kernels.h"

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#ifndef PPO_A_BUILD
#define PPO_A_BUILD 4
#endif
#ifndef PPO_D_BUILD
#define PPO_D_BUILD 32
#endif
#if PPO_A_BUILD == 4 && PPO_D_BUILD == 32
#define PPO_UT_NS ppo_a4
#define PPO_UT_SHARED 1          // this build also carries the width-independent kernels
#elif PPO_A_BUILD == 6 && PPO_D_BUILD == 32
#define PPO_UT_NS ppo_a6
#elif PPO_A_BUILD == 4 && PPO_D_BUILD == 64
#define PPO_UT_NS ppo_a4d64
#else
#error "supported builds: action width 4 or 6 with a 32-wide observation slab, action width 4 with a 64-wide one"
#endif

#define H PPO_H
#define A PPO_A_BUILD
#define AP ((A + 3) / 4 * 4)      // action width padded to whole float4s
#define DP PPO_D_BUILD           // observation columns staged per tile (layer-1 K)
// 64-wide build: layer 2 of the forward pass runs as a bf16 hi/lo split (three kind::f16 MMAs: hi*hi + lo*hi + hi*lo,
// ~2^-16 relative, tighter than TF32) so that the bf16 operands the backward pass needs anyway (H1 hi = wgrad B,
// W2 hi = dgrad B) double as forward operands; the 48 KB this frees pay for the wider X / W1 buffers.
#define UT_SPLIT (DP > 32)
#define UT_ROWS 128
#define UT_THREADS 512
#define UT_TMEM_COLS 512

// In-kernel gradient all-reduce over NVLink peer memory (world > 1; ppo_peer_*): used by the last block of the gradient
// reduction and by the single-CTA optimizer steps.
// Low-latency protocol: every gradient element travels as one 8-byte store {value, sequence number} into slot
// [parity][rank] of every peer's exchange buffer; the receiver polls the element itself until it carries this step's
// sequence number -- an aligned 8-byte store arrives whole, so no fence and no separate flag sit between data and signal.
// Each thread pushes and then collects its own elements; the slots are summed in rank order (the same bits on every rank).
// Parity double-buffers the slots: a rank can only be one step ahead of a peer (it needs the peer's data of step q-1 to get
// to step q), so the slot of step q-2 it overwrites has been consumed.
#define PEER_MAX_WORLD 8
#define PEER_STRIDE 16384                                   // elements per (parity, rank) slot: P <= 16384
#define PEER_BYTES ((size_t)2 * PEER_MAX_WORLD * PEER_STRIDE * 8)
__device__ __forceinline__ void peer_store(uint2* p, float v, unsigned q) {
    // a plain (weak) vector store: the 32 lanes' 8-byte pairs leave as whole 128-byte writes -- measured 20 us per 12 K-element
    // exchange from one SM with st.volatile (one NVLink packet per element), ~2 us coalesced; value and sequence number of
    // an element share one aligned 8-byte word of one sector, so they still arrive together
    asm volatile("st.global.v2.u32 [%0], {%1, %2};" :: "l"(p), "r"(__float_as_uint(v)), "r"(q) : "memory");
}
__device__ __forceinline__ uint2 peer_load(const uint2* p) {
    uint2 r;
    asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p) : "memory");
    return r;
}
// peer_push: this thread's N elements (k = first + i * stride) to every other rank.  peer_collect: the other ranks' copies of
// those elements, returned as rank-ordered sums in own[].  Every push of a step goes out before the first collect (a
// push / collect pair per chunk would pay the link latency once per chunk); the polls of one peer's N elements are all in
// flight before the first is examined, and an element that has not arrived yet is re-polled.
template <int N>
__device__ __forceinline__ void peer_push(const float (&own)[N], int P, int first, int stride, int W, int me, unsigned q,
                                          float* const* peer) {
    const size_t par_off = (size_t)(q & 1u) * PEER_MAX_WORLD * PEER_STRIDE;
    for (int j = 0; j < W; ++j) {
        if (j == me) continue;
        uint2* dst = reinterpret_cast<uint2*>(peer[j]) + par_off + (size_t)me * PEER_STRIDE;
#pragma unroll
        for (int i = 0; i < N; ++i) { const int k = first + i * stride; if (k < P) peer_store(dst + k, own[i], q); }
    }
}
template <int N>
__device__ __forceinline__ void peer_collect(float (&own)[N], int P, int first, int stride, int W, int me, unsigned q,
                                             float* const* peer) {
    const size_t par_off = (size_t)(q & 1u) * PEER_MAX_WORLD * PEER_STRIDE;
    const uint2* mine = reinterpret_cast<const uint2*>(peer[me]) + par_off;
    float sum[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sum[i] = 0.0f;
    for (int j = 0; j < W; ++j) {
        if (j == me) {
#pragma unroll
            for (int i = 0; i < N; ++i) sum[i] += own[i];
            continue;
        }
        const uint2* src = mine + (size_t)j * PEER_STRIDE;
        uint2 v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) { const int k = first + i * stride; v[i] = k < P ? peer_load(src + k) : make_uint2(0u, q); }
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const int k = first + i * stride;
            for (unsigned it = 0; v[i].y != q; ++it) {
                if (it > (1u << 22)) __trap();               // a missing peer becomes an error the host sees, not a hang
                __nanosleep(32);
                v[i] = peer_load(src + k);
            }
            sum[i] += __uint_as_float(v[i].x);
        }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) own[i] = sum[i];
}

namespace PPO_UT_NS {

__device__ __forceinline__ uint32_t ut_smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// K-major canonical (no swizzle) offset of element (r, c) in an [R x K] fp32 matrix; see ppo_tc.cu
__device__ __forceinline__ uint32_t ut_off(int r, int c, int K) {
    return (uint32_t)((r >> 3) * (K * 32) + (c >> 2) * 128 + (r & 7) * 16 + (c & 3) * 4);
}

// same canonical layout for bf16 (8 elements per 16-byte chunk)
__device__ __forceinline__ uint32_t ut_off16(int r, int c, int K) {
    return (uint32_t)((r >> 3) * (K * 16) + (c >> 3) * 128 + (r & 7) * 16 + (c & 7) * 2);
}
__device__ __forceinline__ uint32_t ut_pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint4 ut_pack8(const float* v) {
    return make_uint4(ut_pack2(v[0], v[1]), ut_pack2(v[2], v[3]), ut_pack2(v[4], v[5]), ut_pack2(v[6], v[7]));
}

__device__ __forceinline__ uint64_t ut_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// instruction descriptor: D = F32, M = 128; fmt 2 = TF32 (kind::tf32), 1 = BF16 (kind::f16); majors and N vary
__device__ __forceinline__ constexpr uint32_t ut_idesc(int fmt, int n, int a_mn, int b_mn) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(UT_ROWS >> 4) << 24);
}

template <bool BF16>
__device__ __forceinline__ void ut_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    if (BF16)
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
            :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
            :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}

// D[128 x N] (+)= A B^T over `ksteps` instructions (K = 8 tf32 / 16 bf16 each); per instruction the operand start
// addresses advance by a_step / b_step bytes (256 for a K-major operand; LBO resp. 2*LBO for an MN-major one).
// The descriptors are built once per GEMM; a k step only bumps the 14-bit start-address field (no carry: every
// operand lies below 256 KB).
template <bool BF16, int KSTEPS>
__device__ __forceinline__ void ut_gemm(uint32_t tmem_d, uint32_t a_addr, uint32_t a_lbo, uint32_t a_sbo, uint32_t a_step,
                                        uint32_t b_addr, uint32_t b_lbo, uint32_t b_sbo, uint32_t b_step,
                                        uint32_t idesc, uint32_t accumulate_first) {
    const uint64_t da = ut_desc(a_addr, a_lbo, a_sbo), db = ut_desc(b_addr, b_lbo, b_sbo);
    const uint64_t ia = a_step >> 4, ib = b_step >> 4;
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k)      // unrolled: the descriptors of all k steps are independent adds
        ut_mma<BF16>(tmem_d, da + k * ia, db + k * ib, idesc, k > 0 ? 1u : accumulate_first);
}

__device__ __forceinline__ void ut_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void ut_wait(uint32_t bar, uint32_t parity) {
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

__device__ __forceinline__ void ut_ld32(uint32_t taddr, float (&v)[32]) {
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

__device__ __forceinline__ void ut_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t* u = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32"
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
          "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// MUFU.TANH: one SFU instruction, max relative error 2^-11 -- the same order as the TF32 operand rounding of the
// forward GEMMs.  The rollout forward (ppo_tc.cu) uses the same instruction, so log-probability ratios are consistent.
__device__ __forceinline__ float ut_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

#define UT_FENCE_SYNC()                                                   \
    do {                                                                  \
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      \
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  \
        __syncthreads();                                                  \
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");   \
    } while (0)

// shared-memory plan (bytes): 222.5 KB of the 227 KB a CTA may own
struct UtSmem {
    static constexpr int XB = 0;                              // X  f32       [128 x 32]    16 KB  forward L1 A
    static constexpr int H1C = XB + UT_ROWS * DP * 4;         // H1 f32 pi|vf [128 x 128]   64 KB  forward L2 A
#if UT_SPLIT
    static constexpr int DZ2 = H1C + UT_ROWS * 2 * H * 2;     // dZ2 bf16     [128 x 128]   32 KB  aliases H1 lo (dead after M2)
#else
    static constexpr int DZ2 = H1C;                           // dZ2 bf16     [128 x 128]   32 KB  aliases H1C (dead after M2)
#endif
    static constexpr int H2B = H1C + UT_ROWS * 2 * H * 4;     // H2 bf16 pi|vf[128 x 128]   32 KB  wgrad L3 A
    static constexpr int DZ1 = H2B;                           // dZ1 bf16     [128 x 128]   32 KB  aliases H2B (dead after M3)
#if UT_SPLIT
    // split build: the 64 KB at H1C hold H1 hi (bf16, forward L2 A and wgrad L2 B) then H1 lo (forward only; dZ2 lands there)
    static constexpr int H1B = H1C;
    static constexpr int H1L = H1C + UT_ROWS * 2 * H * 2;
    static constexpr int XBB = H2B + UT_ROWS * 2 * H * 2;     // X  bf16      [128 x 64]    16 KB  wgrad L1 B
#else
    static constexpr int H1B = H2B + UT_ROWS * 2 * H * 2;     // H1 bf16 pi|vf[128 x 128]   32 KB  wgrad L2 B
    static constexpr int XBB = H1B + UT_ROWS * 2 * H * 2;     // X  bf16      [128 x 32]     8 KB  wgrad L1 B
#endif
    static constexpr int DO = XBB + UT_ROWS * DP * 2;         // dOut|1 bf16  [128 x 16]     4 KB
    static constexpr int W1_PI = DO + UT_ROWS * 16 * 2;       // W1 f32       [64 x 32]      8 KB each
    static constexpr int W1_VF = W1_PI + H * DP * 4;
#if UT_SPLIT
    static constexpr int W2B_PI = W1_VF + H * DP * 4;         // W2 hi bf16   [64 x 64]      8 KB each (forward B, dgrad B)
    static constexpr int W2B_VF = W2B_PI + H * H * 2;
    static constexpr int W2L_PI = W2B_VF + H * H * 2;         // W2 lo bf16   [64 x 64]      8 KB each (forward B)
    static constexpr int W2L_VF = W2L_PI + H * H * 2;
    static constexpr int SMALL = W2L_VF + H * H * 2;
#else
    static constexpr int W2_PI = W1_VF + H * DP * 4;          // W2 f32       [64 x 64]     16 KB each
    static constexpr int W2_VF = W2_PI + H * H * 4;
    static constexpr int W2B_PI = W2_VF + H * H * 4;          // W2 bf16      [64 x 64]      8 KB each (dgrad B)
    static constexpr int W2B_VF = W2B_PI + H * H * 2;
    static constexpr int SMALL = W2B_VF + H * H * 2;
#endif
    // floats inside SMALL
    static constexpr int B1 = 0 /* pi 64 | vf 64 */, B2 = 128, W3_PI = 256 /* [64][AP]: AP/4 float4s per hidden unit */,
                         W3_VF = W3_PI + H * AP, B3_PI = W3_VF + H, B3_VF = B3_PI + AP, LOGSTD = B3_VF + 4,
                         RED = LOGSTD + AP /* 24 block-reduction slots */, BAR = RED + 24, TPTR = BAR + 4,
                         FUSED = TPTR + 4 /* adv mean, adv std, clip coefficient, Adam step (as int) */, NSMALL = FUSED + 4;
    // the layer-1 operand buffer XB is dead after M1 and then carries, per tile: the policy-head partial sums of warpgroups
    // 0 and 1 (AP floats per row each), the value-head partials of warpgroups 2 and 3, and each row's loss inputs
    static constexpr int PS_PI = 0, PS_VF = PS_PI + 2 * UT_ROWS * AP * 4, LIN = PS_VF + 2 * UT_ROWS * 4, LIN_ROW = (AP + 4) * 4;
    static_assert(LIN + UT_ROWS * LIN_ROW <= UT_ROWS * DP * 4, "head partials + loss inputs must fit the layer-1 operand buffer");
    static constexpr int TOTAL = SMALL + NSMALL * 4;
    static_assert(2 * A + 7 <= 24, "block-reduction slots");
    static_assert(TOTAL <= 227 * 1024, "a CTA owns at most 227 KB of shared memory");
};

// TMEM column plan
#define UT_T1 0      // 128: layer-1 pre-activations (pi cols 0-63, vf 64-127), kept for tanh' in the backward pass
#define UT_T2 128    // 128: layer-2 pre-activations, later the data gradient dH1
#define UT_DA 256    // 64 : [dZ2]^T H1_pi   (rows 0-63 = dW2_pi)
#define UT_DB 320    // 64 : [dZ2]^T H1_vf   (rows 64-127 = dW2_vf)
#define UT_DW1 384   // DP : [dZ1]^T X       (rows 0-63 dW1_pi, 64-127 dW1_vf)
#define UT_D3 (UT_DW1 + DP)   // 16 : [H2]^T dOut     (rows 0-63 x cols 0..A-1 = dW3_pi^T ; rows 64-127 x col A = dW3_vf)
#define UT_DB2 (UT_D3 + 16)   // 16 : [dZ2]^T dOut|1  (col A+1 = db2)
#define UT_DB1 (UT_DB2 + 16)  // 16 : [dZ1]^T dOut|1  (col A+1 = db1)
static_assert(UT_DB1 + 16 <= UT_TMEM_COLS, "TMEM column plan");

// off: fp32 copy (or -1), off_bf16: bf16 copy (or -1), off_lo: bf16 of the remainder v - bf16(v) (or -1).
// Every load of the thread is issued before the first store (H * K / 512 = 4 or 8 loads in flight per thread).
template <int K>
__device__ __forceinline__ void ut_load_weight(char* smem, int off, const float* g, int d, int off_bf16 = -1, int off_lo = -1) {
    constexpr int N = H * K / UT_THREADS;
    float v[N];
#pragma unroll
    for (int n = 0; n < N; ++n) {
        const int i = threadIdx.x + n * UT_THREADS, j = i / K, k = i % K;
        v[n] = k < d ? __ldcg(g + j * d + k) : 0.0f;
    }
#pragma unroll
    for (int n = 0; n < N; ++n) {
        const int i = threadIdx.x + n * UT_THREADS, j = i / K, k = i % K;
        if (off >= 0) *reinterpret_cast<float*>(smem + off + ut_off(j, k, K)) = v[n];
        const __nv_bfloat16 hi = __float2bfloat16(v[n]);
        if (off_bf16 >= 0) *reinterpret_cast<__nv_bfloat16*>(smem + off_bf16 + ut_off16(j, k, K)) = hi;
        if (off_lo >= 0) *reinterpret_cast<__nv_bfloat16*>(smem + off_lo + ut_off16(j, k, K)) = __float2bfloat16(v[n] - __bfloat162float(hi));
    }
}

// Fused mode: the clip+Adam pass writes each updated parameter (flat index k of the parameter vector) straight into the
// operand / bias slot the next step's MMAs and epilogues read it from -- the same slots the staging at kernel start fills.
__device__ __forceinline__ void ut_store_param(char* smem, float* small, int k, float v, int d, uint32_t d_magic, int pi_count,
                                               int vf_count) {
    if (k >= pi_count + vf_count) { small[UtSmem::LOGSTD + k - pi_count - vf_count] = v; return; }
    const int t = k >= pi_count ? 1 : 0;     // tower
    int r = k - (t ? pi_count : 0);
    if (r < H * d) {
        const int j = (int)(((uint32_t)r * d_magic) >> 22), kk = r - j * d;     // r / d: exact for r < 2^22 / d
        *reinterpret_cast<float*>(smem + (t ? UtSmem::W1_VF : UtSmem::W1_PI) + ut_off(j, kk, DP)) = v;
        return;
    }
    r -= H * d;
    if (r < H) { small[UtSmem::B1 + t * H + r] = v; return; }
    r -= H;
    if (r < H * H) {
        const int j = r / H, kk = r % H;
        const __nv_bfloat16 hi = __float2bfloat16(v);
        *reinterpret_cast<__nv_bfloat16*>(smem + (t ? UtSmem::W2B_VF : UtSmem::W2B_PI) + ut_off16(j, kk, H)) = hi;
#if UT_SPLIT
        *reinterpret_cast<__nv_bfloat16*>(smem + (t ? UtSmem::W2L_VF : UtSmem::W2L_PI) + ut_off16(j, kk, H)) =
            __float2bfloat16(v - __bfloat162float(hi));
#else
        *reinterpret_cast<float*>(smem + (t ? UtSmem::W2_VF : UtSmem::W2_PI) + ut_off(j, kk, H)) = v;
#endif
        return;
    }
    r -= H * H;
    if (r < H) { small[UtSmem::B2 + t * H + r] = v; return; }
    r -= H;
    if (t == 0) {
        if (r < A * H) small[UtSmem::W3_PI + (r % H) * AP + r / H] = v;
        else small[UtSmem::B3_PI + r - A * H] = v;
    } else {
        if (r < H) small[UtSmem::W3_VF + r] = v;
        else small[UtSmem::B3_VF] = v;
    }
}

struct PpoLossCfg { float clip_range, ent_coef, vf_coef, inv_batch, grad_scale, inv_grad_scale; };
// Fused mode (steps > 0; one CTA): `steps` consecutive optimizer steps in one launch -- per step the minibatch's advantage
// statistics, the gradient (written to the caller's gradient buffer), clip_grad_norm_ and Adam on the parameters in global
// memory, which the next step then stages again.  stable_baselines3's batch_size = 128 is one tile per step.
struct PpoFusedCfg { int steps; float lr, beta1, beta2, eps, max_norm; float* params; float* m; float* v; int* step_ctr; float* norm_out;
                     int world, rank; unsigned* seq; float* peer[PEER_MAX_WORLD]; };

// Asynchronously gather 8 consecutive observation columns [8*part, 8*part+8) (per 32-column slab) of rollout row g straight into the
// fp32 layer-1 A operand (cp.async with zero fill for padding columns and dead rows): the random 112-byte row reads
// cost DRAM latency, and unlike register loads they cannot stall the issuing warp.
__device__ __forceinline__ void ut_gather_async(char* smem, const float* __restrict__ obs, int d, long long g, bool live,
                                                int grow, int part) {
    const float* src = obs + (size_t)g * d;
#pragma unroll
    for (int slab = 0; slab < DP / 32; ++slab, part += 4)
    if ((d & 3) == 0) {                                   // rows are 16-byte aligned: two 16-byte copies
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int k = 8 * part + 4 * h;
            const uint32_t dst = ut_smem_u32(smem + UtSmem::XB + ut_off(grow, k, DP));
            const bool ok = live && k < d;
            const float* sp = ok ? src + k : obs;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" :: "r"(dst), "l"(sp), "r"(ok ? 16 : 0) : "memory");
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = 8 * part + i;
            const uint32_t dst = ut_smem_u32(smem + UtSmem::XB + ut_off(grow, k, DP));
            const bool ok = live && k < d;
            const float* sp = ok ? src + k : obs;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" :: "r"(dst), "l"(sp), "r"(ok ? 4 : 0) : "memory");
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// out_partial: [gridDim.x][P] gradient partial sums; out_stats: [gridDim.x][8] (pi loss, v loss, approx kl, clip
// fraction, sum ratio, samples, -, -) as sums over the CTA's samples
//
// 512 threads = 4 warpgroups.  TMEM lane (= sample row of the tile) = tid & 127; warpgroup q = tid >> 7 owns the 32
// activation columns [32q, 32q+32) of the stacked pi|vf layer (q 0,1 = policy tower, 2,3 = value tower) in every
// epilogue, so the per-thread serial work is a quarter of a row and 16 warps hide each other's TMEM/SFU latency.
// tanh' factors are kept in registers (packed bf16) from the forward epilogues instead of being recomputed.
template <bool FUSED, bool P2P = false>
__global__ void __launch_bounds__(UT_THREADS, 1)
ppo_grad_tc_kernel(const float* params, int d, const float* __restrict__ obs, const float* __restrict__ act,
                   const float* __restrict__ logp_old, const float* __restrict__ adv, const float* __restrict__ ret,
                   const long long* __restrict__ idx_all, int batch, const float* __restrict__ adv_stats, PpoLossCfg cfg,
                   float* out_partial, float* __restrict__ out_stats, int P, PpoFusedCfg fz) {
    extern __shared__ __align__(1024) char smem[];
    float* small = reinterpret_cast<float*>(smem + UtSmem::SMALL);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int q = tid >> 7;                  // warpgroup = column block
    const int row = tid & (UT_ROWS - 1);     // sample row inside the tile = TMEM lane
    const int grow = tid >> 2, gpart = tid & 3;   // gather role: row, 8-column part
    const int pi_count = H * d + H + H * H + H + A * H + A;
    const int vf_count = H * d + H + H * H + H + H + 1;
    const float* g_pi = params;
    const float* g_vf = params + pi_count;

    const uint32_t bar = ut_smem_u32(&small[UtSmem::BAR]);
    uint32_t* tptr = reinterpret_cast<uint32_t*>(&small[UtSmem::TPTR]);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(ut_smem_u32(tptr)), "r"((uint32_t)UT_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tptr;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;     // a warp may touch TMEM lanes 32*(warp%4)..+31
    const uint32_t sb = ut_smem_u32(smem);
    uint32_t phase = 0;


#ifdef UT_PROFILE   // experiment builds: phase time stamps (ns) of the last fused step into out_stats[8..]
    unsigned long long ts[8];
    unsigned long long tt[10];     // ... and of its last tile into out_stats[16..]
#define UT_STAMP(i) do { if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts[i])); } while (0)
#define UT_TSTAMP(i) do { if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt[i])); } while (0)
#else
#define UT_TSTAMP(i) do { } while (0)
#define UT_STAMP(i) do { } while (0)
#endif
    const int nsteps = FUSED ? fz.steps : 1;
    // fused mode with whole tiles per minibatch: the steps' index lists form one contiguous tile stream, so the look-ahead
    // (observation gather + indices) of a step's last tile simply runs into the next step's first tile
    const bool stream = FUSED && (batch % UT_ROWS) == 0;
    long long g_loss = 0, g_gat = 0;
    for (int os = 0; os < nsteps; ++os) {
    UT_STAMP(0);
    const long long* __restrict__ idx = idx_all + (size_t)os * batch;
    if (!FUSED || os == 0) {     // later fused steps: the Adam pass of the previous step has already written every slot
    ut_load_weight<DP>(smem, UtSmem::W1_PI, g_pi, d);
    ut_load_weight<DP>(smem, UtSmem::W1_VF, g_vf, d);
#if UT_SPLIT
    ut_load_weight<H>(smem, -1, g_pi + H * d + H, H, UtSmem::W2B_PI, UtSmem::W2L_PI);
    ut_load_weight<H>(smem, -1, g_vf + H * d + H, H, UtSmem::W2B_VF, UtSmem::W2L_VF);
#else
    ut_load_weight<H>(smem, UtSmem::W2_PI, g_pi + H * d + H, H, UtSmem::W2B_PI);
    ut_load_weight<H>(smem, UtSmem::W2_VF, g_vf + H * d + H, H, UtSmem::W2B_VF);
#endif
    if (tid < H) {
        small[UtSmem::B1 + tid] = __ldcg(g_pi + H * d + tid);
        small[UtSmem::B1 + H + tid] = __ldcg(g_vf + H * d + tid);
        small[UtSmem::B2 + tid] = __ldcg(g_pi + H * d + H + H * H + tid);
        small[UtSmem::B2 + H + tid] = __ldcg(g_vf + H * d + H + H * H + tid);
        small[UtSmem::W3_VF + tid] = __ldcg(g_vf + H * d + H + H * H + H + tid);
    }
    for (int i = tid; i < AP * H; i += blockDim.x) {                                               // [j][a], zero padded to AP
        const int j = i / AP, a = i % AP;
        small[UtSmem::W3_PI + i] = a < A ? __ldcg(g_pi + H * d + H + H * H + H + a * H + j) : 0.0f;
    }
    if (tid < A) {
        small[UtSmem::B3_PI + tid] = __ldcg(g_pi + H * d + H + H * H + H + A * H + tid);
        small[UtSmem::LOGSTD + tid] = __ldcg(params + pi_count + vf_count + tid);
    }
    if (tid == 0) small[UtSmem::B3_VF] = __ldcg(g_vf + H * d + H + H * H + H + H);
    }
    if (FUSED) {
        // minibatch advantage statistics (mean, unbiased std) in double, summed in a fixed order; staged in the H2 buffer
        double sa = 0.0, sq = 0.0;
        for (int i = tid; i < batch; i += UT_THREADS) { const double v = (double)adv[idx[i]]; sa += v; sq += v * v; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { sa += __shfl_xor_sync(0xffffffffu, sa, o); sq += __shfl_xor_sync(0xffffffffu, sq, o); }
        double* sd = reinterpret_cast<double*>(smem + UtSmem::H2B);
        if ((tid & 31) == 0) { sd[2 * warp] = sa; sd[2 * warp + 1] = sq; }
        __syncthreads();
        if (tid == 0) {
            double ta = 0.0, tb = 0.0;
            for (int k = 0; k < UT_THREADS / 32; ++k) { ta += sd[2 * k]; tb += sd[2 * k + 1]; }
            // a one-sample minibatch is not normalised (stable_baselines3: normalize_advantage and len(advantages) > 1):
            // mean 0, std 1 make (adv - mean) / (std + 1e-8f) exactly adv
            const double n = (double)batch, mean = batch > 1 ? ta / n : 0.0;
            double var = batch > 1 ? (tb - n * mean * mean) / (n - 1.0) : 1.0;
            if (var < 0.0) var = 0.0;
            small[UtSmem::FUSED] = (float)mean; small[UtSmem::FUSED + 1] = (float)sqrt(var);
        }
    }
    __syncthreads();
    UT_STAMP(1);
    const float adv_mean = FUSED ? small[UtSmem::FUSED] : adv_stats[0];
    const float adv_istd = 1.0f / ((FUSED ? small[UtSmem::FUSED + 1] : adv_stats[1]) + 1e-8f);

    // per-thread running sums over this CTA's samples (warpgroup 0 only): db3_pi[4], db3_vf, dlogstd[4], loss statistics[6]
    float acc_db3[A], acc_db3v = 0.f, acc_dls[A];
#pragma unroll
    for (int a = 0; a < A; ++a) { acc_db3[a] = 0.f; acc_dls[a] = 0.f; }
    float st_pl = 0.f, st_vl = 0.f, st_kl = 0.f, st_clip = 0.f, st_ratio = 0.f, st_n = 0.f;

    const int ntiles = (batch + UT_ROWS - 1) / UT_ROWS;
    uint32_t first = 0;        // 0 on the first tile of this CTA: weight-gradient accumulators start from zero
    // Row indices run one tile ahead of the rows they address, so that neither the observation gather nor the
    // loss-input gather ever waits for an index: g_loss = this tile's sample, g_gat = next tile's gather row.
    const int ntiles_la = stream ? (nsteps - os) * ntiles : ntiles;       // look-ahead bounds (tiles, rows) from this step on
    const int rows_la = stream ? (nsteps - os) * batch : batch;
    if ((int)blockIdx.x < ntiles && !(stream && os > 0)) {
        const int sr = blockIdx.x * UT_ROWS + grow;
        const bool lv = sr < batch;
        ut_gather_async(smem, obs, d, lv ? idx[sr] : 0, lv, grow, gpart);
        const int sl = blockIdx.x * UT_ROWS + row;
        g_loss = sl < batch ? idx[sl] : 0;
        const int sn = (blockIdx.x + gridDim.x) * UT_ROWS + grow;
        g_gat = sn < rows_la ? idx[sn] : 0;
    }
    uint32_t m5_pending = 0;   // the previous tile's layer-1 weight-gradient MMAs are issued together with this tile's M1
    uint32_t m5_acc = 0;
    // M5: layer-1 weight / bias gradients (bf16): DW1 += [dZ1]^T X ; DB1 += [dZ1]^T dOut|1
#define UT_ISSUE_M5()                                                                                                   \
    do {                                                                                                                \
        ut_gemm<true, UT_ROWS / 16>(tmem + UT_DW1, sb + UtSmem::DZ1, 2 * H * 16, 128, 2 * 2 * H * 16, sb + UtSmem::XBB,  \
                                    DP * 16, 128, 2 * DP * 16, ut_idesc(1, DP, 1, 1), m5_acc);                          \
        ut_gemm<true, UT_ROWS / 16>(tmem + UT_DB1, sb + UtSmem::DZ1, 2 * H * 16, 128, 2 * 2 * H * 16, sb + UtSmem::DO,   \
                                    16 * 16, 128, 2 * 16 * 16, ut_idesc(1, 16, 1, 1), m5_acc);                          \
    } while (0)

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        UT_TSTAMP(0);
        // ---- S0: the gathered (already normalised) observations are the fp32 A operand of layer 1: wait for this
        //      thread's async copies (issued one tile ago), then make them visible block-wide
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        UT_FENCE_SYNC();       // also publishes the previous tile's dZ1
        UT_TSTAMP(1);
        // ---- M1: forward layer 1, both towers in one N = 128 GEMM (W1_pi and W1_vf are adjacent and form one
        //      [128 x 32] K-major B operand); then, behind the commit, M5 of the previous tile: it runs under E1 and is
        //      covered by M2's commit, before anything it reads (dZ1 = the H2 buffer, X bf16, dOut) is rewritten
        if (tid == 0) {
            ut_gemm<false, DP / 8>(tmem + UT_T1, sb + UtSmem::XB, 128, DP * 32, 256, sb + UtSmem::W1_PI, 128, DP * 32, 256,
                           ut_idesc(2, 2 * H, 0, 0), 0u);
            ut_commit(bar);
            if (m5_pending) UT_ISSUE_M5();
        }
        m5_acc = m5_pending;
        ut_wait(bar, phase); phase ^= 1u;
        UT_TSTAMP(2);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // bf16 copy of X (B operand of the layer-1 weight gradient): packed now, stored once the previous tile's M5,
        // which still reads the old copy, has drained (after the M2 wait)
        uint4 xbb[DP / 32];
#pragma unroll
        for (int slab = 0; slab < DP / 32; ++slab) {
            const int k = 8 * (gpart + 4 * slab);
            const float4 xa = *reinterpret_cast<const float4*>(smem + UtSmem::XB + ut_off(grow, k, DP));
            const float4 xb = *reinterpret_cast<const float4*>(smem + UtSmem::XB + ut_off(grow, k + 4, DP));
            const float x8[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
            xbb[slab] = ut_pack8(x8);
        }
        // loss inputs of the tile's samples: gathered by warpgroup 0 only (four separate random lines per sample; doing it
        // in all four warpgroups quadrupled the L1 wavefronts and stalled the block on the load queue), requested here so
        // that they fly under E1, M2 and E2, and shared through smem next to the head partials
        const int srow = tile * UT_ROWS + row;
        const bool live = srow < batch;
        float av[AP];
#pragma unroll
        for (int a = 0; a < AP; ++a) av[a] = 0.f;
        float lpo = 0.f, advv = 0.f, retv = 0.f;
        if (q == 0 && live) {
            if (A == 4) {
                const float4 a4 = reinterpret_cast<const float4*>(act)[g_loss];
                av[0] = a4.x; av[1] = a4.y; av[2] = a4.z; av[3] = a4.w;
            } else {                                      // rows of A floats: 8-byte aligned for even A
                const float2* ap = reinterpret_cast<const float2*>(act + (size_t)g_loss * A);
#pragma unroll
                for (int a = 0; a < A / 2; ++a) { const float2 t = ap[a]; av[2 * a] = t.x; av[2 * a + 1] = t.y; }
            }
            lpo = logp_old[g_loss]; advv = adv[g_loss]; retv = ret[g_loss];
        }
        // ---- E1: H1 = tanh(z1 + b1): fp32 for the forward, bf16 for the weight gradient of layer 2; keep 1 - H1^2
        uint32_t d1p[16], d2p[16];
        {
            float v[32];
            ut_ld32(tmem + UT_T1 + lane_base + q * 32, v);
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const int j = q * 32 + 8 * c8;
                float h[8], dd[8];
                const float4 ba = *reinterpret_cast<const float4*>(small + UtSmem::B1 + j), bb = *reinterpret_cast<const float4*>(small + UtSmem::B1 + j + 4);
                const float bias[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                for (int r = 0; r < 8; ++r) { h[r] = ut_tanh(v[8 * c8 + r] + bias[r]); dd[r] = fmaf(-h[r], h[r], 1.0f); }
#if UT_SPLIT
                {
                    const uint4 hi = ut_pack8(h);
                    *reinterpret_cast<uint4*>(smem + UtSmem::H1B + ut_off16(row, j, 2 * H)) = hi;
                    const uint32_t hw[4] = {hi.x, hi.y, hi.z, hi.w};
                    float lo[8];
#pragma unroll
                    for (int r = 0; r < 8; ++r)       // a bf16 is the top half of an fp32: hi as float by a shift / mask
                        lo[r] = h[r] - __uint_as_float((r & 1) ? (hw[r >> 1] & 0xffff0000u) : (hw[r >> 1] << 16));
                    *reinterpret_cast<uint4*>(smem + UtSmem::H1L + ut_off16(row, j, 2 * H)) = ut_pack8(lo);
                }
#else
                *reinterpret_cast<float4*>(smem + UtSmem::H1C + ut_off(row, j, 2 * H)) = make_float4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<float4*>(smem + UtSmem::H1C + ut_off(row, j + 4, 2 * H)) = make_float4(h[4], h[5], h[6], h[7]);
                *reinterpret_cast<uint4*>(smem + UtSmem::H1B + ut_off16(row, j, 2 * H)) = ut_pack8(h);
#endif
#pragma unroll
                for (int r = 0; r < 4; ++r) d1p[4 * c8 + r] = ut_pack2(dd[2 * r], dd[2 * r + 1]);
            }
        }
        UT_FENCE_SYNC();
        UT_TSTAMP(3);
        // ---- M2: forward layer 2 (A = the tower's 64-column sub-block of H1C)
        if (tid == 0) {
#if UT_SPLIT
            // z2 = H1 W2^T as hi*hi + lo*hi + hi*lo (bf16 operands, fp32 accumulation); tower t = columns 64t.. of H1
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const uint32_t ahi = sb + UtSmem::H1B + t * 8 * 128, alo = sb + UtSmem::H1L + t * 8 * 128;
                const uint32_t bhi = sb + (t ? UtSmem::W2B_VF : UtSmem::W2B_PI), blo = sb + (t ? UtSmem::W2L_VF : UtSmem::W2L_PI);
                ut_gemm<true, H / 16>(tmem + UT_T2 + t * H, ahi, 128, 2 * H * 16, 256, bhi, 128, H * 16, 256, ut_idesc(1, H, 0, 0), 0u);
                ut_gemm<true, H / 16>(tmem + UT_T2 + t * H, alo, 128, 2 * H * 16, 256, bhi, 128, H * 16, 256, ut_idesc(1, H, 0, 0), 1u);
                ut_gemm<true, H / 16>(tmem + UT_T2 + t * H, ahi, 128, 2 * H * 16, 256, blo, 128, H * 16, 256, ut_idesc(1, H, 0, 0), 1u);
            }
#else
            ut_gemm<false, H / 8>(tmem + UT_T2, sb + UtSmem::H1C, 128, 2 * H * 32, 256, sb + UtSmem::W2_PI, 128, H * 32, 256,
                           ut_idesc(2, H, 0, 0), 0u);
            ut_gemm<false, H / 8>(tmem + UT_T2 + H, sb + UtSmem::H1C + 16 * 128, 128, 2 * H * 32, 256, sb + UtSmem::W2_VF, 128, H * 32, 256,
                           ut_idesc(2, H, 0, 0), 0u);
#endif
            ut_commit(bar);
        }
        ut_wait(bar, phase); phase ^= 1u;
        UT_TSTAMP(4);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int slab = 0; slab < DP / 32; ++slab)
            *reinterpret_cast<uint4*>(smem + UtSmem::XBB + ut_off16(grow, 8 * (gpart + 4 * slab), DP)) = xbb[slab];
        // ---- E2: H2 = tanh(z2 + b2) (bf16 copy for the head weight gradient); partial head sums over this
        //      warpgroup's 32 hidden units (policy: 4 action means; value: 1)
        {
            float v[32];
            ut_ld32(tmem + UT_T2 + lane_base + q * 32, v);
            float ps[AP];
#pragma unroll
            for (int a = 0; a < AP; ++a) ps[a] = 0.f;
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const int j = q * 32 + 8 * c8;
                float h[8];
                const float4 ba = *reinterpret_cast<const float4*>(small + UtSmem::B2 + j), bb = *reinterpret_cast<const float4*>(small + UtSmem::B2 + j + 4);
                const float bias[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                for (int r = 0; r < 8; ++r) h[r] = ut_tanh(v[8 * c8 + r] + bias[r]);
                if (q < 2) {
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
#pragma unroll
                        for (int a4i = 0; a4i < AP / 4; ++a4i) {
                            const float4 w = *reinterpret_cast<const float4*>(small + UtSmem::W3_PI + (j + r) * AP + 4 * a4i);
                            ps[4 * a4i + 0] = fmaf(w.x, h[r], ps[4 * a4i + 0]); ps[4 * a4i + 1] = fmaf(w.y, h[r], ps[4 * a4i + 1]);
                            ps[4 * a4i + 2] = fmaf(w.z, h[r], ps[4 * a4i + 2]); ps[4 * a4i + 3] = fmaf(w.w, h[r], ps[4 * a4i + 3]);
                        }
                    }
                } else {
                    const float4 wa = *reinterpret_cast<const float4*>(small + UtSmem::W3_VF + j - H), wb = *reinterpret_cast<const float4*>(small + UtSmem::W3_VF + j - H + 4);
                    ps[0] = fmaf(wa.x, h[0], ps[0]); ps[0] = fmaf(wa.y, h[1], ps[0]); ps[0] = fmaf(wa.z, h[2], ps[0]); ps[0] = fmaf(wa.w, h[3], ps[0]);
                    ps[0] = fmaf(wb.x, h[4], ps[0]); ps[0] = fmaf(wb.y, h[5], ps[0]); ps[0] = fmaf(wb.z, h[6], ps[0]); ps[0] = fmaf(wb.w, h[7], ps[0]);
                }
                *reinterpret_cast<uint4*>(smem + UtSmem::H2B + ut_off16(row, j, 2 * H)) = ut_pack8(h);
#pragma unroll
                for (int r = 0; r < 4; ++r)
                    d2p[4 * c8 + r] = ut_pack2(fmaf(-h[2 * r], h[2 * r], 1.0f), fmaf(-h[2 * r + 1], h[2 * r + 1], 1.0f));
            }
            // XB is dead after M1: it carries the head partials of the four warpgroups and the loss inputs of each row
            if (q < 2) {
#pragma unroll
                for (int a4i = 0; a4i < AP / 4; ++a4i)
                    *reinterpret_cast<float4*>(smem + UtSmem::XB + UtSmem::PS_PI + ((q * UT_ROWS + row) * AP + 4 * a4i) * 4) =
                        make_float4(ps[4 * a4i], ps[4 * a4i + 1], ps[4 * a4i + 2], ps[4 * a4i + 3]);
            } else {
                *reinterpret_cast<float*>(smem + UtSmem::XB + UtSmem::PS_VF + ((q - 2) * UT_ROWS + row) * 4) = ps[0];
            }
            if (q == 0) {
                char* lin = smem + UtSmem::XB + UtSmem::LIN + row * UtSmem::LIN_ROW;
#pragma unroll
                for (int a4i = 0; a4i < AP / 4; ++a4i)
                    *reinterpret_cast<float4*>(lin + 16 * a4i) = make_float4(av[4 * a4i], av[4 * a4i + 1], av[4 * a4i + 2], av[4 * a4i + 3]);
                *reinterpret_cast<float4*>(lin + AP * 4) = make_float4(lpo, advv, retv, 0.f);
            }
        }
        __syncthreads();
        UT_TSTAMP(5);
        if (q != 0) {
            const char* lin = smem + UtSmem::XB + UtSmem::LIN + row * UtSmem::LIN_ROW;
#pragma unroll
            for (int a4i = 0; a4i < AP / 4; ++a4i) {
                const float4 t = *reinterpret_cast<const float4*>(lin + 16 * a4i);
                av[4 * a4i] = t.x; av[4 * a4i + 1] = t.y; av[4 * a4i + 2] = t.z; av[4 * a4i + 3] = t.w;
            }
            const float4 t = *reinterpret_cast<const float4*>(lin + AP * 4);
            lpo = t.x; advv = t.y; retv = t.z;
        }
        // ---- losses and their gradients w.r.t. the head outputs (stable_baselines3 PPO.train)
        float dout[AP], doutv = 0.f;     // pre-scaled by grad_scale
#pragma unroll
        for (int a = 0; a < AP; ++a) dout[a] = 0.f;
        {
            float mean[AP];
#pragma unroll
            for (int a4i = 0; a4i < AP / 4; ++a4i) {
                const float4 p0 = *reinterpret_cast<const float4*>(smem + UtSmem::XB + UtSmem::PS_PI + ((0 * UT_ROWS + row) * AP + 4 * a4i) * 4);
                const float4 p1 = *reinterpret_cast<const float4*>(smem + UtSmem::XB + UtSmem::PS_PI + ((1 * UT_ROWS + row) * AP + 4 * a4i) * 4);
                mean[4 * a4i + 0] = small[UtSmem::B3_PI + 4 * a4i + 0] + p0.x + p1.x; mean[4 * a4i + 1] = small[UtSmem::B3_PI + 4 * a4i + 1] + p0.y + p1.y;
                mean[4 * a4i + 2] = small[UtSmem::B3_PI + 4 * a4i + 2] + p0.z + p1.z; mean[4 * a4i + 3] = small[UtSmem::B3_PI + 4 * a4i + 3] + p0.w + p1.w;
            }
            const float pv0 = *reinterpret_cast<const float*>(smem + UtSmem::XB + UtSmem::PS_VF + (0 * UT_ROWS + row) * 4);
            const float pv1 = *reinterpret_cast<const float*>(smem + UtSmem::XB + UtSmem::PS_VF + (1 * UT_ROWS + row) * 4);
            const float val = small[UtSmem::B3_VF] + pv0 + pv1;
            if (live) {
                float z[A], sinv[A], lp = 0.0f;
#pragma unroll
                for (int a = 0; a < A; ++a) {
                    const float ls = small[UtSmem::LOGSTD + a];
                    sinv[a] = __expf(-ls);
                    z[a] = (av[a] - mean[a]) * sinv[a];
                    lp += -0.5f * z[a] * z[a] - ls - 0.91893853320467274178f;
                }
                const float lr = lp - lpo;
                const float ratio = __expf(lr);
                const float an = (advv - adv_mean) * adv_istd;
                const float s1 = an * ratio, s2 = an * fminf(fmaxf(ratio, 1.0f - cfg.clip_range), 1.0f + cfg.clip_range);
                // d/dlogp of -min(s1, s2): the unclipped branch carries gradient, the clamped one does not
                const float dlp = (s1 <= s2) ? -an * ratio * cfg.inv_batch : 0.0f;
                const float dv = cfg.vf_coef * 2.0f * (val - retv) * cfg.inv_batch;
#pragma unroll
                for (int a = 0; a < A; ++a) dout[a] = dlp * z[a] * sinv[a];
                if (q == 0) {     // sums are kept once per sample
#pragma unroll
                    for (int a = 0; a < A; ++a) { acc_db3[a] += dout[a]; acc_dls[a] += dlp * (z[a] * z[a] - 1.0f); }
                    acc_db3v += dv;
                    st_pl += -fminf(s1, s2); st_vl += (retv - val) * (retv - val);
                    st_kl += (ratio - 1.0f) - lr; st_clip += (fabsf(ratio - 1.0f) > cfg.clip_range) ? 1.0f : 0.0f;
                    st_ratio += ratio; st_n += 1.0f;
                }
                // scaled up before rounding to bf16 so that 1/batch factors do not underflow its range
#pragma unroll
                for (int a = 0; a < A; ++a) dout[a] *= cfg.grad_scale;
                doutv = dv * cfg.grad_scale;
            }
            if (q == 0) {
                // dOut row (bf16): [dmean0..A-1, dvalue, 1, 0...]; the ones column turns the same MMAs into bias-gradient sums
                float row16[16];
#pragma unroll
                for (int c = 0; c < 16; ++c) row16[c] = c < A ? dout[c] : (c == A ? doutv : (c == A + 1 ? (live ? 1.0f : 0.0f) : 0.0f));
                *reinterpret_cast<uint4*>(smem + UtSmem::DO + ut_off16(row, 0, 16)) = ut_pack8(row16);
                *reinterpret_cast<uint4*>(smem + UtSmem::DO + ut_off16(row, 8, 16)) = ut_pack8(row16 + 8);
            }
        }
        // ---- E3: dZ2 = (dOut W3) * tanh'(z2) for this warpgroup's columns (bf16, scaled) into the first half of the
        //      H1C area (dead after M2) -- the H2 copy stays intact for the head weight gradient
        {
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const int j = q * 32 + 8 * c8;
                float o[8];
                float wv[8];
                if (q >= 2) {
                    const float4 wa = *reinterpret_cast<const float4*>(small + UtSmem::W3_VF + j - H), wb = *reinterpret_cast<const float4*>(small + UtSmem::W3_VF + j - H + 4);
                    wv[0] = wa.x; wv[1] = wa.y; wv[2] = wa.z; wv[3] = wa.w; wv[4] = wb.x; wv[5] = wb.y; wv[6] = wb.z; wv[7] = wb.w;
                }
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    float dh;
                    if (q < 2) {
                        dh = 0.0f;
#pragma unroll
                        for (int a4i = 0; a4i < AP / 4; ++a4i) {
                            const float4 w = *reinterpret_cast<const float4*>(small + UtSmem::W3_PI + (j + r) * AP + 4 * a4i);
                            dh += dout[4 * a4i] * w.x + dout[4 * a4i + 1] * w.y + dout[4 * a4i + 2] * w.z + dout[4 * a4i + 3] * w.w;
                        }
                    } else {
                        dh = doutv * wv[r];
                    }
                    const __nv_bfloat162 dd = *reinterpret_cast<const __nv_bfloat162*>(&d2p[4 * c8 + (r >> 1)]);
                    o[r] = dh * ((r & 1) ? __high2float(dd) : __low2float(dd));
                }
                *reinterpret_cast<uint4*>(smem + UtSmem::DZ2 + ut_off16(row, j, 2 * H)) = ut_pack8(o);
            }
        }
        UT_FENCE_SYNC();
        UT_TSTAMP(6);
        // XB (layer-1 operand, then head partials) is free from here on: start the next tile's observation gather, and
        // fetch the indices for the iteration after it
        {
            const int nt = tile + gridDim.x;
            const int sr = nt * UT_ROWS + grow;
            ut_gather_async(smem, obs, d, g_gat, nt < ntiles_la && sr < rows_la, grow, gpart);
            const int sl = nt * UT_ROWS + row;
            g_loss = (nt < ntiles_la && sl < rows_la) ? idx[sl] : 0;
            const int sn = (nt + gridDim.x) * UT_ROWS + grow;
            g_gat = sn < rows_la ? idx[sn] : 0;
        }
        // ---- M3 + M4 (bf16).  Committed part: the head weight gradient (reads the H2 copy that E4 overwrites) and the
        //      data gradient into layer 1 (E4 consumes it).  The layer-2 weight / bias gradients go out behind the commit:
        //      they run under E4 and the next tile's S0 and are covered by the next commit.
        if (tid == 0) {
            // D3 += [H2]^T dOut   (A and B MN-major; K = 128 samples)
            ut_gemm<true, UT_ROWS / 16>(tmem + UT_D3, sb + UtSmem::H2B, 2 * H * 16, 128, 2 * 2 * H * 16, sb + UtSmem::DO, 16 * 16, 128, 2 * 16 * 16, ut_idesc(1, 16, 1, 1), first);
            // dH1 = dZ2 W2: A = the tower's K-major sub-block of the dZ2 buffer, B = W2 (bf16) read MN-major
            ut_gemm<true, H / 16>(tmem + UT_T2, sb + UtSmem::DZ2, 128, 2 * H * 16, 256, sb + UtSmem::W2B_PI, H * 16, 128, 2 * H * 16,
                          ut_idesc(1, H, 0, 1), 0u);
            ut_gemm<true, H / 16>(tmem + UT_T2 + H, sb + UtSmem::DZ2 + 8 * 128, 128, 2 * H * 16, 256, sb + UtSmem::W2B_VF, H * 16, 128, 2 * H * 16, ut_idesc(1, H, 0, 1), 0u);
            ut_commit(bar);
            // [Da | Db] += [dZ2]^T [H1_pi | H1_vf] as one N = 128 GEMM: rows 0-63 x cols 0-63 = dW2_pi,
            // rows 64-127 x cols 64-127 = dW2_vf (the cross-tower blocks are computed and ignored)
            ut_gemm<true, UT_ROWS / 16>(tmem + UT_DA, sb + UtSmem::DZ2, 2 * H * 16, 128, 2 * 2 * H * 16, sb + UtSmem::H1B, 2 * H * 16, 128, 2 * 2 * H * 16, ut_idesc(1, 2 * H, 1, 1), first);
            ut_gemm<true, UT_ROWS / 16>(tmem + UT_DB2, sb + UtSmem::DZ2, 2 * H * 16, 128, 2 * 2 * H * 16, sb + UtSmem::DO, 16 * 16, 128, 2 * 16 * 16, ut_idesc(1, 16, 1, 1), first);
        }
        ut_wait(bar, phase); phase ^= 1u;
        UT_TSTAMP(7);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- E4: dZ1 = dH1 * tanh'(z1) (bf16, already scaled) over the H2 copy (M3 has consumed it); its MMAs (M5)
        //      go out behind the next tile's M1
        {
            float v[32];
            ut_ld32(tmem + UT_T2 + lane_base + q * 32, v);
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const int j = q * 32 + 8 * c8;
                float o[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const __nv_bfloat162 dd = *reinterpret_cast<const __nv_bfloat162*>(&d1p[4 * c8 + (r >> 1)]);
                    o[r] = v[8 * c8 + r] * ((r & 1) ? __high2float(dd) : __low2float(dd));
                }
                *reinterpret_cast<uint4*>(smem + UtSmem::DZ1 + ut_off16(row, j, 2 * H)) = ut_pack8(o);
            }
        }
        first = 1u;
        m5_pending = 1u;
        UT_TSTAMP(8);
    }
    if (!stream) asm volatile("cp.async.wait_group 0;" ::: "memory");      // the last iteration's (empty) look-ahead gather
    if (first != 0u) {
        UT_FENCE_SYNC();
        if (tid == 0) { UT_ISSUE_M5(); ut_commit(bar); }
        ut_wait(bar, phase); phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
#undef UT_ISSUE_M5
    UT_STAMP(2);

    // ---- read the accumulated weight gradients out of TMEM into this CTA's partial
    //      (TMEM lane = output neuron: lanes 0-63 policy tower, 64-127 value tower; warpgroup q takes a column slice)
    float* outp = out_partial + (size_t)blockIdx.x * P;
    const bool is_pi = row < H;
    const int j = is_pi ? row : row - H;                 // neuron index inside the tower
    const int tower_off = is_pi ? 0 : pi_count;
    const int o_w1 = tower_off, o_b1 = o_w1 + H * d, o_w2 = o_b1 + H, o_b2 = o_w2 + H * H, o_w3 = o_b2 + H;
    if (first != 0u) {
        {   // dW2: rows 0-63 of Da, rows 64-127 of Db; 16 columns per warpgroup
            float v[16];
            ut_ld16(tmem + (is_pi ? UT_DA : UT_DB) + lane_base + q * 16, v);
            float* dst = outp + o_w2 + j * H + q * 16;
            // a warp-wide scalar store touches 32 sectors per instruction: 16-byte stores where the row allows
            if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
#pragma unroll
                for (int c = 0; c < 16; c += 4)
                    *reinterpret_cast<float4*>(dst + c) = make_float4(v[c] * cfg.inv_grad_scale, v[c + 1] * cfg.inv_grad_scale,
                                                                      v[c + 2] * cfg.inv_grad_scale, v[c + 3] * cfg.inv_grad_scale);
            } else {
#pragma unroll
                for (int c = 0; c < 16; ++c) dst[c] = v[c] * cfg.inv_grad_scale;
            }
        }
        if (q < 2) {   // dW1: DP/2 columns each
#pragma unroll
            for (int c0 = q * (DP / 2); c0 < (q + 1) * (DP / 2); c0 += 16) {
                float v[16];
                ut_ld16(tmem + UT_DW1 + lane_base + c0, v);
                float* dst = outp + o_w1 + j * d + c0;
                if ((d & 3) == 0 && (reinterpret_cast<uintptr_t>(outp + o_w1) & 15u) == 0) {
#pragma unroll
                    for (int c = 0; c < 16; c += 4)
                        if (c0 + c < d)
                            *reinterpret_cast<float4*>(dst + c) = make_float4(v[c] * cfg.inv_grad_scale, v[c + 1] * cfg.inv_grad_scale,
                                                                              v[c + 2] * cfg.inv_grad_scale, v[c + 3] * cfg.inv_grad_scale);
                } else {
#pragma unroll
                    for (int c = 0; c < 16; ++c) if (c0 + c < d) dst[c] = v[c] * cfg.inv_grad_scale;
                }
            }
        } else if (q == 2) {   // head weights
            float v3[16];
            ut_ld16(tmem + UT_D3 + lane_base, v3);
            if (is_pi) {
#pragma unroll
                for (int a = 0; a < A; ++a) outp[o_w3 + a * H + j] = v3[a] * cfg.inv_grad_scale;
            } else {
                outp[o_w3 + j] = v3[A] * cfg.inv_grad_scale;
            }
        } else {               // hidden biases (ones column)
            float vb2[16], vb1[16];
            ut_ld16(tmem + UT_DB2 + lane_base, vb2);
            ut_ld16(tmem + UT_DB1 + lane_base, vb1);
            outp[o_b2 + j] = vb2[A + 1] * cfg.inv_grad_scale;
            outp[o_b1 + j] = vb1[A + 1] * cfg.inv_grad_scale;
        }
    } else {
        // this CTA had no tile: its partial is all zeros
        for (int k = tid; k < P; k += blockDim.x) outp[k] = 0.0f;
    }
    // small sums (held by warpgroup 0): warp shuffle, one slot per (warp, sum) in the dead H2 buffer, then a
    // fixed-order sum over the four warps -- no floating-point atomics, the update is bit-reproducible
    float* wred = reinterpret_cast<float*>(smem + UtSmem::H2B);     // dead after the last M5; XB may hold the next step's rows
    if (q == 0) {
        // slots: db3_pi[A], db3_vf, dlog_std[A], then the six loss statistics
        float red[2 * A + 7];
#pragma unroll
        for (int a = 0; a < A; ++a) { red[a] = acc_db3[a]; red[A + 1 + a] = acc_dls[a]; }
        red[A] = acc_db3v;
        red[2 * A + 1] = st_pl; red[2 * A + 2] = st_vl; red[2 * A + 3] = st_kl; red[2 * A + 4] = st_clip; red[2 * A + 5] = st_ratio;
        red[2 * A + 6] = st_n;
#pragma unroll
        for (int k = 0; k < 2 * A + 7; ++k) {
            float x = red[k];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
            if ((tid & 31) == 0) wred[warp * 24 + k] = x;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid < 2 * A + 7) small[UtSmem::RED + tid] = (wred[tid] + wred[24 + tid]) + (wred[48 + tid] + wred[72 + tid]);
    __syncthreads();
    if (tid < A) {
        outp[pi_count - A + tid] = small[UtSmem::RED + tid];                                  // db3_pi
        // entropy bonus: loss += -ent_coef * mean(entropy), d/dlog_std = -ent_coef (added once, by CTA 0)
        outp[pi_count + vf_count + tid] = small[UtSmem::RED + A + 1 + tid] + (blockIdx.x == 0 ? -cfg.ent_coef : 0.0f);
    }
    if (tid == 0) outp[pi_count + vf_count - 1] = small[UtSmem::RED + A];                     // db3_vf
    if (tid < 8) {
        float v = 0.0f;
        if (tid < 6) v = small[UtSmem::RED + 2 * A + 1 + tid];
        out_stats[(size_t)blockIdx.x * 8 + tid] = v;
    }
    if (FUSED) {
        // ---- clip_grad_norm_ + Adam on the gradient this CTA has just written (the arithmetic of ppo_adam_kernel)
        __threadfence();
        __syncthreads();
        UT_STAMP(3);
        constexpr int NP = 16384 / UT_THREADS;
        float gscale = 1.0f;
        if (P2P && fz.world > 1) {
            // gradient all-reduce over NVLink peer memory (value + sequence number per 8-byte store, see the top of the file):
            // every rank's CTA pushes its elements to the others, collects theirs, and leaves the rank-ordered sum in outp
            const unsigned qn = fz.seq[0] + 1u;
#pragma unroll 1
            for (int i0 = 0; i0 < NP; i0 += 8) {
                if (i0 * UT_THREADS >= P) break;
                float own[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int k = tid + (i0 + i) * UT_THREADS; own[i] = k < P ? __ldcg(outp + k) : 0.0f; }
                peer_push<8>(own, P, tid + i0 * UT_THREADS, UT_THREADS, fz.world, fz.rank, qn, fz.peer);
            }
#pragma unroll 1
            for (int i0 = 0; i0 < NP; i0 += 8) {
                if (i0 * UT_THREADS >= P) break;
                float own[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int k = tid + (i0 + i) * UT_THREADS; own[i] = k < P ? __ldcg(outp + k) : 0.0f; }
                peer_collect<8>(own, P, tid + i0 * UT_THREADS, UT_THREADS, fz.world, fz.rank, qn, fz.peer);
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int k = tid + (i0 + i) * UT_THREADS; if (k < P) outp[k] = own[i]; }
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) fz.seq[0] = qn;
            gscale = 1.0f / (float)fz.world;
        }
        // squared norm over this thread's parameters (k = tid + 512 i); every load issued before the first use
        float ss = 0.0f;
        {
            float g[NP];
#pragma unroll
            for (int i = 0; i < NP; ++i) { const int k = tid + i * UT_THREADS; g[i] = k < P ? __ldcg(outp + k) * gscale : 0.0f; }
#pragma unroll
            for (int i = 0; i < NP; ++i) ss = fmaf(g[i], g[i], ss);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if ((tid & 31) == 0) wred[warp] = ss;
        __syncthreads();
        if (tid == 0) {
            float x = 0.0f;
            for (int k = 0; k < UT_THREADS / 32; ++k) x += wred[k];
            const float norm = sqrtf(x);
            const int t = fz.step_ctr[0] + 1;
            small[UtSmem::FUSED + 2] = fminf(1.0f, fz.max_norm / (norm + 1e-6f));
            small[UtSmem::FUSED + 3] = __int_as_float(t);
            fz.step_ctr[0] = t;
            if (fz.norm_out != nullptr) fz.norm_out[0] = norm;
        }
        __syncthreads();
        UT_STAMP(4);
        const float coef = small[UtSmem::FUSED + 2];
        const float tf = (float)__float_as_int(small[UtSmem::FUSED + 3]);
        const float inv_bc1 = 1.0f / (1.0f - powf(fz.beta1, tf)), inv_bc2 = 1.0f / (1.0f - powf(fz.beta2, tf));
        const uint32_t d_magic = ((1u << 22) + (uint32_t)d - 1u) / (uint32_t)d;
#pragma unroll 1
        for (int i0 = 0; i0 < NP; i0 += 8) {          // eight parameters at a time: 32 loads in flight, then arithmetic
            if (i0 * UT_THREADS >= P) break;
            float gk[8], mk[8], vk[8], pk[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k = tid + (i0 + i) * UT_THREADS;
                const bool ok = k < P;
                gk[i] = ok ? __ldcg(outp + k) * gscale : 0.0f;
                mk[i] = ok ? fz.m[k] : 0.0f; vk[i] = ok ? fz.v[k] : 0.0f; pk[i] = ok ? __ldcg(fz.params + k) : 0.0f;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k = tid + (i0 + i) * UT_THREADS;
                if (k < P) {
                    const float gg = gk[i] * coef;
                    const float m1 = fz.beta1 * mk[i] + (1.0f - fz.beta1) * gg;
                    const float v1 = fz.beta2 * vk[i] + (1.0f - fz.beta2) * gg * gg;
                    fz.m[k] = m1; fz.v[k] = v1;
                    const float pn = pk[i] - fz.lr * (m1 * inv_bc1) / (sqrtf(v1 * inv_bc2) + fz.eps);
                    fz.params[k] = pn;
                    ut_store_param(smem, small, k, pn, d, d_magic, pi_count, vf_count);
                }
            }
        }
        __threadfence();
        __syncthreads();       // the next step stages the updated parameters
        UT_STAMP(5);
#ifdef UT_PROFILE
        if (tid == 0) for (int i = 0; i < 5; ++i) out_stats[8 + i] = (float)(ts[i + 1] - ts[i]);
        if (tid == 0) for (int i = 0; i < 8; ++i) out_stats[16 + i] = (float)(tt[i + 1] - tt[i]);
#endif
    }
    }   // optimizer steps
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"((uint32_t)UT_TMEM_COLS) : "memory");
}

}  // namespace PPO_UT_NS

#ifdef PPO_UT_SHARED
// ------------------------------------------------------------------ minibatch advantage statistics (mean, unbiased std)
// scratch: [0] block-arrival counter, [2 + 2b], [3 + 2b] = block b's sum / sum of squares; the last block to arrive adds the
// block partials in index order (no floating-point atomics: the statistics do not depend on the block schedule)
// blockIdx.y = minibatch of a window of consecutive minibatches (its own index slice, scratch slice and output pair)
#define ADV_MAX_BLOCKS 592
#define ADV_SCRATCH_DOUBLES (2 + 2 * ADV_MAX_BLOCKS)
__global__ void __launch_bounds__(256)
ppo_adv_stats_kernel(const float* __restrict__ adv, const long long* __restrict__ idx, int batch, double* __restrict__ scratch,
                     float* __restrict__ out) {
    __shared__ double s_a[8], s_b[8];
    __shared__ bool is_last;
    idx += (size_t)blockIdx.y * batch; scratch += (size_t)blockIdx.y * ADV_SCRATCH_DOUBLES; out += 2 * blockIdx.y;
    double a = 0.0, b = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < batch; i += gridDim.x * blockDim.x) {
        double v = (double)adv[idx[i]];
        a += v; b += v * v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    if ((threadIdx.x & 31) == 0) { s_a[threadIdx.x >> 5] = a; s_b[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ta = 0, tb = 0;
        for (int k = 0; k < 8; ++k) { ta += s_a[k]; tb += s_b[k]; }
        scratch[2 + 2 * blockIdx.x] = ta; scratch[3 + 2 * blockIdx.x] = tb;
        __threadfence();
        double prev = atomicAdd(&scratch[0], 1.0);
        is_last = (prev == (double)(gridDim.x - 1));
    }
    __syncthreads();
    if (!is_last || threadIdx.x >= 32) return;
    __threadfence();
    const volatile double* sc = scratch;
    double ta = 0.0, tb = 0.0;
    for (int k = threadIdx.x; k < (int)gridDim.x; k += 32) { ta += sc[2 + 2 * k]; tb += sc[3 + 2 * k]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { ta += __shfl_xor_sync(0xffffffffu, ta, o); tb += __shfl_xor_sync(0xffffffffu, tb, o); }
    if (threadIdx.x != 0) return;
    // torch.std(): unbiased; a one-sample minibatch is not normalised (mean 0, std 1: see ppo_grad_tc_kernel)
    double n = (double)batch, mean = batch > 1 ? ta / n : 0.0;
    double var = batch > 1 ? (tb - n * mean * mean) / (n - 1.0) : 1.0;
    if (var < 0.0) var = 0.0;
    out[0] = (float)mean; out[1] = (float)sqrt(var);
    scratch[0] = 0.0;
}

// ------------------------------------------------------------------ partial-gradient reduction: grad[k] = sum_c partial[c][k]
// block = 64 parameters x 16 slices of the CTA axis: 16 independent load chains per parameter instead of one
#define RED_KX 64
#define RED_CY 16
// adam.enabled: single-process update (no all-reduce between gradient and optimizer) -- the last block to finish its slice
// of the reduction runs clip + Adam on the complete gradient, saving the optimizer's own launch
struct PpoAdamArgs { int enabled; float lr, beta1, beta2, eps, max_norm; float* params; float* m; float* v; int* step_ctr; float* norm_out;
                     unsigned* arrivals; int world, rank; unsigned* seq; float* peer[PEER_MAX_WORLD]; };
#define ADAM_THREADS 1024
#define ADAM_PER 16          // parameters per thread held in registers: P <= 16384
__device__ __forceinline__ void ppo_adam_block(float* params, const float* grad, float* m, float* v, int P, float lr, float beta1,
                                               float beta2, float eps, float max_norm, float grad_scale, int* step_ctr,
                                               float* norm_out, float* s_red, float* s_coef);
__global__ void __launch_bounds__(RED_KX * RED_CY)
ppo_grad_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ stats_partial, int ncta, int P,
                       float* grad, float* __restrict__ stats, PpoAdamArgs adam) {
    __shared__ float s_part[RED_CY][RED_KX + 1];
    const int kx = threadIdx.x % RED_KX, cy = threadIdx.x / RED_KX;
    const int k = blockIdx.x * RED_KX + kx;
    float s = 0.0f;
    if (k < P)
        for (int c = cy; c < ncta; c += RED_CY) s += partial[(size_t)c * P + k];
    s_part[cy][kx] = s;
    __syncthreads();
    if (cy == 0 && k < P) {
        float t = 0.0f;
#pragma unroll
        for (int c = 0; c < RED_CY; ++c) t += s_part[c][kx];          // fixed order: deterministic
        grad[k] = t;
    }
    if (blockIdx.x == 0 && threadIdx.x < 8 && stats != nullptr) {
        float t = 0.0f;
        for (int c = 0; c < ncta; ++c) t += stats_partial[(size_t)c * 8 + threadIdx.x];
        stats[threadIdx.x] = t;
    }
    if (!adam.enabled) return;
    __shared__ bool is_last;
    __shared__ float s_red[32];
    __shared__ float s_coef;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned prev = atomicAdd(adam.arrivals, 1u);
        is_last = prev == gridDim.x - 1;
        if (is_last) *adam.arrivals = 0u;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    float scale = 1.0f;
    if (adam.world > 1) {
        const unsigned q = adam.seq[0] + 1u;                 // sequence number of this optimizer step (same on every rank)
        {
            float own[ADAM_PER];
#pragma unroll
            for (int i = 0; i < ADAM_PER; ++i) { const int k = threadIdx.x + i * ADAM_THREADS; own[i] = k < P ? __ldcg(grad + k) : 0.0f; }
            peer_push<ADAM_PER>(own, P, threadIdx.x, ADAM_THREADS, adam.world, adam.rank, q, adam.peer);
            peer_collect<ADAM_PER>(own, P, threadIdx.x, ADAM_THREADS, adam.world, adam.rank, q, adam.peer);
#pragma unroll
            for (int i = 0; i < ADAM_PER; ++i) {    // what an all-reduce(sum) leaves in the gradient buffer
                const int k = threadIdx.x + i * ADAM_THREADS;
                if (k < P) grad[k] = own[i];
            }
        }
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) adam.seq[0] = q;
        scale = 1.0f / (float)adam.world;
    }
    ppo_adam_block(adam.params, grad, adam.m, adam.v, P, adam.lr, adam.beta1, adam.beta2, adam.eps, adam.max_norm, scale,
                   adam.step_ctr, adam.norm_out, s_red, &s_coef);
}

// ------------------------------------------------------------------ clip_grad_norm_ + Adam, one block
static_assert(ADAM_THREADS == RED_KX * RED_CY, "the reduction's last block runs the Adam body");
// the whole update by ONE block of ADAM_THREADS threads; grad may have been written by other blocks of the same launch
// (ppo_grad_reduce_kernel's last block), hence the L2 loads
__device__ __forceinline__ void ppo_adam_block(float* params, const float* grad, float* m, float* v, int P, float lr, float beta1,
                                               float beta2, float eps, float max_norm, float grad_scale, int* step_ctr,
                                               float* norm_out, float* s_red, float* s_coef) {
    // every load of the update is issued before the norm reduction so that the second pass only does arithmetic
    float g[ADAM_PER], mk[ADAM_PER], vk[ADAM_PER], pk[ADAM_PER];
    float ss = 0.0f;
#pragma unroll
    for (int i = 0; i < ADAM_PER; ++i) {
        const int k = threadIdx.x + i * ADAM_THREADS;
        const bool ok = k < P;
        g[i] = ok ? __ldcg(grad + k) * grad_scale : 0.0f;
        mk[i] = ok ? m[k] : 0.0f; vk[i] = ok ? v[k] : 0.0f; pk[i] = ok ? params[k] : 0.0f;
        ss = fmaf(g[i], g[i], ss);
    }
    const int t = step_ctr[0] + 1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x < 32) {
        float x = s_red[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (threadIdx.x == 0) {
            const float norm = sqrtf(x);
            *s_coef = fminf(1.0f, max_norm / (norm + 1e-6f));          // torch.nn.utils.clip_grad_norm_
            if (norm_out != nullptr) norm_out[0] = norm;
            step_ctr[0] = t;
        }
    }
    __syncthreads();
    const float coef = *s_coef;
    const float bc1 = 1.0f - powf(beta1, (float)t), bc2 = 1.0f - powf(beta2, (float)t);
    const float inv_bc1 = 1.0f / bc1, inv_bc2 = 1.0f / bc2;
#pragma unroll
    for (int i = 0; i < ADAM_PER; ++i) {
        const int k = threadIdx.x + i * ADAM_THREADS;
        if (k < P) {
            const float gg = g[i] * coef;
            const float m1 = beta1 * mk[i] + (1.0f - beta1) * gg;
            const float v1 = beta2 * vk[i] + (1.0f - beta2) * gg * gg;
            m[k] = m1; v[k] = v1;
            params[k] = pk[i] - lr * (m1 * inv_bc1) / (sqrtf(v1 * inv_bc2) + eps);   // torch.optim.Adam (no amsgrad / decay)
        }
    }
}

__global__ void __launch_bounds__(ADAM_THREADS)
ppo_adam_kernel(float* params, const float* grad, float* m, float* v, int P, float lr, float beta1, float beta2, float eps,
                float max_norm, float grad_scale, int* step_ctr, float* norm_out) {
    __shared__ float s_red[32];
    __shared__ float s_coef;
    ppo_adam_block(params, grad, m, v, P, lr, beta1, beta2, eps, max_norm, grad_scale, step_ctr, norm_out, s_red, &s_coef);
}

// ------------------------------------------------------------------ launchers
size_t ppok_peer_bytes() { return (size_t)PEER_BYTES; }
static int g_ut_sm_count_shared = 0;

int ppok_update_grid(int batch) {
    if (g_ut_sm_count_shared == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return -1;
        if (cudaDeviceGetAttribute(&g_ut_sm_count_shared, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    }
    const int ntiles = (batch + UT_ROWS - 1) / UT_ROWS;
    return ntiles < g_ut_sm_count_shared ? ntiles : g_ut_sm_count_shared;
}

// nmb consecutive minibatches (idx slices of `batch`) in one launch: scratch / adv_stats slices per minibatch
void ppok_launch_adv_stats(const float* adv, const long long* idx, int batch, int nmb, double* scratch, float* adv_stats, cudaStream_t st) {
    int sblocks = (batch + 255) / 256;            // one gathered element per thread up to 4 blocks per SM
    if (sblocks > ADV_MAX_BLOCKS) sblocks = ADV_MAX_BLOCKS;
    ppo_adv_stats_kernel<<<dim3(sblocks, nmb), 256, 0, st>>>(adv, idx, batch, scratch, adv_stats);
}

void ppok_launch_grad_reduce(const float* partial, const float* stats_partial, int grid, int P, float* grad, float* stats,
                             const PpokAdam* adam, cudaStream_t st) {
    PpoAdamArgs a{};
    if (adam != nullptr) {
        a = PpoAdamArgs{1, adam->lr, adam->beta1, adam->beta2, adam->eps, adam->max_norm, adam->params, adam->m, adam->v, adam->step_ctr,
                        adam->norm_out, adam->arrivals, adam->world, adam->rank, adam->seq, {}};
        for (int j = 0; j < PEER_MAX_WORLD; ++j) a.peer[j] = j < adam->world ? adam->peer[j] : nullptr;
    }
    ppo_grad_reduce_kernel<<<(P + RED_KX - 1) / RED_KX, RED_KX * RED_CY, 0, st>>>(partial, stats_partial, grid, P, grad, stats, a);
}

cudaError_t ppok_adam(float* params, const float* grad, float* m, float* v, int P, float lr, float beta1, float beta2, float eps,
                      float max_norm, float grad_scale, int* step_ctr, float* norm_out, cudaStream_t st) {
    if (P > ADAM_THREADS * ADAM_PER) return cudaErrorInvalidValue;
    ppo_adam_kernel<<<1, ADAM_THREADS, 0, st>>>(params, grad, m, v, P, lr, beta1, beta2, eps, max_norm, grad_scale, step_ctr, norm_out);
    return cudaGetLastError();
}
#endif  // PPO_UT_SHARED

void ppok_launch_adv_stats(const float* adv, const long long* idx, int batch, int nmb, double* scratch, float* adv_stats, cudaStream_t st);
void ppok_launch_grad_reduce(const float* partial, const float* stats_partial, int grid, int P, float* grad, float* stats,
                             const PpokAdam* adam, cudaStream_t st);

namespace PPO_UT_NS {
static bool g_ut_attr_set = false, g_ut_fused_attr_set = false;

cudaError_t ppok_minibatch_grad(const float* params, int d, const float* obs, const float* act, const float* logp_old,
                                const float* adv, const float* ret, const long long* idx, int batch, float clip_range,
                                float ent_coef, float vf_coef, double* scratch, float* adv_stats, float* partial,
                                float* stats_partial, float* grad, float* stats, cudaStream_t st, const PpokAdam* adam,
                                int have_adv_stats) {
    if (d > DP) return cudaErrorInvalidValue;
    if (!g_ut_attr_set) {
        cudaError_t e = cudaFuncSetAttribute(ppo_grad_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UtSmem::TOTAL);
        if (e != cudaSuccess) return e;
        g_ut_attr_set = true;
    }
    const int grid = ppok_update_grid(batch);
    if (grid <= 0) return cudaErrorUnknown;
    const int H_ = PPO_H, A_ = A;
    const int P = (H_ * d + H_ + H_ * H_ + H_ + A_ * H_ + A_) + (H_ * d + H_ + H_ * H_ + H_ + H_ + 1) + A_;
    if (!have_adv_stats) ppok_launch_adv_stats(adv, idx, batch, 1, scratch, adv_stats, st);
    // per-sample head gradients carry a 1/batch factor; rescale them to O(1) before the bf16 rounding of the backward
    // operands (a power of two, so the scaling itself is exact) and undo it when the accumulators are read out
    float gs = 1.0f;
    while (gs < (float)batch && gs < 1048576.0f) gs *= 2.0f;
    PpoLossCfg cfg{clip_range, ent_coef, vf_coef, 1.0f / (float)batch, gs, 1.0f / gs};
    PpoFusedCfg fz{};
    ppo_grad_tc_kernel<false><<<grid, UT_THREADS, UtSmem::TOTAL, st>>>(params, d, obs, act, logp_old, adv, ret, idx, batch, adv_stats, cfg,
                                                             partial, stats_partial, P, fz);
    ppok_launch_grad_reduce(partial, stats_partial, grid, P, grad, stats, adam, st);
    return cudaGetLastError();
}

// `steps` consecutive optimizer steps over idx[0 .. steps*batch) in ONE single-CTA launch (see PpoFusedCfg)
cudaError_t ppok_minibatch_steps(float* params, int d, const float* obs, const float* act, const float* logp_old, const float* adv,
                                 const float* ret, const long long* idx, int batch, int steps, float clip_range, float ent_coef,
                                 float vf_coef, float* m, float* v, float lr, float beta1, float beta2, float eps, float max_norm,
                                 int* step_ctr, float* norm_out, float* grad, float* stats, cudaStream_t st, int world, int rank,
                                 void* const* peers, unsigned* seq) {
    if (d > DP || steps <= 0 || world > PEER_MAX_WORLD) return cudaErrorInvalidValue;
    if (!g_ut_fused_attr_set) {
        cudaError_t e = cudaFuncSetAttribute(ppo_grad_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, UtSmem::TOTAL);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(ppo_grad_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, UtSmem::TOTAL);
        if (e != cudaSuccess) return e;
        g_ut_fused_attr_set = true;
    }
    const int H_ = PPO_H, A_ = A;
    const int P = (H_ * d + H_ + H_ * H_ + H_ + A_ * H_ + A_) + (H_ * d + H_ + H_ * H_ + H_ + H_ + 1) + A_;
    float gs = 1.0f;
    while (gs < (float)batch && gs < 1048576.0f) gs *= 2.0f;
    PpoLossCfg cfg{clip_range, ent_coef, vf_coef, 1.0f / (float)batch, gs, 1.0f / gs};
    PpoFusedCfg fz{steps, lr, beta1, beta2, eps, max_norm, params, m, v, step_ctr, norm_out, world > 1 ? world : 1, rank, seq, {}};
    for (int j = 0; j < PEER_MAX_WORLD; ++j) fz.peer[j] = (world > 1 && j < world) ? static_cast<float*>(peers[j]) : nullptr;
    if (world > 1)
        ppo_grad_tc_kernel<true, true><<<1, UT_THREADS, UtSmem::TOTAL, st>>>(params, d, obs, act, logp_old, adv, ret, idx, batch, nullptr,
                                                                          cfg, grad, stats, P, fz);
    else
        ppo_grad_tc_kernel<true, false><<<1, UT_THREADS, UtSmem::TOTAL, st>>>(params, d, obs, act, logp_old, adv, ret, idx, batch, nullptr,
                                                                           cfg, grad, stats, P, fz);
    return cudaGetLastError();
}
}  // namespace PPO_UT_NS
