// fw_kernels.cu -- sm_100a kernels of the batched fixed-wing env step.
//
// K1 fw_step_kernel : one thread per env; one launch == one agent step (30 Hz) == inner_per_step x
//                     substeps_per_inner physics substeps at 240 Hz, fused with the waypoint observation,
//                     reward, termination/truncation, SubprocVecEnv-style auto-reset and the flattened
//                     observation write.  Replaces FixedwingBaseEnv.step + Aviary.step
//                     (/root/reference/envs/fixedwing_envs/fixedwing_base_env.py:314-348) for all envs at once.
// K2 fw_reset_kernel: masked reset (fixedwing_base_env.py:193-257).
//
// Memory plan: state lives in six float4/int4 SoA planes (fw_device.cuh FwPlanes): every access is a
// 16-byte fully coalesced LDG.128/STG.128.  The [N,obs_dim] row-major observation the VecEnv contract
// demands is staged per warp in shared memory and written with ONE bulk async copy
// (cp.async.bulk.global.shared::cta -> SASS UBLKCP) of 32*obs_dim*4 contiguous bytes, instead of 32 strided
// row stores.  Aircraft/task constants arrive as a __grid_constant__ kernel parameter, i.e. in the constant
// bank.  On sm_100a an FP instruction cannot name a c[][] operand any more: each constant reaches the pipe through a
// uniform register filled by an LDCU (ncu: 720 LDCU among the 7,161 warp-instructions of an env-step before packing),
// so the constants of the hot substep are stored as 16-byte groups in order of use (FwDev::hot / rbk) and fetched with
// LDCU.128.  All threads use the same address, which is the case the constant cache is built for; shared-memory
// staging would cost an LDS per use instead.
#include "fw_device.cuh"
#include "fw_objlock.cuh"
#include "fw_pack.cuh"
#include "fw_kernels.h"

#include <cstdlib>
#include <cstring>

#define FW_BLOCK 64
// 8 resident blocks/SM x 64 threads x 128 registers = the whole 64K register file: 148 x 512 = 75,776 >= 65,536
// envs, so a 64K-env launch is a single wave
#ifndef FW_MIN_BLOCKS
#define FW_MIN_BLOCKS 8
#endif

__device__ __forceinline__ uint32_t fw_smem_addr(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Flush one warp's staged observation rows (32 x D floats, dense) to global memory.
// acc (optional): this block's slot of the observation-moment accumulators, double[2 * D] = column sums | sums of squares
// (VecNormalize's RunningMeanStd.update of the very observations being flushed, SURVEY section 8 row f1): lane c sums column
// c over the warp's rows out of shared memory -- a few instructions per env-step instead of a kernel that re-reads the batch.
template <int ROWS = 32>
__device__ __forceinline__ void fw_flush_obs(float* __restrict__ dst_base, const float* stage_warp, int D,
                                             int first_env, int n, int lane, bool bulk_ok, double* acc = nullptr) {
    const int rows = min(ROWS, n - first_env);
    float* dst = dst_base + (size_t)first_env * D;
    if (acc != nullptr) {
        __syncwarp();
        for (int c = lane; c < D; c += 32) {
            // in double: a column with a large mean and a small spread (altitude, airspeed) loses its variance to fp32 sums
            double sm = 0.0, sq = 0.0;
            for (int r = 0; r < rows; ++r) { const double x = (double)stage_warp[r * D + c]; sm += x; sq = fma(x, x, sq); }
            atomicAdd(acc + c, sm);
            atomicAdd(acc + D + c, sq);
        }
    }
    if (bulk_ok && rows == ROWS) {
        // generic-proxy writes -> async proxy, then one elected lane issues the TMA bulk store
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            uint32_t bytes = (uint32_t)ROWS * (uint32_t)D * 4u;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(dst), "r"(fw_smem_addr(stage_warp)), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        __syncwarp();
    } else {
        __syncwarp();
        for (int k = lane; k < rows * D; k += 32) dst[k] = stage_warp[k];
        __syncwarp();
    }
}

// One agent step of env i held in registers (FixedwingBaseEnv.step + SubprocVecEnv reset-on-done).
// Returns the reward; flag bits in `bits`; the observation (if TASK != 0) is left in `row`.
template <int TASK, bool STD, bool FIELD = false>
__device__ __forceinline__ float fw_env_step(const FwDev& p, const FwPlanes& pl, EnvState& e, int i,
                                             uint32_t gid, float a0, float a1, float a2, float a3, const float4& w0_in,
                                             const float4& w1_in, float& ep_ret, float* row, float* term_obs_row,
                                             uint32_t& bits, int& tidx_info) {
    float4 w0 = w0_in, w1 = w1_in;
    // checked on entry as well: the per-coordinate velocity clamp below turns a NaN velocity into -max_vel (fmaxf/fminf
    // return the non-NaN operand, in the oracle's C fmax/fmin too), which would launder a poisoned state
    const bool fault_in = !fw_state_finite(e);
    // FixedwingBaseEnv.step: reward reset once, thrust remapped to [0,1], setpoint latched
    float reward = -0.1f;
    bool term = false, trunc = false, col = false, oob = false, complete = false;
    float cmd[6];
    fw_map_setpoint(p, a0, a1, a2, a3 * 0.5f + 0.5f, cmd);
    float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
    bool have_noise = false;
    int obs_tidx = e.tidx;

    for (int it = 0; it < p.inner_per_step; ++it) {
        if (term || trunc) break;
        bool contact = false;                       // Aviary.step: contact_array &= False
        for (int s = 0; s < p.substeps_per_inner; ++s) {
            const int ps = e.physics_steps;
            float nz = 0.0f;
            if (p.noise_ratio > 0.0f) {
                if (!have_noise || (ps & 3) == 0) {
                    float nn[4];
                    fw_normals4(p, gid, e.episode, (uint32_t)ps >> 2, nn);
                    n0 = nn[0]; n1 = nn[1]; n2 = nn[2]; n3 = nn[3];
                    have_noise = true;
                }
                const int q = ps & 3;
                nz = q == 0 ? n0 : (q == 1 ? n1 : (q == 2 ? n2 : n3));
            }
            fw_substep_wind<STD, FIELD>(p, e, cmd, w0, w1, nz, contact);
        }
        // compute_state: WaypointHandler.distance_to_targets (old <- new, new <- |delta_0|)
        float old_dist = e.new_dist;
        obs_tidx = e.tidx;
        if (TASK >= 1 && e.tidx < p.num_targets) {
            float dx = pl.targets[(size_t)(e.tidx * 3 + 0) * p.n + i] - e.px;
            float dy = pl.targets[(size_t)(e.tidx * 3 + 1) * p.n + i] - e.py;
            float dz = pl.targets[(size_t)(e.tidx * 3 + 2) * p.n + i] - e.pz;
            e.new_dist = sqrtf(dx * dx + dy * dy + dz * dz);
        }
        // compute_base_term_trunc_reward
        if (e.step_count > p.max_steps) trunc = true;
        if (contact) { reward = -100.0f; col = true; term = true; }
        if (e.px * e.px + e.py * e.py + e.pz * e.pz > p.dome2) { reward = -100.0f; oob = true; term = true; }
        if (TASK == 1 && e.tidx < p.num_targets && !(p.early_return_on_crash && (col || oob))) {
            if (!p.sparse_reward) {
                reward += fmaxf(3.0f * (old_dist - e.new_dist), 0.0f);
                reward += 1.0f / e.new_dist;
            }
            if (e.new_dist < p.goal_reach) {
                reward = 100.0f;
                e.tidx += 1;                                  // advance_targets
                const bool all = e.tidx >= p.num_targets;
                if (p.complete_truncates && all) trunc = true;
            }
        }
    }
    e.step_count += 1;
    if (TASK == 1) complete = e.tidx >= p.num_targets;     // info["env_complete"] is sticky within an episode
    tidx_info = e.tidx;                                    // info["num_targets_reached"], before any auto-reset
    const bool fault = fault_in || !fw_state_finite(e);    // poisoned state: terminate without reward, count, reset
    if (fault) { term = true; trunc = false; col = false; oob = false; reward = 0.0f; }

    const bool done = term || trunc;
    if (TASK != 0 && row != nullptr) fw_write_obs(p, pl, e, i, obs_tidx, a0, a1, a2, a3, row);
    ep_ret += reward;
    if (done) {
        if (TASK != 0 && term_obs_row != nullptr && !fault)
            for (int k = 0; k < p.obs_dim; ++k) term_obs_row[k] = row[k];
        if (fault) atomicAdd(&pl.stats[8], 1.0);
        atomicAdd(&pl.stats[0], 1.0);
        atomicAdd(&pl.stats[1], (double)ep_ret);
        atomicAdd(&pl.stats[2], (double)e.step_count);
        atomicAdd(&pl.stats[3], (double)e.tidx);
        if (col) atomicAdd(&pl.stats[4], 1.0);
        if (oob) atomicAdd(&pl.stats[5], 1.0);
        if (complete) atomicAdd(&pl.stats[6], 1.0);
        // SubprocVecEnv worker: obs = env.reset()
        fw_reset_env<FIELD>(p, pl, e, i, gid, e.episode + 1u);
        if (p.wind_mode != 0) { w0 = pl.w0[i]; w1 = pl.w1[i]; }
        if (TASK != 0 && row != nullptr) fw_write_obs(p, pl, e, i, 0, 0.f, 0.f, 0.f, 0.f, row);
        if (fault && TASK != 0 && term_obs_row != nullptr)     // a finite stand-in: the first observation of the new episode
            for (int k = 0; k < p.obs_dim; ++k) term_obs_row[k] = row[k];
        ep_ret = 0.0f;
    }
    bits = (term ? 1u : 0u) | (trunc ? 2u : 0u) | (col ? 4u : 0u) | (oob ? 8u : 0u) | (complete ? 16u : 0u) | (fault ? 64u : 0u);
    return reward;
}

// FixedwingLowLevelEnv.step (fixedwing_lowlevel_env.py:97-141): six-channel surface/thrust command (Fixedwing mode -1),
// ONE Aviary.step (2 physics substeps) per env step, psi/h/V tracking reward, altitude-band termination, truncation at
// `max_steps` (>=); SubprocVecEnv reset-on-done.  No warm-up substeps and no ground-contact / dome test in this env.
template <bool STD, bool FIELD = false>
__device__ __forceinline__ float fw_env_step_lowlevel(const FwDev& p, const FwPlanes& pl, EnvState& e, int i, uint32_t gid,
                                                      const float a[6], const float4& w0_in, const float4& w1_in, float& ep_ret,
                                                      float* row, float* term_obs_row, uint32_t& bits) {
    float4 w0 = w0_in, w1 = w1_in;
    const bool fault_in = !fw_state_finite(e);           // see fw_env_step
    e.step_count += 1;                                   // self._episode_steps += 1
    float cmd[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) cmd[c] = a[c];             // mode -1: cmd = setpoint
    bool contact = false;
    float nn[4] = {0.f, 0.f, 0.f, 0.f};
    bool have_noise = false;
    for (int s = 0; s < p.substeps_per_inner; ++s) {
        const int ps = e.physics_steps;
        float nz = 0.0f;
        if (p.noise_ratio > 0.0f) {
            if (!have_noise || (ps & 3) == 0) { fw_normals4(p, gid, e.episode, (uint32_t)ps >> 2, nn); have_noise = true; }
            const int q = ps & 3;
            nz = q == 0 ? nn[0] : (q == 1 ? nn[1] : (q == 2 ? nn[2] : nn[3]));
        }
        fw_substep_wind<STD, FIELD>(p, e, cmd, w0, w1, nz, contact);
    }
    float yaw, speed, tref[3];
    fw_write_obs_lowlevel(pl, e, i, p.n, a, row, yaw, speed, tref);
    // _wrap_pi with Python's floored modulo
    float dpsi = tref[0] - yaw + FWD_PI;
    dpsi -= 2.0f * FWD_PI * floorf(dpsi * (0.5f / FWD_PI));
    dpsi -= FWD_PI;
    float reward = -(fabsf(dpsi) + fabsf(tref[1] - e.pz) + 0.5f * fabsf(tref[2] - speed)) + 0.1f;
    bool term = false, oob = false;
    if (e.pz < 1.0f || e.pz > 100.0f) { term = true; oob = true; reward -= 100.0f; }
    const bool trunc = e.step_count >= p.max_steps;
    const bool fault = fault_in || !fw_state_finite(e);
    if (fault) { term = true; oob = false; reward = 0.0f; }
    ep_ret += reward;
    if (term || trunc) {
        if (term_obs_row != nullptr && row != nullptr && !fault)
            for (int k = 0; k < p.obs_dim; ++k) term_obs_row[k] = row[k];
        if (fault) atomicAdd(&pl.stats[8], 1.0);
        atomicAdd(&pl.stats[0], 1.0);
        atomicAdd(&pl.stats[1], (double)ep_ret);
        atomicAdd(&pl.stats[2], (double)e.step_count);
        if (oob) atomicAdd(&pl.stats[5], 1.0);
        fw_reset_env<FIELD>(p, pl, e, i, gid, e.episode + 1u);
        if (row != nullptr) {
            const float z6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            fw_write_obs_lowlevel(pl, e, i, p.n, z6, row, yaw, speed, tref);
            if (fault && term_obs_row != nullptr)
                for (int k = 0; k < p.obs_dim; ++k) term_obs_row[k] = row[k];
        }
        ep_ret = 0.0f;
    }
    bits = (term ? 1u : 0u) | (trunc ? 2u : 0u) | (oob ? 8u : 0u) | (fault ? 64u : 0u);
    return reward;
}

// K1.  RANDOM_ACT: actions U(-1,1)^4 from Philox keyed (seed, global env id, episode, step_count); `spl` agent
// steps per launch with the state held in registers between them (the random-action sweep never needs the
// intermediate observations, so nothing but the final state goes back to HBM).
template <int TASK, bool RANDOM_ACT, bool STD, bool FIELD = false>
__global__ void __launch_bounds__(FW_BLOCK, FW_MIN_BLOCKS)
fw_step_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, const float4* __restrict__ act,
               float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ flg,
               float* __restrict__ term_obs, int spl, int bulk_ok) {
    extern __shared__ __align__(128) float stage[];
    // Programmatic dependent launch (bits 1-2 of `bulk_ok`): let the next launch of the chain start placing its blocks as
    // this one's finish -- the 54 % of the schedulers that hold 3 warps instead of 4 otherwise idle through the last quarter
    // of every launch -- and, when that next launch reads what this one writes (mode 1), make it wait for our completion
    // before it touches the planes.  Mode 2 = the chain steps a different env batch next (fw_rollout_random over handles).
    const int pdl = (bulk_ok >> 1) & 3;
    bulk_ok &= 1;
    if (pdl != 0) asm volatile("griddepcontrol.launch_dependents;");
    if (pdl == 1) asm volatile("griddepcontrol.wait;" ::: "memory");
    const int i = p.i_begin + blockIdx.x * FW_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int D = p.obs_dim;
    float* stage_warp = stage + (size_t)warp * 32 * D;
    float* row = (TASK != 0 && TASK != 3 && obs != nullptr) ? stage_warp + (size_t)lane * D : nullptr;

    if (i < p.i_end) {
        const uint32_t gid = p.env_id0 + (uint32_t)i;
        EnvState e;
        fw_load(pl, i, e);
        float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;
        if (p.wind_mode != 0) { w0 = pl.w0[i]; w1 = pl.w1[i]; }
        float ep_ret = pl.ep_ret[i];
        float reward = 0.f;
        uint32_t bits = 0u;
        int tidx_info = 0;
        if (TASK == 3) {
            float* orow = obs != nullptr ? stage_warp + (size_t)lane * D : nullptr;
            const int nst = RANDOM_ACT ? spl : 1;
            for (int st = 0; st < nst; ++st) {
                float a6[6];
                if (RANDOM_ACT) {
                    uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid, e.episode, (uint32_t)e.step_count, FWD_STREAM_ACTION);
                    uint4 r2 = fw_philox(p.seed_lo, p.seed_hi, gid, e.episode, (uint32_t)e.step_count | 0x40000000u, FWD_STREAM_ACTION);
                    a6[0] = 2.0f * fw_u01(r.x) - 1.0f; a6[1] = 2.0f * fw_u01(r.y) - 1.0f; a6[2] = 2.0f * fw_u01(r.z) - 1.0f;
                    a6[3] = 2.0f * fw_u01(r.w) - 1.0f; a6[4] = 2.0f * fw_u01(r2.x) - 1.0f; a6[5] = 2.0f * fw_u01(r2.y) - 1.0f;
                } else {
                    const float2* af = reinterpret_cast<const float2*>(act) + (size_t)i * 3;     // [N, 6] row-major
                    const float2 u0 = af[0], u1 = af[1], u2 = af[2];
                    a6[0] = u0.x; a6[1] = u0.y; a6[2] = u1.x; a6[3] = u1.y; a6[4] = u2.x; a6[5] = u2.y;
                }
                if (p.wind_mode != 0 && st > 0) { w0 = pl.w0[i]; w1 = pl.w1[i]; }
                reward = fw_env_step_lowlevel<STD, FIELD>(p, pl, e, i, gid, a6, w0, w1, ep_ret, st == nst - 1 ? orow : nullptr,
                                                   (!RANDOM_ACT && term_obs != nullptr && orow != nullptr) ? term_obs + (size_t)i * D : nullptr,
                                                   bits);
            }
        } else if (RANDOM_ACT) {
            for (int st = 0; st < spl; ++st) {
                uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid, e.episode, (uint32_t)e.step_count, FWD_STREAM_ACTION);
                float a0 = 2.0f * fw_u01(r.x) - 1.0f, a1 = 2.0f * fw_u01(r.y) - 1.0f;
                float a2 = 2.0f * fw_u01(r.z) - 1.0f, a3 = 2.0f * fw_u01(r.w) - 1.0f;
                if (p.wind_mode != 0 && st > 0) { w0 = pl.w0[i]; w1 = pl.w1[i]; }
                reward = fw_env_step<TASK, STD, FIELD>(p, pl, e, i, gid, a0, a1, a2, a3, w0, w1, ep_ret,
                                           st == spl - 1 ? row : nullptr, nullptr, bits, tidx_info);
            }
        } else {
            float4 a = act[i];
            reward = fw_env_step<TASK, STD, FIELD>(p, pl, e, i, gid, a.x, a.y, a.z, a.w, w0, w1, ep_ret, row,
                                       (TASK != 0 && term_obs != nullptr && row != nullptr) ? term_obs + (size_t)i * D : nullptr,
                                       bits, tidx_info);
        }
        pl.ep_ret[i] = ep_ret;
        fw_store(pl, i, e);
        if (rew != nullptr) rew[i] = reward;
        if (flg != nullptr) flg[i] = (uint8_t)bits;
        if (TASK == 1 && !RANDOM_ACT && pl.tidx_out != nullptr) pl.tidx_out[i] = (uint8_t)tidx_info;
    }
    if (TASK != 0 && obs != nullptr) {
        const int first_env = p.i_begin + blockIdx.x * FW_BLOCK + warp * 32;
        if (first_env < p.i_end)
            fw_flush_obs(obs, stage_warp, D, first_env, p.i_end, lane, bulk_ok != 0,
                         (!RANDOM_ACT && pl.obs_acc != nullptr) ? pl.obs_acc + (size_t)(blockIdx.x & (FW_OBS_ACC_SLOTS - 1)) * 2 * D : nullptr);
    }
}

// ================================================================== K1p: two environments per thread (fw_pack.cuh)
// The same agent step as fw_step_kernel for the standard aircraft layout, with the physics of a PAIR of envs (2t, 2t+1)
// carried in the two lanes of packed fp32x2 instructions.  Everything per-env that is not arithmetic (flags, rewards,
// waypoint bookkeeping, auto-reset) is the scalar code above, run once per lane.
#define FW2_THREADS 64
// 4 resident blocks/SM x 64 threads x 255 registers; 148 x 4 x 128 = 75,776 >= 65,536 envs: a 64K-env launch is one wave
#ifndef FW2_MIN_BLOCKS
#define FW2_MIN_BLOCKS 4
#endif
#define FW2_SNAP 20       // floats of physical state snapshotted when a lane finishes in the middle of an agent step

__device__ __forceinline__ void fw2_snapshot(float* snap, const EnvState2& e, int k) {
    snap[0] = e.px[k]; snap[1] = e.py[k]; snap[2] = e.pz[k];
    snap[3] = e.qx[k]; snap[4] = e.qy[k]; snap[5] = e.qz[k]; snap[6] = e.qw[k];
    snap[7] = e.vx[k]; snap[8] = e.vy[k]; snap[9] = e.vz[k];
    snap[10] = e.wx[k]; snap[11] = e.wy[k]; snap[12] = e.wz[k];
#pragma unroll
    for (int s = 0; s < FWD_NSURF; ++s) snap[13 + s] = e.act[s][k];
    snap[18] = e.thr[k]; snap[19] = __int_as_float(e.physics_steps[k]);
}
__device__ __forceinline__ void fw2_restore(const float* snap, EnvState2& e, int k) {
    fw_set(e.px.v, k, snap[0]); fw_set(e.py.v, k, snap[1]); fw_set(e.pz.v, k, snap[2]);
    fw_set(e.qx.v, k, snap[3]); fw_set(e.qy.v, k, snap[4]); fw_set(e.qz.v, k, snap[5]); fw_set(e.qw.v, k, snap[6]);
    fw_set(e.vx.v, k, snap[7]); fw_set(e.vy.v, k, snap[8]); fw_set(e.vz.v, k, snap[9]);
    fw_set(e.wx.v, k, snap[10]); fw_set(e.wy.v, k, snap[11]); fw_set(e.wz.v, k, snap[12]);
#pragma unroll
    for (int s = 0; s < FWD_NSURF; ++s) fw_set(e.act[s].v, k, snap[13 + s]);
    fw_set(e.thr.v, k, snap[18]); e.physics_steps[k] = __float_as_int(snap[19]);
}

// motor-noise draw of lane k for its physics step (the normals are redrawn every fourth step, as in fw_env_step)
__device__ __forceinline__ float fw2_noise(const FwDev& p, uint32_t gid, uint32_t episode, int ps, float (&nn)[4], bool& have) {
    if (!have || (ps & 3) == 0) { fw_normals4(p, gid, episode, (uint32_t)ps >> 2, nn); have = true; }
    const int q = ps & 3;
    return q == 0 ? nn[0] : (q == 1 ? nn[1] : (q == 2 ? nn[2] : nn[3]));
}

// FixedwingBaseEnv.step + SubprocVecEnv reset-on-done for the pair (tasks 0 and 1): fw_env_step, lane by lane
template <int TASK>
__device__ __forceinline__ void fw_env_step2(const FwDev& p, const FwPlanes& pl, EnvState2& e, int i0, uint32_t gid0,
                                             const float (&a)[2][4], float4 (&w0)[2], float4 (&w1)[2], float (&ep_ret)[2],
                                             float* const (&row)[2], float* const (&term_row)[2], float* snap,
                                             float (&reward)[2], uint32_t (&bits)[2], int (&tidx_info)[2], bool has1) {
    // lane y of the last thread of an odd batch mirrors lane x: it computes along and has no side effects
    const bool valid[2] = {true, has1};
    bool term[2] = {false, false}, trunc[2] = {false, false}, col[2] = {false, false}, oob[2] = {false, false};
    bool frozen[2] = {false, false}, fault_in[2], have_noise[2] = {false, false};
    float nn[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    int obs_tidx[2] = {e.tidx[0], e.tidx[1]};
    f2 cmd[6];
    {
        float c0[6], c1[6];
        fw_map_setpoint(p, a[0][0], a[0][1], a[0][2], a[0][3] * 0.5f + 0.5f, c0);
        fw_map_setpoint(p, a[1][0], a[1][1], a[1][2], a[1][3] * 0.5f + 0.5f, c1);
#pragma unroll
        for (int c = 0; c < 6; ++c) cmd[c] = f2(c0[c], c1[c]);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) { reward[k] = -0.1f; fault_in[k] = !fw_state_finite(fw_lane(e, k)); }

    for (int it = 0; it < p.inner_per_step; ++it) {
        const bool live[2] = {!(term[0] || trunc[0]), valid[1] && !(term[1] || trunc[1])};
        if (!live[0] && !live[1]) break;
        bool contact[2] = {false, false};
        for (int s = 0; s < p.substeps_per_inner; ++s) {
            f2 nz(0.0f), wx(0.0f), wy(0.0f), wz(0.0f);
            if (p.noise_ratio > 0.0f)
                nz = f2(fw2_noise(p, gid0, e.episode[0], e.physics_steps[0], nn[0], have_noise[0]),
                        fw2_noise(p, gid0 + 1u, e.episode[1], e.physics_steps[1], nn[1], have_noise[1]));
            if (p.wind_mode != 0) {
                float x0, y0, z0, x1, y1, z1;
                fw_wind(p, e.physics_steps[0], w0[0], w1[0], x0, y0, z0);
                fw_wind(p, e.physics_steps[1], w0[1], w1[1], x1, y1, z1);
                wx = f2(x0, x1); wy = f2(y0, y1); wz = f2(z0, z1);
            }
            fw_substep_p(p, e, cmd, wx, wy, wz, nz, contact);
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (!live[k]) continue;            // this lane broke out of the loop earlier (`if term or trunc: break`)
            const int i = i0 + k;
            const float px = e.px[k], py = e.py[k], pz = e.pz[k];
            // compute_state: WaypointHandler.distance_to_targets (old <- new, new <- |delta_0|)
            const float old_dist = e.new_dist[k];
            float new_dist = old_dist;
            obs_tidx[k] = e.tidx[k];
            if (TASK >= 1 && e.tidx[k] < p.num_targets) {
                const float dx = pl.targets[(size_t)(e.tidx[k] * 3 + 0) * p.n + i] - px;
                const float dy = pl.targets[(size_t)(e.tidx[k] * 3 + 1) * p.n + i] - py;
                const float dz = pl.targets[(size_t)(e.tidx[k] * 3 + 2) * p.n + i] - pz;
                new_dist = sqrtf(dx * dx + dy * dy + dz * dz);
                fw_set(e.new_dist.v, k, new_dist);
            }
            // compute_base_term_trunc_reward
            if (e.step_count[k] > p.max_steps) trunc[k] = true;
            if (contact[k]) { reward[k] = -100.0f; col[k] = true; term[k] = true; }
            if (px * px + py * py + pz * pz > p.dome2) { reward[k] = -100.0f; oob[k] = true; term[k] = true; }
            if (TASK == 1 && e.tidx[k] < p.num_targets && !(p.early_return_on_crash && (col[k] || oob[k]))) {
                if (!p.sparse_reward) {
                    reward[k] += fmaxf(3.0f * (old_dist - new_dist), 0.0f);
                    reward[k] += 1.0f / new_dist;
                }
                if (new_dist < p.goal_reach) {
                    reward[k] = 100.0f;
                    e.tidx[k] += 1;                                  // advance_targets
                    if (p.complete_truncates && e.tidx[k] >= p.num_targets) trunc[k] = true;
                }
            }
            // a lane that ends its step before the last inner iteration keeps riding in the packed arithmetic of its
            // neighbour: park the state its observation has to show
            if ((term[k] || trunc[k]) && it + 1 < p.inner_per_step) { fw2_snapshot(snap + k * FW2_SNAP, e, k); frozen[k] = true; }
        }
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        if (!valid[k]) continue;
        if (frozen[k]) fw2_restore(snap + k * FW2_SNAP, e, k);
        const int i = i0 + k;
        const uint32_t gid = gid0 + (uint32_t)k;
        e.step_count[k] += 1;
        bool complete = false;
        if (TASK == 1) complete = e.tidx[k] >= p.num_targets;
        tidx_info[k] = e.tidx[k];
        EnvState ek = fw_lane(e, k);
        const bool fault = fault_in[k] || !fw_state_finite(ek);
        if (fault) { term[k] = true; trunc[k] = false; col[k] = false; oob[k] = false; reward[k] = 0.0f; }
        const bool done = term[k] || trunc[k];
        if (TASK != 0 && row[k] != nullptr) fw_write_obs(p, pl, ek, i, obs_tidx[k], a[k][0], a[k][1], a[k][2], a[k][3], row[k]);
        ep_ret[k] += reward[k];
        if (done) {
            if (TASK != 0 && term_row[k] != nullptr && !fault)
                for (int c = 0; c < p.obs_dim; ++c) term_row[k][c] = row[k][c];
            if (fault) atomicAdd(&pl.stats[8], 1.0);
            atomicAdd(&pl.stats[0], 1.0);
            atomicAdd(&pl.stats[1], (double)ep_ret[k]);
            atomicAdd(&pl.stats[2], (double)ek.step_count);
            atomicAdd(&pl.stats[3], (double)ek.tidx);
            if (col[k]) atomicAdd(&pl.stats[4], 1.0);
            if (oob[k]) atomicAdd(&pl.stats[5], 1.0);
            if (complete) atomicAdd(&pl.stats[6], 1.0);
            fw_reset_env(p, pl, ek, i, gid, ek.episode + 1u);         // SubprocVecEnv worker: obs = env.reset()
            if (p.wind_mode != 0) { w0[k] = pl.w0[i]; w1[k] = pl.w1[i]; }
            if (TASK != 0 && row[k] != nullptr) fw_write_obs(p, pl, ek, i, 0, 0.f, 0.f, 0.f, 0.f, row[k]);
            if (fault && TASK != 0 && term_row[k] != nullptr)
                for (int c = 0; c < p.obs_dim; ++c) term_row[k][c] = row[k][c];
            ep_ret[k] = 0.0f;
            fw_set_lane(e, k, ek);
        }
        bits[k] = (term[k] ? 1u : 0u) | (trunc[k] ? 2u : 0u) | (col[k] ? 4u : 0u) | (oob[k] ? 8u : 0u) | (complete ? 16u : 0u) |
                  (fault ? 64u : 0u);
    }
}

// FixedwingLowLevelEnv.step for the pair (task 3): fw_env_step_lowlevel, lane by lane
__device__ __forceinline__ void fw_env_step2_lowlevel(const FwDev& p, const FwPlanes& pl, EnvState2& e, int i0, uint32_t gid0,
                                                      const float (&a)[2][6], float4 (&w0)[2], float4 (&w1)[2],
                                                      float (&ep_ret)[2], float* const (&row)[2], float* const (&term_row)[2],
                                                      float (&reward)[2], uint32_t (&bits)[2], bool has1) {
    bool fault_in[2], have_noise[2] = {false, false};
    float nn[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    f2 cmd[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) cmd[c] = f2(a[0][c], a[1][c]);
#pragma unroll
    for (int k = 0; k < 2; ++k) { fault_in[k] = !fw_state_finite(fw_lane(e, k)); e.step_count[k] += 1; }
    bool contact[2] = {false, false};
    for (int s = 0; s < p.substeps_per_inner; ++s) {
        f2 nz(0.0f), wx(0.0f), wy(0.0f), wz(0.0f);
        if (p.noise_ratio > 0.0f)
            nz = f2(fw2_noise(p, gid0, e.episode[0], e.physics_steps[0], nn[0], have_noise[0]),
                    fw2_noise(p, gid0 + 1u, e.episode[1], e.physics_steps[1], nn[1], have_noise[1]));
        if (p.wind_mode != 0) {
            float x0, y0, z0, x1, y1, z1;
            fw_wind(p, e.physics_steps[0], w0[0], w1[0], x0, y0, z0);
            fw_wind(p, e.physics_steps[1], w0[1], w1[1], x1, y1, z1);
            wx = f2(x0, x1); wy = f2(y0, y1); wz = f2(z0, z1);
        }
        fw_substep_p(p, e, cmd, wx, wy, wz, nz, contact);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        if (k == 1 && !has1) continue;
        const int i = i0 + k;
        EnvState ek = fw_lane(e, k);
        float yaw, speed, tref[3];
        fw_write_obs_lowlevel(pl, ek, i, p.n, a[k], row[k], yaw, speed, tref);
        float dpsi = tref[0] - yaw + FWD_PI;
        dpsi -= 2.0f * FWD_PI * floorf(dpsi * (0.5f / FWD_PI));
        dpsi -= FWD_PI;
        reward[k] = -(fabsf(dpsi) + fabsf(tref[1] - ek.pz) + 0.5f * fabsf(tref[2] - speed)) + 0.1f;
        bool term = false, oob = false;
        if (ek.pz < 1.0f || ek.pz > 100.0f) { term = true; oob = true; reward[k] -= 100.0f; }
        const bool trunc = ek.step_count >= p.max_steps;
        const bool fault = fault_in[k] || !fw_state_finite(ek);
        if (fault) { term = true; oob = false; reward[k] = 0.0f; }
        ep_ret[k] += reward[k];
        if (term || trunc) {
            if (term_row[k] != nullptr && row[k] != nullptr && !fault)
                for (int c = 0; c < p.obs_dim; ++c) term_row[k][c] = row[k][c];
            if (fault) atomicAdd(&pl.stats[8], 1.0);
            atomicAdd(&pl.stats[0], 1.0);
            atomicAdd(&pl.stats[1], (double)ep_ret[k]);
            atomicAdd(&pl.stats[2], (double)ek.step_count);
            if (oob) atomicAdd(&pl.stats[5], 1.0);
            fw_reset_env(p, pl, ek, i, gid0 + (uint32_t)k, ek.episode + 1u);
            if (p.wind_mode != 0) { w0[k] = pl.w0[i]; w1[k] = pl.w1[i]; }
            if (row[k] != nullptr) {
                const float z6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                fw_write_obs_lowlevel(pl, ek, i, p.n, z6, row[k], yaw, speed, tref);
                if (fault && term_row[k] != nullptr)
                    for (int c = 0; c < p.obs_dim; ++c) term_row[k][c] = row[k][c];
            }
            ep_ret[k] = 0.0f;
            fw_set_lane(e, k, ek);
        }
        bits[k] = (term ? 1u : 0u) | (trunc ? 2u : 0u) | (oob ? 8u : 0u) | (fault ? 64u : 0u);
    }
}

// smem: [obs staging: 128 rows x D] [snapshots: 64 threads x 2 x FW2_SNAP]
template <int TASK, bool RANDOM_ACT>
__global__ void __launch_bounds__(FW2_THREADS, FW2_MIN_BLOCKS)
fw_step2_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, const float4* __restrict__ act,
                float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ flg,
                float* __restrict__ term_obs, int spl, int bulk_ok) {
    extern __shared__ __align__(128) float stage[];
    const int t = blockIdx.x * FW2_THREADS + threadIdx.x;
    const int i0 = p.i_begin + 2 * t;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int D = p.obs_dim;
    float* stage_warp = stage + (size_t)warp * 64 * D;
    float* snap = stage + (size_t)(FW2_THREADS * 2) * (D > 0 ? D : 1) + (size_t)threadIdx.x * 2 * FW2_SNAP;
    const bool want_obs = TASK != 0 && obs != nullptr;

    if (i0 < p.i_end) {
        const bool has1 = i0 + 1 < p.i_end;
        const uint32_t gid0 = p.env_id0 + (uint32_t)i0;
        EnvState2 e;
        fw_load2(pl, i0, p.i_end, e);
        const int i1 = has1 ? i0 + 1 : i0;
        float4 w0[2], w1[2];
        w0[0] = w0[1] = w1[0] = w1[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.wind_mode != 0) { w0[0] = pl.w0[i0]; w1[0] = pl.w1[i0]; w0[1] = pl.w0[i1]; w1[1] = pl.w1[i1]; }
        float ep_ret[2] = {pl.ep_ret[i0], pl.ep_ret[i1]};
        float reward[2] = {0.f, 0.f};
        uint32_t bits[2] = {0u, 0u};
        int tidx_info[2] = {0, 0};
        float* const row[2] = {want_obs ? stage_warp + (size_t)(2 * lane) * D : nullptr,
                               want_obs ? stage_warp + (size_t)(2 * lane + 1) * D : nullptr};
        const bool want_term = !RANDOM_ACT && want_obs && term_obs != nullptr;
        float* const term_row[2] = {want_term ? term_obs + (size_t)i0 * D : nullptr, (want_term && has1) ? term_obs + (size_t)i1 * D : nullptr};
        float* const no_row[2] = {nullptr, nullptr};
        const int nst = RANDOM_ACT ? spl : 1;
        for (int st = 0; st < nst; ++st) {
            if (p.wind_mode != 0 && st > 0) { w0[0] = pl.w0[i0]; w1[0] = pl.w1[i0]; w0[1] = pl.w0[i1]; w1[1] = pl.w1[i1]; }
            const bool last = st == nst - 1;
            if (TASK == 3) {
                float a6[2][6];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    if (RANDOM_ACT) {
                        const uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid0 + k, e.episode[k], (uint32_t)e.step_count[k], FWD_STREAM_ACTION);
                        const uint4 r2 = fw_philox(p.seed_lo, p.seed_hi, gid0 + k, e.episode[k], (uint32_t)e.step_count[k] | 0x40000000u, FWD_STREAM_ACTION);
                        a6[k][0] = 2.0f * fw_u01(r.x) - 1.0f; a6[k][1] = 2.0f * fw_u01(r.y) - 1.0f; a6[k][2] = 2.0f * fw_u01(r.z) - 1.0f;
                        a6[k][3] = 2.0f * fw_u01(r.w) - 1.0f; a6[k][4] = 2.0f * fw_u01(r2.x) - 1.0f; a6[k][5] = 2.0f * fw_u01(r2.y) - 1.0f;
                    } else {
                        const float2* af = reinterpret_cast<const float2*>(act) + (size_t)(k ? i1 : i0) * 3;     // [N, 6] row-major
                        const float2 u0 = af[0], u1 = af[1], u2 = af[2];
                        a6[k][0] = u0.x; a6[k][1] = u0.y; a6[k][2] = u1.x; a6[k][3] = u1.y; a6[k][4] = u2.x; a6[k][5] = u2.y;
                    }
                }
                if (last) fw_env_step2_lowlevel(p, pl, e, i0, gid0, a6, w0, w1, ep_ret, row, term_row, reward, bits, has1);
                else fw_env_step2_lowlevel(p, pl, e, i0, gid0, a6, w0, w1, ep_ret, no_row, no_row, reward, bits, has1);
            } else {
                float a4[2][4];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    if (RANDOM_ACT) {
                        const uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid0 + k, e.episode[k], (uint32_t)e.step_count[k], FWD_STREAM_ACTION);
                        a4[k][0] = 2.0f * fw_u01(r.x) - 1.0f; a4[k][1] = 2.0f * fw_u01(r.y) - 1.0f;
                        a4[k][2] = 2.0f * fw_u01(r.z) - 1.0f; a4[k][3] = 2.0f * fw_u01(r.w) - 1.0f;
                    } else {
                        const float4 v = act[k ? i1 : i0];
                        a4[k][0] = v.x; a4[k][1] = v.y; a4[k][2] = v.z; a4[k][3] = v.w;
                    }
                }
                if (last) fw_env_step2<TASK>(p, pl, e, i0, gid0, a4, w0, w1, ep_ret, row, term_row, snap, reward, bits, tidx_info, has1);
                else fw_env_step2<TASK>(p, pl, e, i0, gid0, a4, w0, w1, ep_ret, no_row, no_row, snap, reward, bits, tidx_info, has1);
            }
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (k == 1 && !has1) break;
            const int i = i0 + k;
            pl.ep_ret[i] = ep_ret[k];
            fw_store(pl, i, fw_lane(e, k));
            if (rew != nullptr) rew[i] = reward[k];
            if (flg != nullptr) flg[i] = (uint8_t)bits[k];
            if (TASK == 1 && !RANDOM_ACT && pl.tidx_out != nullptr) pl.tidx_out[i] = (uint8_t)tidx_info[k];
        }
    }
    if (want_obs) {
        const int first_env = p.i_begin + (blockIdx.x * FW2_THREADS + warp * 32) * 2;
        if (first_env < p.i_end)
            fw_flush_obs<64>(obs, stage_warp, D, first_env, p.i_end, lane, bulk_ok != 0,
                             (!RANDOM_ACT && pl.obs_acc != nullptr) ? pl.obs_acc + (size_t)(blockIdx.x & (FW_OBS_ACC_SLOTS - 1)) * 2 * D : nullptr);
    }
}

template <bool FIELD = false>
__global__ void __launch_bounds__(FW_BLOCK)
fw_reset_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, const uint8_t* __restrict__ mask,
                float* __restrict__ obs, int bulk_ok, int emit_only) {
    extern __shared__ __align__(128) float stage[];
    const int i = blockIdx.x * FW_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int D = p.obs_dim;
    float* stage_warp = stage + (size_t)warp * 32 * D;
    float* row = stage_warp + (size_t)lane * D;
    if (i < p.n) {
        EnvState e;
        fw_load(pl, i, e);
        const bool sel = !emit_only && (mask == nullptr || mask[i] != 0);
        if (sel) {
            fw_reset_env<FIELD>(p, pl, e, i, p.env_id0 + (uint32_t)i, e.episode + 1u);
            pl.ep_ret[i] = 0.0f;
            fw_store(pl, i, e);
        }
        // unselected envs re-emit their current observation (last action unknown -> zeros)
        if (p.task == 3) {
            const float z6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            float yaw, speed, tref[3];
            fw_write_obs_lowlevel(pl, e, i, p.n, z6, row, yaw, speed, tref);
        } else if (p.task != 0) fw_write_obs(p, pl, e, i, e.tidx, 0.f, 0.f, 0.f, 0.f, row);
    }
    if (p.task != 0 && obs != nullptr) {
        const int first_env = blockIdx.x * FW_BLOCK + warp * 32;
        if (first_env < p.n) fw_flush_obs(obs, stage_warp, D, first_env, p.n, lane, bulk_ok != 0);
    }
}

// ================================================================== Waypoint + ObjLock task (warp-converged kernels)
// The camera frame is produced warp-cooperatively (fw_objlock.cuh: ol_capture_warp), so every lane of a warp has to
// arrive at each capture point: these kernels replace `break` / early exits by per-lane predicates.

// reset of the lanes with `doing` set: begin_reset, waypoints, duck/obstacles, warm-up with the camera frame PyFlyt
// captures at physics step 12 of it, then the compute_state of end_reset (fixedwing_waypoint_objlock_env.py:170-195)
template <int TASK, bool FIELD = false>
__device__ __forceinline__ void ol_reset_lanes(const FwDev& p, const FwPlanes& pl, bool doing, EnvState& e, OlState& ol,
                                               float* so, float* depth_row, float* hs, int i, uint32_t gid, uint32_t episode,
                                               int tid) {
    float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;
    if (doing) {
        fw_reset_begin<FIELD>(p, pl, e, i, gid, episode, w0, w1);
        if (TASK == 2) {
            fw_sample_targets(p, pl, i, gid, episode);
            ol_reset(p, pl, ol, i, gid, episode, so, tid, FW_BLOCK);
        } else {
            ol_reset_duck(p, pl, ol, i, gid, episode, so, hs, tid, FW_BLOCK);
        }
    }
    __syncwarp();
    int dn = 0;
    while (dn < p.warmup_substeps) {                       // trip count depends on the config only: warp-uniform
        int next = p.warmup_substeps;
        if (p.cam_interval > 0) next = min(next, (dn / p.cam_interval + 1) * p.cam_interval);
        if (doing) fw_warm<FIELD>(p, e, w0, w1, next - dn, false);
        dn = next;
        const bool need = doing && p.cam_interval > 0 && dn % p.cam_interval == 0 && dn % p.substeps_per_inner == 0;
        ol_capture_warp(p, need, e, ol, so, tid, FW_BLOCK, depth_row);
    }
    if (doing) {
        fw_reset_finish(p, pl, e, i);
        ol_vision_and_phase(p, ol, TASK == 2 && e.tidx >= p.num_targets);
        if (TASK == 4) ol_hist_push(p, ol, hs, tid, FW_BLOCK);
    }
}

// ---- pre-warmed spare episodes (see FwPlanes)
#define OL_REFILL_PER_WARP 8      // requests served per warp pass: the camera serves a warp's frames one after the other, so
                                  // a full warp would spend 32 frame times on the warm-up frame alone (140 us measured)

__device__ __forceinline__ float4 sp_ld(const float4* p) { return __ldcg(p); }     // L2: written by another block of a
__device__ __forceinline__ int4 sp_ld(const int4* p) { return __ldcg(p); }         // (possibly concurrent) launch
__device__ __forceinline__ float sp_ld(const float* p) { return __ldcg(p); }

// Try to start episode `want` of env i from its spare.  On success the live per-episode planes (wind, targets, obstacle
// table) and the shared-memory copies are overwritten from the spare and the tag is cleared.
template <int TASK>
__device__ __forceinline__ bool ol_take_spare(const FwDev& p, const FwPlanes& pl, EnvState& e, OlState& ol, float* so, float* hs,
                                              int i, uint32_t want, int tid, float4& w0, float4& w1) {
    const int tag = *reinterpret_cast<volatile const int*>(&pl.sp_s5[i].z);
    if ((uint32_t)tag != want) return false;
    __threadfence();                                   // acquire: the planes were written before the tag
    const float4 a = sp_ld(&pl.sp_s0[i]), b = sp_ld(&pl.sp_s1[i]), c = sp_ld(&pl.sp_s2[i]), d = sp_ld(&pl.sp_s3[i]), f = sp_ld(&pl.sp_s4[i]);
    const int4 g = sp_ld(&pl.sp_s5[i]);
    const float4 dk = sp_ld(&pl.sp_dk[i]), v0 = sp_ld(&pl.sp_v0[i]), v1 = sp_ld(&pl.sp_v1[i]), v2 = sp_ld(&pl.sp_v2[i]);
    const int4 v3 = sp_ld(&pl.sp_v3[i]);
    if (p.wind_mode != 0) { w0 = sp_ld(&pl.sp_w0[i]); w1 = sp_ld(&pl.sp_w1[i]); pl.w0[i] = w0; pl.w1[i] = w1; }
    e.px = a.x; e.py = a.y; e.pz = a.z; e.thr = a.w;
    e.qx = b.x; e.qy = b.y; e.qz = b.z; e.qw = b.w;
    e.vx = c.x; e.vy = c.y; e.vz = c.z; e.act[0] = c.w;
    e.wx = d.x; e.wy = d.y; e.wz = d.z; e.act[1] = d.w;
    e.act[2] = f.x; e.act[3] = f.y; e.act[4] = f.z; e.new_dist = f.w;
    e.step_count = g.x; e.physics_steps = g.y; e.episode = want; e.tidx = g.w;
    ol.dkx = dk.x; ol.dky = dk.y; ol.dkz = dk.z;
    ol.last_cx = v0.x; ol.last_cy = v0.y; ol.last_area = v0.z; ol.last_depth = v0.w;
    ol.f_cx = v1.x; ol.f_cy = v1.y; ol.f_area = v1.z; ol.f_depth = v1.w;
    ol.f_dl = v2.x; ol.f_dc = v2.y; ol.f_dr = v2.z; ol.prev_est = v2.w;
    ol.duck_phase = v3.x & 1; ol.has_prev = (v3.x >> 1) & 1; ol.post_wp = (v3.x >> 2) & 1; ol.cam_valid = (v3.x >> 3) & 1;
    ol.f_visible = (v3.x >> 4) & 1; ol.n_obst = (v3.x >> 8) & 0xff;
    ol.seen = v3.y; ol.lock = v3.z; ol.since = v3.w;
    ol.vis_dl = ol.vis_dc = ol.vis_dr = 0.0f; ol.vis_flag = 0.0f;
    // the per-episode tables: loads in batches of eight before their stores, so that one lane's copy costs a few L2 round
    // trips instead of one per element
    const size_t n = (size_t)p.n;
    const int nt = p.num_targets * 3;
    for (int t0 = 0; t0 < nt; t0 += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (t0 + u < nt) ? sp_ld(&pl.sp_targets[(size_t)(t0 + u) * n + i]) : 0.0f;
#pragma unroll
        for (int u = 0; u < 8; ++u) if (t0 + u < nt) pl.targets[(size_t)(t0 + u) * n + i] = v[u];
    }
    const int no = ol.n_obst * 3;
    for (int t0 = 0; t0 < no; t0 += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (t0 + u < no) ? sp_ld(&pl.sp_obst[(size_t)(t0 + u) * n + i]) : 0.0f;
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (t0 + u < no) { pl.obst[(size_t)(t0 + u) * n + i] = v[u]; so[(t0 + u) * FW_BLOCK + tid] = v[u]; }
    }
    if (TASK == 4) {
        for (int t0 = 0; t0 < p.hist_slots; t0 += 8) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (t0 + u < p.hist_slots) ? sp_ld(&pl.sp_hist[(size_t)(t0 + u) * n + i]) : 0.0f;
#pragma unroll
            for (int u = 0; u < 8; ++u) if (t0 + u < p.hist_slots) OL_H(hs, t0 + u, tid, FW_BLOCK) = v[u];
        }
    }
    pl.sp_s5[i].z = -1;                                 // consumed
    return true;
}

// ask for the spare of episode `episode` of env i to be prepared
__device__ __forceinline__ void ol_request_spare(const FwPlanes& pl, int i, uint32_t episode) {
    if (pl.refill_list == nullptr) return;
    const int idx = atomicAdd(pl.refill_count, 1);
    if (idx < pl.refill_cap) pl.refill_list[idx] = make_int2(i, (int)episode);
}

// the FwPlanes whose primary pointers are the spare set: the code of the in-step reset then writes there
__device__ __forceinline__ FwPlanes ol_spare_view(const FwPlanes& pl) {
    FwPlanes v = pl;
    v.s0 = pl.sp_s0; v.s1 = pl.sp_s1; v.s2 = pl.sp_s2; v.s3 = pl.sp_s3; v.s4 = pl.sp_s4; v.s5 = pl.sp_s5;
    v.w0 = pl.sp_w0; v.w1 = pl.sp_w1; v.targets = pl.sp_targets;
    v.dk = pl.sp_dk; v.v0 = pl.sp_v0; v.v1 = pl.sp_v1; v.v2 = pl.sp_v2; v.v3 = pl.sp_v3; v.obst = pl.sp_obst; v.hist = pl.sp_hist;
    return v;
}

// flattened observation of either ObjLock task into `row`
template <int TASK>
__device__ __forceinline__ void ol_write_obs(const FwDev& p, const FwPlanes& pl, const EnvState& e, const OlState& ol,
                                             const float* hs, int i, int obs_tidx, float a0, float a1, float a2, float a3,
                                             float* row, int tid) {
    if (TASK == 2) fw_write_obs(p, pl, e, i, obs_tidx, a0, a1, a2, a3, row, true, ol.dkx, ol.dky, ol.dkz);
    else {
        fw_write_obs(p, pl, e, i, 0, a0, a1, a2, a3, row);            // context_len == 0: the attitude block only
        ol_write_obs_duck_tail(p, e, ol, hs, tid, FW_BLOCK, row + ((p.angle_repr == 0 ? 12 : 13) + 10));
    }
}

// Episode end of the lanes with `done` set (all 32 lanes call): terminal observation, episode statistics, then the
// SubprocVecEnv worker's obs = env.reset().  The next episode normally waits ready-made in the env's spare planes; lanes
// without a valid spare (first episodes after an injected state, two finishes in quick succession, FWSIM_SPARE=0) run the
// reset inline.  (Inlined: out-of-line versions -- `e` / `ol` passed through local copies, or the refill as a role of this
// kernel's leading blocks -- measured 3-15 % slower: the step kernel is sensitive to its stack frame, profiles/r2_objlock.md.)
template <int TASK, bool FIELD = false>
__device__ __forceinline__ void ol_finish_episode(const FwDev& p, const FwPlanes& pl, bool done, uint32_t info, EnvState& e,
                                                      OlState& ol, float4& w0, float4& w1, float& ep_ret, float* so,
                                                      float* depth_row, float* hs, int i, uint32_t gid, float* row,
                                                      float* term_obs_row) {
    const int tid = threadIdx.x;
    const bool fault = info & 1u;
    if (done) {
        if (term_obs_row != nullptr && !fault)
            for (int k = 0; k < p.obs_dim; ++k) term_obs_row[k] = row[k];
        if (fault) atomicAdd(&pl.stats[8], 1.0);
        atomicAdd(&pl.stats[0], 1.0);
        atomicAdd(&pl.stats[1], (double)ep_ret);
        atomicAdd(&pl.stats[2], (double)e.step_count);
        atomicAdd(&pl.stats[3], (double)e.tidx);
        if (info & 2u) atomicAdd(&pl.stats[4], 1.0);
        if (info & 4u) atomicAdd(&pl.stats[5], 1.0);
        if (info & 8u) atomicAdd(&pl.stats[6], 1.0);
        if (info & 16u) atomicAdd(&pl.stats[7], 1.0);
    }
    bool inline_reset = done;
    if (done && pl.sp_s5 != nullptr) {
        const uint32_t want = e.episode + 1u;
        inline_reset = !ol_take_spare<TASK>(p, pl, e, ol, so, hs, i, want, tid, w0, w1);
        ol_request_spare(pl, i, want + 1u);
        atomicAdd(&pl.stats[inline_reset ? 10 : 9], 1.0);      // fw_spare_stats: resets served inline / from a spare
    }
    if (__any_sync(0xffffffffu, inline_reset))
        ol_reset_lanes<TASK, FIELD>(p, pl, inline_reset, e, ol, so, depth_row, hs, i, gid, e.episode + 1u, tid);
    if (done) {
        if (p.wind_mode != 0 && inline_reset) { w0 = pl.w0[i]; w1 = pl.w1[i]; }
        if (row != nullptr) ol_write_obs<TASK>(p, pl, e, ol, hs, i, 0, 0.f, 0.f, 0.f, 0.f, row, tid);
        if (fault && term_obs_row != nullptr && row != nullptr)
            for (int k = 0; k < p.obs_dim; ++k) term_obs_row[k] = row[k];
        ep_ret = 0.0f;
    }
}

// one agent step for the whole warp; `active` = lane owns an env
template <int TASK, bool STD, bool FIELD = false>
__device__ __forceinline__ float fw_env_step_objlock(const FwDev& p, const FwPlanes& pl, bool active, EnvState& e, OlState& ol,
                                                     float* so, float* depth_row, float* hs, int i, uint32_t gid, float a0, float a1,
                                                     float a2, float a3, float4& w0, float4& w1, float& ep_ret, float* row,
                                                     float* term_obs_row, uint32_t& bits, int& tidx_info) {
    const int tid = threadIdx.x;
    const bool fault_in = active && !fw_state_finite(e);   // see fw_env_step
    float reward = -0.1f;
    bool term = false, trunc = false, col = false, oob = false, complete = false, strike = false;
    float cmd[6];
    fw_map_setpoint(p, a0, a1, a2, a3 * 0.5f + 0.5f, cmd);
    float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
    bool have_noise = false;
    int obs_tidx = e.tidx;
    bool duck_near = false;
    const uint32_t cand = active ? ol_contact_candidates(p, e, ol, so, tid, FW_BLOCK, duck_near) : 0u;

    for (int it = 0; it < p.inner_per_step; ++it) {
        const bool run = active && !(term || trunc);        // FixedwingBaseEnv.step: `if termination or truncation: break`
        bool contact = false;
        if (run) {
            // one copy of the substep in the loop body: this kernel's inner iteration (substeps + camera + rewards) is
            // instruction-cache bound (ncu: no_instruction ~0.9 stalls per issue), unrolling the pair of substeps costs 10 KB
#pragma unroll 1
            for (int s = 0; s < p.substeps_per_inner; ++s) {
                const int ps = e.physics_steps;
                float nz = 0.0f;
                if (p.noise_ratio > 0.0f) {
                    if (!have_noise || (ps & 3) == 0) {
                        float nn[4];
                        fw_normals4(p, gid, e.episode, (uint32_t)ps >> 2, nn);
                        n0 = nn[0]; n1 = nn[1]; n2 = nn[2]; n3 = nn[3];
                        have_noise = true;
                    }
                    const int q = ps & 3;
                    nz = q == 0 ? n0 : (q == 1 ? n1 : (q == 2 ? n2 : n3));
                }
                if (FIELD) {
                    FwFieldT ft;
                    fw_field_time(p, ps, w0, ft);
                    contact = contact || ol_contact(p, e, ol, so, tid, FW_BLOCK, cand, duck_near);    // pose
                    fw_substep<STD, true>(p, e, cmd, 0.0f, 0.0f, 0.0f, nz, contact, ft);
                } else {
                    float wx, wy, wz;
                    fw_wind(p, ps, w0, w1, wx, wy, wz);
                    contact = contact || ol_contact(p, e, ol, so, tid, FW_BLOCK, cand, duck_near);    // pose
                    fw_substep<STD>(p, e, cmd, wx, wy, wz, nz, contact);
                }
            }
        }
        // drone.update_last(): camera frame every cam_interval physics steps
        const bool need = run && p.cam_interval > 0 && (e.physics_steps % p.cam_interval) == 0;
        ol_capture_warp(p, need, e, ol, so, tid, FW_BLOCK, depth_row);
        if (run) {
            // compute_state
            float old_dist = e.new_dist;
            obs_tidx = e.tidx;
            if (TASK == 2 && e.tidx < p.num_targets) {
                float dx = pl.targets[(size_t)(e.tidx * 3 + 0) * p.n + i] - e.px;
                float dy = pl.targets[(size_t)(e.tidx * 3 + 1) * p.n + i] - e.py;
                float dz = pl.targets[(size_t)(e.tidx * 3 + 2) * p.n + i] - e.pz;
                e.new_dist = sqrtf(dx * dx + dy * dy + dz * dz);
            }
            ol_vision_and_phase(p, ol, TASK == 2 && e.tidx >= p.num_targets);
            if (TASK == 4) ol_hist_push(p, ol, hs, tid, FW_BLOCK);
            // compute_base_term_trunc_reward
            if (e.step_count > p.max_steps) trunc = true;
            if (contact) { reward = -100.0f; col = true; term = true; }
            if (e.px * e.px + e.py * e.py + e.pz * e.pz > p.dome2) { reward = -100.0f; oob = true; term = true; }
            if (!(col || oob)) {                       // early return on crash (objlock_env.py:282-283)
                if (TASK == 4) {
                    ol_duck_reward(p, e, ol, reward, term, complete, strike);
                } else if (e.tidx < p.num_targets) {
                    if (!p.sparse_reward) {
                        reward += fmaxf(3.0f * (old_dist - e.new_dist), 0.0f);
                        reward += 1.0f / e.new_dist;
                    }
                    if (e.new_dist < p.goal_reach) {
                        reward = 100.0f;
                        e.tidx += 1;
                        if (e.tidx >= p.num_targets) { term = false; trunc = false; }    // keep flying into the duck phase
                    }
                    reward -= ol_obstacle_penalty(p, ol, false);
                } else {
                    term = false;
                    reward -= ol_obstacle_penalty(p, ol, true);
                    if (ol.duck_phase) {
                        if (!p.sparse_reward && ol.last_depth > 0.0f) reward += 1.0f / fmaxf(ol.last_depth, 2.0f);
                        if (ol.last_cx > 0.0f) {
                            float ddx = ol.last_cx - 0.5f, ddy = ol.last_cy - 0.5f;
                            if (sqrtf(ddx * ddx + ddy * ddy) < 0.35f) { ol.lock += 1; reward += p.lock_step_reward; }
                            else ol.lock = 0;
                        } else ol.lock = 0;
                        const float est = ol.last_depth;
                        if (ol.has_prev && est > 0.0f) {
                            float diff = ol.prev_est - est;
                            if (diff > 0.0f) reward += diff * p.approach_scale;
                        }
                        ol.prev_est = est; ol.has_prev = 1;
                        if (ol.lock >= p.lock_hold && est > 0.0f && est <= p.strike_dist) {
                            term = true; reward += p.strike_reward; complete = true; strike = true;
                        }
                    }
                }
            }
        }
    }
    if (active) e.step_count += 1;
    tidx_info = e.tidx;                                    // info["num_targets_reached"], before any auto-reset
    const bool fault = fault_in || (active && !fw_state_finite(e));   // poisoned state: terminate without reward, count, reset
    if (fault) { term = true; trunc = false; col = false; oob = false; complete = false; strike = false; reward = 0.0f; }
    const bool done = active && (term || trunc);
    if (active && row != nullptr) ol_write_obs<TASK>(p, pl, e, ol, hs, i, obs_tidx, a0, a1, a2, a3, row, tid);
    if (active) ep_ret += reward;
    if (__any_sync(0xffffffffu, done)) {
        const uint32_t info = (fault ? 1u : 0u) | (col ? 2u : 0u) | (oob ? 4u : 0u) | (complete ? 8u : 0u) | (strike ? 16u : 0u);
        ol_finish_episode<TASK, FIELD>(p, pl, done, info, e, ol, w0, w1, ep_ret, so, depth_row, hs, i, gid, row, term_obs_row);
    }
    bits = (term ? 1u : 0u) | (trunc ? 2u : 0u) | (col ? 4u : 0u) | (oob ? 8u : 0u) | (complete ? 16u : 0u) | (strike ? 32u : 0u) |
           (fault ? 64u : 0u);
    return reward;
}

// smem: [obs staging (FW_BLOCK x D)] [obstacle table (num_obstacles x 3 x FW_BLOCK)] [depth rows (warps x cam_res)]
//       [task 4: vision history (hist_slots x FW_BLOCK)]
__device__ __forceinline__ void ol_smem_carve(const FwDev& p, float* stage, float*& so, float*& depth_row, float*& hs) {
    so = stage + (size_t)FW_BLOCK * (p.obs_dim > 0 ? p.obs_dim : 1);
    float* rows = so + (size_t)(p.num_obstacles > 0 ? p.num_obstacles : 1) * 3 * FW_BLOCK;
    depth_row = rows + (size_t)(threadIdx.x >> 5) * p.cam_res;
    hs = rows + (size_t)(FW_BLOCK / 32) * p.cam_res;
}

// launch bound 7 blocks/SM x 64 threads (register cap 146; ptxas settles at 128 with ~70 bytes of spills, so 8 blocks fit):
// 148 x 448 = 66,304 >= 65,536 envs, a single wave either way
template <bool RANDOM_ACT, int TASK, bool STD, bool FIELD = false>
__global__ void __launch_bounds__(FW_BLOCK, 7)
fw_step_objlock_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, const float4* __restrict__ act,
                       float* __restrict__ obs, float* __restrict__ rew, uint8_t* __restrict__ flg,
                       float* __restrict__ term_obs, int spl, int bulk_ok) {
    extern __shared__ __align__(128) float stage[];
    const int bx = (int)blockIdx.x;
    const int i = p.i_begin + bx * FW_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int D = p.obs_dim;
    float* stage_warp = stage + (size_t)warp * 32 * D;
    float* row = obs != nullptr ? stage_warp + (size_t)lane * D : nullptr;
    float *so, *depth_row, *hs;
    ol_smem_carve(p, stage, so, depth_row, hs);
    const bool active = i < p.i_end;
    const uint32_t gid = p.env_id0 + (uint32_t)i;
    EnvState e = {};
    OlState ol = {};
    float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;
    float ep_ret = 0.f, reward = 0.f;
    uint32_t bits = 0u;
    int tidx_info = 0;
    if (active) {
        fw_load(pl, i, e);
        ol_load(pl, i, ol);
        ol_stage_obstacles(p, pl, i, ol.n_obst, so, threadIdx.x, FW_BLOCK);
        if (TASK == 4) ol_hist_load(p, pl, i, hs, threadIdx.x, FW_BLOCK);
        if (p.wind_mode != 0) { w0 = pl.w0[i]; w1 = pl.w1[i]; }
        ep_ret = pl.ep_ret[i];
    }
    __syncwarp();
    const int nsteps = RANDOM_ACT ? spl : 1;
    for (int st = 0; st < nsteps; ++st) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        if (active) {
            if (RANDOM_ACT) {
                uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid, e.episode, (uint32_t)e.step_count, FWD_STREAM_ACTION);
                a0 = 2.0f * fw_u01(r.x) - 1.0f; a1 = 2.0f * fw_u01(r.y) - 1.0f;
                a2 = 2.0f * fw_u01(r.z) - 1.0f; a3 = 2.0f * fw_u01(r.w) - 1.0f;
            } else {
                float4 a = act[i];
                a0 = a.x; a1 = a.y; a2 = a.z; a3 = a.w;
            }
        }
        reward = fw_env_step_objlock<TASK, STD, FIELD>(p, pl, active, e, ol, so, depth_row, hs, i, gid, a0, a1, a2, a3, w0, w1, ep_ret,
                                     (st == nsteps - 1) ? row : nullptr,
                                     (!RANDOM_ACT && term_obs != nullptr && row != nullptr && active) ? term_obs + (size_t)i * D : nullptr,
                                     bits, tidx_info);
    }
    if (active) {
        pl.ep_ret[i] = ep_ret;
        fw_store(pl, i, e);
        ol_store(pl, i, ol);
        if (TASK == 4) ol_hist_store(p, pl, i, hs, threadIdx.x, FW_BLOCK);
        if (rew != nullptr) rew[i] = reward;
        if (flg != nullptr) flg[i] = (uint8_t)bits;
        if (TASK == 2 && !RANDOM_ACT && pl.tidx_out != nullptr) pl.tidx_out[i] = (uint8_t)tidx_info;
    }
    if (obs != nullptr) {
        const int first_env = p.i_begin + bx * FW_BLOCK + warp * 32;
        if (first_env < p.i_end)
            fw_flush_obs(obs, stage_warp, D, first_env, p.i_end, lane, bulk_ok != 0,
                         (!RANDOM_ACT && pl.obs_acc != nullptr) ? pl.obs_acc + (size_t)(bx & (FW_OBS_ACC_SLOTS - 1)) * 2 * D : nullptr);
    }
}

template <int TASK, bool FIELD = false>
__global__ void __launch_bounds__(FW_BLOCK)
fw_reset_objlock_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, const uint8_t* __restrict__ mask,
                        float* __restrict__ obs, int bulk_ok, int emit_only) {
    extern __shared__ __align__(128) float stage[];
    const int i = blockIdx.x * FW_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int D = p.obs_dim;
    float* stage_warp = stage + (size_t)warp * 32 * D;
    float* row = stage_warp + (size_t)lane * D;
    float *so, *depth_row, *hs;
    ol_smem_carve(p, stage, so, depth_row, hs);
    const bool active = i < p.n;
    EnvState e = {};
    OlState ol = {};
    if (active) {
        fw_load(pl, i, e); ol_load(pl, i, ol);
        if (TASK == 4) ol_hist_load(p, pl, i, hs, threadIdx.x, FW_BLOCK);
    }
    const bool sel = active && !emit_only && (mask == nullptr || mask[i] != 0);
    ol_reset_lanes<TASK, FIELD>(p, pl, sel, e, ol, so, depth_row, hs, i, p.env_id0 + (uint32_t)i, e.episode + 1u, threadIdx.x);
    if (sel) {
        pl.ep_ret[i] = 0.0f;
        fw_store(pl, i, e);
        ol_store(pl, i, ol);
        if (TASK == 4) ol_hist_store(p, pl, i, hs, threadIdx.x, FW_BLOCK);
    }
    if (active) ol_write_obs<TASK>(p, pl, e, ol, hs, i, e.tidx, 0.f, 0.f, 0.f, 0.f, row, threadIdx.x);
    if (obs != nullptr) {
        const int first_env = blockIdx.x * FW_BLOCK + warp * 32;
        if (first_env < p.n) fw_flush_obs(obs, stage_warp, D, first_env, p.n, lane, bulk_ok != 0);
    }
}

// Producer side of the spare episodes, a kernel of its own (its stack frame and registers stay out of the step kernel):
// entry k of the list = (env index, episode).  OL_REFILL_PER_WARP requests per warp pass -- begin_reset, waypoints / duck /
// obstacles, the warm-up under wind with its camera frame, end_reset's compute_state -- through ol_reset_lanes on the
// spare view of the planes, i.e. the very code of the in-step reset; data first, tag last.  The last block to finish
// clears the list's counter for the step launch that appends to it next.
// whole_batch > 0: episode (live episode + 1) of every env 0..whole_batch-1, full warps (fw_create, right after the first reset).
#define FW_REFILL_GRID 64
template <int TASK, bool FIELD = false>
__global__ void __launch_bounds__(FW_BLOCK, 7)
fw_refill_objlock_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, const int2* __restrict__ list,
                         int* __restrict__ count, int* __restrict__ blocks_done, int cap, int whole_batch) {
    extern __shared__ __align__(128) float stage[];
    float *so, *depth_row, *hs;
    ol_smem_carve(p, stage, so, depth_row, hs);
    const FwPlanes sv = ol_spare_view(pl);
    const int n = whole_batch > 0 ? whole_batch : min(*reinterpret_cast<volatile int*>(count), cap);
    const int per = whole_batch > 0 ? 32 : OL_REFILL_PER_WARP;
    const int lane = threadIdx.x & 31;
    const int wg = blockIdx.x * (FW_BLOCK / 32) + (threadIdx.x >> 5), nw = gridDim.x * (FW_BLOCK / 32);
    for (int base = wg * per; base < n; base += nw * per) {
        const int idx = base + lane;
        const bool doing = lane < per && idx < n;
        int2 ent = make_int2(0, 0);
        if (doing) ent = whole_batch > 0 ? make_int2(idx, pl.s5[idx].z + 1) : list[idx];
        const int i = ent.x;
        EnvState e = {};
        OlState ol = {};
        ol_reset_lanes<TASK, FIELD>(p, sv, doing, e, ol, so, depth_row, hs, i, p.env_id0 + (uint32_t)i, (uint32_t)ent.y, threadIdx.x);
        if (doing) {
            sv.s0[i] = make_float4(e.px, e.py, e.pz, e.thr);
            sv.s1[i] = make_float4(e.qx, e.qy, e.qz, e.qw);
            sv.s2[i] = make_float4(e.vx, e.vy, e.vz, e.act[0]);
            sv.s3[i] = make_float4(e.wx, e.wy, e.wz, e.act[1]);
            sv.s4[i] = make_float4(e.act[2], e.act[3], e.act[4], e.new_dist);
            ol_store(sv, i, ol);
            if (TASK == 4) ol_hist_store(p, sv, i, hs, threadIdx.x, FW_BLOCK);
            __threadfence();                            // release: everything above is visible before the tag
            sv.s5[i] = make_int4(e.step_count, e.physics_steps, ent.y, e.tidx);
        }
        __syncwarp();
    }
    if (whole_batch == 0) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(blocks_done, 1) == (int)gridDim.x - 1) { *count = 0; *blocks_done = 0; __threadfence(); }
        }
    }
}

// one thread: run the deterministic warm-up once so resets can copy its result
__global__ void fw_warm_kernel(const __grid_constant__ FwDev p, const FwPlanes pl, float* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    EnvState e;
    FwDev q = p;   // local copy with task 0: no target sampling, no plane writes
    q.task = 0; q.wind_mode = 0; q.warm_cached = 0;
    fw_reset_env(q, pl, e, 0, 0u, 0u);
    out[0] = e.px; out[1] = e.py; out[2] = e.pz;
    out[3] = e.qx; out[4] = e.qy; out[5] = e.qz; out[6] = e.qw;
    out[7] = e.vx; out[8] = e.vy; out[9] = e.vz;
    out[10] = e.wx; out[11] = e.wy; out[12] = e.wz;
    for (int s = 0; s < FWD_NSURF; ++s) out[13 + s] = e.act[s];
    out[18] = e.thr; out[19] = 0.0f;
}

// ------------------------------------------------------------------ launchers
static inline size_t stage_bytes(const FwDev& p) {
    size_t obs = (size_t)(FW_BLOCK / 32) * 32 * (size_t)(p.obs_dim > 0 ? p.obs_dim : 1) * 4;
    size_t obst = (p.task == 2 || p.task == 4) ? ((size_t)(p.num_obstacles > 0 ? p.num_obstacles : 1) * 3 * FW_BLOCK +
                                                  (size_t)(FW_BLOCK / 32) * p.cam_res) * 4 : 0;
    size_t hist = p.task == 4 ? (size_t)p.hist_slots * FW_BLOCK * 4 : 0;
    return obs + obst + hist;
}
static inline int grid_for(int n) { return (n + FW_BLOCK - 1) / FW_BLOCK; }

typedef void (*fw_step_fn)(const FwDev, const FwPlanes, const float4*, float*, float*, uint8_t*, float*, int, int);

// a step kernel with its launch geometry
struct StepLaunch {
    fw_step_fn fn;
    int threads, envs_per_block;
    size_t smem;
};

static inline size_t stage_bytes2(const FwDev& p) {
    return ((size_t)(FW2_THREADS * 2) * (size_t)(p.obs_dim > 0 ? p.obs_dim : 1) + (size_t)FW2_THREADS * 2 * FW2_SNAP) * 4;
}

// FwConfig.packed_pairs selects the two-env-per-thread kernels per handle; FWSIM_PACKED=1 / 0 overrides it for every
// handle of the process (A/B measurements)
static bool packed_enabled(const FwDev& p) {
    const char* e = getenv("FWSIM_PACKED");
    if (e != nullptr && *e != 0) return atoi(e) != 0;
    return p.packed != 0;
}

// the gridded-wind (FIELD) instantiations of the one-env kernels, selected by wind_mode 3
static fw_step_fn step_fn_field(const FwDev& p, bool random_act) {
    const int task = p.task;
    const bool sg = p.std_geom != 0;
    const bool r = random_act;
    switch (task) {
    case 0: return sg ? (r ? fw_step_kernel<0, true, true, true> : fw_step_kernel<0, false, true, true>)
                      : (r ? fw_step_kernel<0, true, false, true> : fw_step_kernel<0, false, false, true>);
    case 1: return sg ? (r ? fw_step_kernel<1, true, true, true> : fw_step_kernel<1, false, true, true>)
                      : (r ? fw_step_kernel<1, true, false, true> : fw_step_kernel<1, false, false, true>);
    case 3: return sg ? (r ? fw_step_kernel<3, true, true, true> : fw_step_kernel<3, false, true, true>)
                      : (r ? fw_step_kernel<3, true, false, true> : fw_step_kernel<3, false, false, true>);
    case 2: return sg ? (r ? fw_step_objlock_kernel<true, 2, true, true> : fw_step_objlock_kernel<false, 2, true, true>)
                      : (r ? fw_step_objlock_kernel<true, 2, false, true> : fw_step_objlock_kernel<false, 2, false, true>);
    case 4: return sg ? (r ? fw_step_objlock_kernel<true, 4, true, true> : fw_step_objlock_kernel<false, 4, true, true>)
                      : (r ? fw_step_objlock_kernel<true, 4, false, true> : fw_step_objlock_kernel<false, 4, false, true>);
    default: return nullptr;
    }
}

static StepLaunch step_launch(const FwDev& p, bool random_act) {
    const int task = p.task;
    const bool std_geom = p.std_geom != 0;
    fw_step_fn fn = nullptr;
    // gridded wind: one env per thread (the packed path does not sample fields)
    if (p.wind_mode == 3) return StepLaunch{step_fn_field(p, random_act), FW_BLOCK, FW_BLOCK, stage_bytes(p)};
    // two envs per thread on the packed fp32x2 path: standard layout, no quaternion step limiter (fw_pack.cuh)
    if (std_geom && !p.quat_limiter && packed_enabled(p) && (task == 0 || task == 1 || task == 3)) {
        if (task == 0) fn = random_act ? fw_step2_kernel<0, true> : fw_step2_kernel<0, false>;
        if (task == 1) fn = random_act ? fw_step2_kernel<1, true> : fw_step2_kernel<1, false>;
        if (task == 3) fn = random_act ? fw_step2_kernel<3, true> : fw_step2_kernel<3, false>;
        return StepLaunch{fn, FW2_THREADS, FW2_THREADS * 2, stage_bytes2(p)};
    }
    if (task == 0 && std_geom) fn = random_act ? fw_step_kernel<0, true, true> : fw_step_kernel<0, false, true>;
    else if (task == 1 && std_geom) fn = random_act ? fw_step_kernel<1, true, true> : fw_step_kernel<1, false, true>;
    else if (task == 3 && std_geom) fn = random_act ? fw_step_kernel<3, true, true> : fw_step_kernel<3, false, true>;
    else if (task == 3) fn = random_act ? fw_step_kernel<3, true, false> : fw_step_kernel<3, false, false>;
    else if (task == 0) fn = random_act ? fw_step_kernel<0, true, false> : fw_step_kernel<0, false, false>;
    else if (task == 1) fn = random_act ? fw_step_kernel<1, true, false> : fw_step_kernel<1, false, false>;
    else if (task == 2 && std_geom) fn = random_act ? fw_step_objlock_kernel<true, 2, true> : fw_step_objlock_kernel<false, 2, true>;
    else if (task == 4 && std_geom) fn = random_act ? fw_step_objlock_kernel<true, 4, true> : fw_step_objlock_kernel<false, 4, true>;
    else if (task == 2) fn = random_act ? fw_step_objlock_kernel<true, 2, false> : fw_step_objlock_kernel<false, 2, false>;
    else if (task == 4) fn = random_act ? fw_step_objlock_kernel<true, 4, false> : fw_step_objlock_kernel<false, 4, false>;
    return StepLaunch{fn, FW_BLOCK, FW_BLOCK, stage_bytes(p)};
}

// dynamic shared memory beyond the 48 KB default needs an explicit opt-in per kernel (large obstacle tables or camera
// rows); returns false when the request exceeds what an SM offers
static bool smem_opt_in(const void* fn, size_t bytes) {
    if (bytes <= 48 * 1024) return true;
    if (bytes > 227 * 1024) return false;
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess;
}

cudaError_t fwk_launch_step(const FwDev& p, const FwPlanes& pl, const float* act, float* obs, float* rew, uint8_t* flg,
                            float* term_obs, bool random_act, int spl, cudaStream_t st) {
    const StepLaunch L = step_launch(p, random_act);
    if (L.fn == nullptr) return cudaErrorNotSupported;
    // the bulk store of a warp's observation rows needs a 16-byte aligned destination and size
    const int rows = L.envs_per_block == FW_BLOCK ? 32 : 64;
    const int bulk_ok = (obs != nullptr) && ((reinterpret_cast<uintptr_t>(obs) & 15u) == 0) && ((p.obs_dim * rows * 4) % 16 == 0) &&
                        (((size_t)p.i_begin * p.obs_dim * 4) % 16 == 0);
    if (!smem_opt_in((const void*)L.fn, L.smem)) return cudaErrorInvalidValue;
    const int n = p.i_end - p.i_begin;
    L.fn<<<(n + L.envs_per_block - 1) / L.envs_per_block, L.threads, L.smem, st>>>(p, pl, reinterpret_cast<const float4*>(act), obs, rew,
                                                                                  flg, term_obs, spl, bulk_ok);
    return cudaGetLastError();
}

// Append one random-action step launch to a CUDA graph (explicit node: works without stream capture, so the
// graph can later be launched on any stream including the legacy default stream torch hands us).
// pdl: 0 = ordinary dependencies; 1 / 2 = the single dependency (if any) becomes a programmatic edge and the kernel runs in
// PDL mode 1 / 2 (see fw_step_kernel) -- only the one-env-per-thread K1 kernels implement the prologue
bool fwk_step_supports_pdl(const FwDev& p) { return step_launch(p, true).envs_per_block == FW_BLOCK && (p.task == 0 || p.task == 1 || p.task == 3); }

cudaError_t fwk_graph_add_random_step(cudaGraph_t g, cudaGraphNode_t* deps, int ndeps, const FwDev& p, const FwPlanes& pl,
                                      int spl, cudaGraphNode_t* out, int pdl) {
    const StepLaunch L = step_launch(p, true);
    if (L.fn == nullptr) return cudaErrorNotSupported;
    if (!smem_opt_in((const void*)L.fn, L.smem)) return cudaErrorInvalidValue;
    if (pdl != 0 && (!fwk_step_supports_pdl(p) || ndeps > 1)) pdl = 0;
    FwDev pc = p; FwPlanes plc = pl;
    const float4* act = nullptr; float* obs = nullptr; float* rew = nullptr; uint8_t* flg = nullptr; float* term = nullptr;
    int spl_ = spl, bulk = pdl << 1;
    void* args[] = {&pc, &plc, &act, &obs, &rew, &flg, &term, &spl_, &bulk};
    cudaKernelNodeParams kp;
    memset(&kp, 0, sizeof(kp));
    kp.func = (void*)L.fn;
    const int n = p.i_end - p.i_begin;
    kp.gridDim = dim3((n + L.envs_per_block - 1) / L.envs_per_block); kp.blockDim = dim3(L.threads);
    kp.sharedMemBytes = (unsigned)L.smem;
    kp.kernelParams = args; kp.extra = nullptr;
    if (pdl == 0 || ndeps == 0) return cudaGraphAddKernelNode(out, g, deps, ndeps, &kp);
    cudaError_t e = cudaGraphAddKernelNode(out, g, nullptr, 0, &kp);
    if (e != cudaSuccess) return e;
    cudaGraphEdgeData ed;
    memset(&ed, 0, sizeof(ed));
    ed.from_port = cudaGraphKernelNodePortProgrammatic;
    ed.type = cudaGraphDependencyTypeProgrammatic;
    return cudaGraphAddDependencies_v2(g, deps, out, &ed, 1);
}

typedef void (*fw_refill_fn)(const FwDev, const FwPlanes, const int2*, int*, int*, int, int);
static fw_refill_fn refill_fn(const FwDev& p) {
    if (p.wind_mode == 3) return p.task == 2 ? fw_refill_objlock_kernel<2, true> : fw_refill_objlock_kernel<4, true>;
    return p.task == 2 ? fw_refill_objlock_kernel<2> : fw_refill_objlock_kernel<4>;
}

static int refill_grid(int work, bool whole_batch) {
    const int per_block = (FW_BLOCK / 32) * (whole_batch ? 32 : OL_REFILL_PER_WARP);
    const int grid = (work + per_block - 1) / per_block;
    const int gmax = whole_batch ? 1036 : FW_REFILL_GRID;
    return grid > gmax ? gmax : (grid < 1 ? 1 : grid);
}

// serve a request list (whole_batch == 0) or prepare the next episode of every env (whole_batch = n, right after fw_create)
cudaError_t fwk_launch_refill(const FwDev& p, const FwPlanes& pl, const int2* list, int* count, int* blocks_done, int cap,
                              int whole_batch, cudaStream_t st) {
    if (p.task != 2 && p.task != 4) return cudaErrorNotSupported;
    auto fn = refill_fn(p);
    if (!smem_opt_in((const void*)fn, stage_bytes(p))) return cudaErrorInvalidValue;
    fn<<<refill_grid(whole_batch > 0 ? whole_batch : cap, whole_batch > 0), FW_BLOCK, stage_bytes(p), st>>>(p, pl, list, count, blocks_done,
                                                                                                          cap, whole_batch);
    return cudaGetLastError();
}

cudaError_t fwk_graph_add_refill(cudaGraph_t g, cudaGraphNode_t* deps, int ndeps, const FwDev& p, const FwPlanes& pl,
                                 const int2* list, int* count, int* blocks_done, int cap, cudaGraphNode_t* out) {
    auto fn = refill_fn(p);
    if (!smem_opt_in((const void*)fn, stage_bytes(p))) return cudaErrorInvalidValue;
    FwDev pc = p; FwPlanes plc = pl;
    const int2* l = list; int* c = count; int* bd = blocks_done; int cap_ = cap, wb = 0;
    void* args[] = {&pc, &plc, &l, &c, &bd, &cap_, &wb};
    cudaKernelNodeParams kp;
    memset(&kp, 0, sizeof(kp));
    kp.func = (void*)fn;
    kp.gridDim = dim3(refill_grid(cap, false)); kp.blockDim = dim3(FW_BLOCK);
    kp.sharedMemBytes = (unsigned)stage_bytes(p);
    kp.kernelParams = args; kp.extra = nullptr;
    cudaError_t e = cudaGraphAddKernelNode(out, g, deps, ndeps, &kp);
    if (e != cudaSuccess) return e;
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess && lo != hi) {
        cudaKernelNodeAttrValue v;
        memset(&v, 0, sizeof(v));
        v.priority = lo;                               // numerically largest = lowest priority: the step's blocks go first
        (void)cudaGraphKernelNodeSetAttribute(*out, cudaLaunchAttributePriority, &v);
        (void)cudaGetLastError();
    }
    return cudaSuccess;
}

cudaError_t fwk_launch_reset(const FwDev& p, const FwPlanes& pl, const uint8_t* mask, float* obs, bool emit_only,
                             cudaStream_t st) {
    const int bulk_ok = (obs != nullptr) && ((reinterpret_cast<uintptr_t>(obs) & 15u) == 0);
    const bool field = p.wind_mode == 3;
    if (p.task == 2 || p.task == 4) {
        auto fn = field ? (p.task == 2 ? fw_reset_objlock_kernel<2, true> : fw_reset_objlock_kernel<4, true>)
                        : (p.task == 2 ? fw_reset_objlock_kernel<2> : fw_reset_objlock_kernel<4>);
        if (!smem_opt_in((const void*)fn, stage_bytes(p))) return cudaErrorInvalidValue;
        fn<<<grid_for(p.n), FW_BLOCK, stage_bytes(p), st>>>(p, pl, mask, obs, bulk_ok, emit_only ? 1 : 0);
    } else {
        auto fn = field ? fw_reset_kernel<true> : fw_reset_kernel<false>;
        fn<<<grid_for(p.n), FW_BLOCK, stage_bytes(p), st>>>(p, pl, mask, obs, bulk_ok, emit_only ? 1 : 0);
    }
    return cudaGetLastError();
}

cudaError_t fwk_launch_warm(const FwDev& p, const FwPlanes& pl, float* out, cudaStream_t st) {
    fw_warm_kernel<<<1, 32, 0, st>>>(p, pl, out);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ FP32 FMA-chain peak (roofline denominator)
// MEASURED_PEAKS.json has no non-tensor FP32 entry; SURVEY section 8(d) asks the first GPU run to measure one.
__global__ void __launch_bounds__(256) fw_fma_peak_kernel(float* out, int iters, float a, float b) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f;
    float x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    float s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456f) out[0] = s;   // keep the chain alive
}

cudaError_t fwk_fma_peak(int sm_count, int iters, float* scratch, double* flops_per_launch, cudaStream_t st) {
    const int blocks = sm_count * 8, threads = 256;
    fw_fma_peak_kernel<<<blocks, threads, 0, st>>>(scratch, iters, 0.999f, 0.001f);
    *flops_per_launch = (double)blocks * threads * (double)iters * 64.0 * 2.0;
    return cudaGetLastError();
}
