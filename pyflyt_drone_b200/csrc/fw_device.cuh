// fw_device.cuh -- device-side model of one fixed-wing environment (fp32, one thread per env).
//
// Replaces, per 240 Hz physics substep, what the reference runs through PyFlyt + PyBullet on the CPU:
//   Fixedwing.update_control / update_physics / update_state, LiftingSurface(s), Motors, stepSimulation
//   (call sites: /root/reference/envs/fixedwing_envs/fixedwing_base_env.py:331,339), and per agent step
//   FixedwingBaseEnv.step (:314-348), compute_base_term_trunc_reward (:296-312), the waypoint
//   compute_state / compute_term_trunc_reward (/root/reference/envs/fixedwing_waypoint_objlock_env.py:197-343)
//   and FlattenWaypointEnv.observation (/root/reference/envs/flatten_waypoint_env.py:52-72).
// Aircraft constants: /root/reference/my_models/fixedwing/fixewing.yaml:1-71 (folded into SurfDev by fw_api.cu).
#pragma once
#define FW_OBS_ACC_SLOTS 64

#include <cuda_runtime.h>
#include <stdint.h>

#define FWD_NSURF 5
#define FWD_MAX_COL 16
#define FWD_MAX_TARGETS 16

#define FWD_STREAM_TARGETS 1u
#define FWD_STREAM_NOISE 2u
#define FWD_STREAM_ACTION 3u
#define FWD_STREAM_WIND 4u
#define FWD_STREAM_DUCK 5u
#define FWD_STREAM_OBST 6u

#define FWD_PI 3.14159265358979323846f
#define FWD_HALF_PI 1.57079632679489661923f

// per-surface constants, all derived on the host in double and rounded once
struct SurfDev {
    float k_act;        // dt / tau
    float defl_rad;     // deflection limit, radians
    float defl_deg;     // deflection limit, degrees
    float cla;          // Cl_alpha_3D
    float tau_eta;      // aero_tau * eta  (= delta_Cl / (cla * deflection))
    float omf;          // 1 - flap_to_chord
    float a0_base, asp_base, asn_base;  // radians
    float inv_pi_ar;    // 1 / (pi * aspect)
    float cd0;
    float stall_k;      // 0.41 * (1 - exp(-17 / aspect))
    float qarea;        // 0.5 * rho * area
    float chord;
    float lift[3], fwd[3], tq[3], r[3];
    float ra[3], rb[3];   // r x lift, r x fwd: moment arms of the normal / parallel force components about O
    // folded products (one FMA each in the kernel): te = k_te * act; shift = k_shift * act;
    // CM * chord = -CN * (cm0c + cm1c * |alpha_eff|); induced-angle slope cla * inv_pi_ar
    float k_te, k_shift, cm0c, cm1c, cla_ipa;
};

// The per-surface constants the standard-layout substep reads, packed in the order of use as six 16-byte groups: on
// sm_100a every constant operand reaches the FP pipe through a uniform register filled by an LDCU, and one LDCU.128
// fetches a whole group (the scalar fields of SurfDev cost one LDCU each: 90 of the 629 instructions of a substep).
//   g0: k_act, r.x, r.y, r.z          g1: a0_base, k_te, asp_base, asn_base     g2: k_shift, cla, cla_ipa, cd0
//   g3: defl (deg|rad as cd90_degrees says), stall_k, cm1c, cm0c                g4: qarea, ra.x, ra.y, ra.z
//   g5: rb.x, rb.y, rb.z, -
struct SurfHot {
    float k_act, r[3];
    float a0_base, k_te, asp_base, asn_base;
    float k_shift, cla, cla_ipa, cd0;
    float defl_sel, stall_k, cm1c, cm0c;
    float qarea, ra[3];
    float rb[3];
};

__device__ __forceinline__ SurfHot fw_load_hot(const float4 (&g)[6]) {
    const float4 g0 = g[0], g1 = g[1], g2 = g[2], g3 = g[3], g4 = g[4], g5 = g[5];
    SurfHot h;
    h.k_act = g0.x; h.r[0] = g0.y; h.r[1] = g0.z; h.r[2] = g0.w;
    h.a0_base = g1.x; h.k_te = g1.y; h.asp_base = g1.z; h.asn_base = g1.w;
    h.k_shift = g2.x; h.cla = g2.y; h.cla_ipa = g2.z; h.cd0 = g2.w;
    h.defl_sel = g3.x; h.stall_k = g3.y; h.cm1c = g3.z; h.cm0c = g3.w;
    h.qarea = g4.x; h.ra[0] = g4.y; h.ra[1] = g4.z; h.ra[2] = g4.w;
    h.rb[0] = g5.x; h.rb[1] = g5.y; h.rb[2] = g5.z;
    return h;
}

// Rigid-body / motor constants of the standard-layout substep, packed the same way (fw_api.cu: derive()):
//   0: motor_k, noise_ratio, thrust_max, torque_max      1: r_motor.y, r_motor.z, gravity, mass
//   2: com.xyz, max_vel                                  3-4: inertia[0..7]        5: inertia[8], lateral minv 0,2,4 ...
//   5.y-7.z: lateral block minv[0,2,4,12,14,16,24,26,28]   7.w-9.w: longitudinal block minv[7,9,11,19,21,23,31,33,35]
#define FWD_RBK 10

struct FwDev {
    alignas(16) float4 hot[FWD_NSURF][6];
    alignas(16) float4 rbk[FWD_RBK];
    SurfDev surf[FWD_NSURF];
    // motor
    float motor_k, noise_ratio, thrust_max, torque_max;
    float r_motor[3], thrust_unit[3];
    // rigid body about O
    float mass;
    float com[3];
    float inertia[9];
    float minv[36];
    float col[FWD_MAX_COL][3];
    float col_radius, contact_margin;
    int n_col;
    // simulator
    float dt, gravity, max_vel;
    float sign_ail_l, sign_ail_r, sign_pitch, sign_yaw;
    int substeps_per_inner, inner_per_step, warmup_substeps;
    int freestream_3d, cd90_degrees, quat_limiter;
    // env
    int task, num_targets, sparse_reward, angle_repr, max_steps, context_len, obs_dim, act_dim;
    int early_return_on_crash, complete_truncates;
    float goal_reach, dome, dome2, spawn_size, min_height;
    float start_pos[3], start_vel[3];
    // wind
    int wind_mode, wind_randomize, wind_rand_phase, wind_start_substep;
    float wind_base[3], wind_base_lo[3], wind_base_hi[3];
    float gust_amp[3], gust_amp_lo[3], gust_amp_hi[3];
    float gust_omega, gust_phase;   // 2*pi*f
    float gust_cyc;                 // f * dt: gust cycles per physics substep
    // ObjLock task (fixedwing_waypoint_objlock_env.py:42-168)
    int num_obstacles, cam_interval, lock_hold, switch_min_seen, cam_res;
    float obst_radius, obst_h_lo, obst_h_hi, obst_safe, obst_scale, obst_max_pen;
    float strike_dist, strike_reward, lock_step_reward, approach_scale, switch_min_area;
    float duck_radius, cam_offset[3], cam_near, cam_far;
    // camera model: 0 tracking chase camera, 1 fixed camera with body-frame forward / up-hint axes cam_fb / cam_ub
    int cam_mode;
    float cam_fb[3], cam_ub[3];
    // duck-only task (fixedwing_objlock_env.py:37-118)
    int hist_len, use_deltas, lock_decay, hist_slots;     // hist_slots = 9 * hist_len + 4
    float duck_dist_scale, lock_center_radius, centering_scale, visible_step_reward, area_reward_scale;
    float lock_lost_penalty, approach_clip;
    // cached post-warm-up state (valid when no wind acts during the warm-up): pos3 quat4 vel3 omega3 act5 thr
    int warm_cached;
    float warm[20];
    // 1 when the aircraft has the standard layout the STD kernels are specialised for (see fw_substep)
    int std_geom;
    // 1: step tasks 0/1/3 with two envs per thread on the packed fp32x2 path (fw_pack.cuh; needs std_geom, no quat limiter)
    int packed;
    // rng / sharding
    uint32_t seed_lo, seed_hi, env_id0;
    int n;
    // env range [i_begin, i_end) a step launch covers (whole batch by default; the host lane launches chunks so that
    // the device-to-host copy of one chunk overlaps the kernel of the next)
    int i_begin, i_end;
    // gridded wind field (wind_mode 3, fw_set_wind_field): world-frame wind as float4 lattice points [nt][nz][ny][nx] in HBM,
    // owned by the handle and fixed before the first launch.  Per env, w0 holds the episode's spatial shift (xyz, metres; the
    // field is sampled at position - shift) and time offset (w, seconds).
    const float4* wf;
    int wf_n[4];                          // nx, ny, nz, nt
    int wf_pts;                           // nx * ny * nz: points per time slice
    float wf_origin[3], wf_inv_sp[3];     // lattice origin, 1 / spacing
    float wf_max[3];                      // n - 1 per axis: the clamp of the lattice coordinate
    float wf_sps, wf_inv_tstep, wf_nt, wf_inv_nt;   // dt / t_step (slices per substep), 1 / t_step, nt, 1 / nt
    float wf_period;                      // nt * t_step: the time offset is drawn from [0, period)
    float wf_shift_lo[3], wf_shift_hi[3];
    int wf_rand_time;
};

// time pair of the gridded field for one substep, shared by all surfaces: slices a, b and the weight of b.  on = false before
// the wind starts (stamp < 0 or < wind_start_substep): the surfaces then see calm air.
struct FwFieldT {
    const float4* a;
    const float4* b;
    float wb;
    float sx, sy, sz;     // the episode's spatial shift
    bool on;
};

// SoA state in HBM: float4 planes (16-byte coalesced accesses, one plane element per env)
struct FwPlanes {
    float4* s0;   // pos.xyz, throttle
    float4* s1;   // quat xyzw
    float4* s2;   // vel.xyz, act0
    float4* s3;   // omega.xyz, act1
    float4* s4;   // act2, act3, act4, new_dist
    int4* s5;     // step_count, physics_steps, episode, target_idx
    float4* w0;   // wind base xyz, gust phase
    float4* w1;   // gust amp xyz, -
    float* targets;  // [T][3][N]
    float* ep_ret;   // [N]
    double* stats;   // [16] global accumulators: [0..7] episode statistics (fw_episode_stats), [8] non-finite-state resets
    uint8_t* tidx_out;  // [N] info["num_targets_reached"] of the step just taken (before any auto-reset); may be host-mapped
    // optional: FW_OBS_ACC_SLOTS x double[2 * obs_dim] = column sums | sums of squares of the observations a step writes
    // (slot = block index mod FW_OBS_ACC_SLOTS, spreading the atomics); fw_set_obs_accumulator, consumed by ppo_moments_finalize
    double* obs_acc;
    // ObjLock task only
    float4* dk;      // duck xyz
    float4* v0;      // last_cx, last_cy, last_area, last_depth
    float4* v1;      // frame cx, cy, area, depth
    float4* v2;      // frame d_left, d_center, d_right, prev_est_dist
    int4* v3;        // bits (duck_phase, has_prev, post_wp, cam_valid, frame_visible, n_obst<<8), seen, lock, since
    float* obst;     // [MAX_OBST][3][N]  x, y, height
    float* hist;     // duck-only task: [9 * hist_len + 4][N] vision history rows (newest first) then the four deltas
    // Pre-warmed spare episodes (camera tasks): a second set of the planes above holding every env's NEXT episode already
    // reset, warmed up and observed.  The state an env resets to depends only on (seed, env id, episode), so it can be
    // prepared ahead of time by fw_refill_objlock_kernel -- a few requests per warp, on a side stream beside the next step --
    // instead of by the one or two finished lanes of a stepping warp dragging 30 idle ones through 20 warm-up substeps and
    // a camera frame.  sp_s5[i].z (the episode number) is the validity tag: an env that finishes episode k takes the spare
    // iff the tag reads k + 1, else it resets inline; either way it appends (i, k + 2) to the request list of the launch.
    // All nullptr / 0 when the feature is off.
    float4 *sp_s0, *sp_s1, *sp_s2, *sp_s3, *sp_s4;
    int4* sp_s5;
    float4 *sp_w0, *sp_w1;
    float* sp_targets;
    float4 *sp_dk, *sp_v0, *sp_v1, *sp_v2;
    int4* sp_v3;
    float* sp_obst;
    float* sp_hist;
    int2* refill_list;   // [refill_cap] (env index, episode to prepare): requests of THIS launch
    int* refill_count;
    int refill_cap;
};

struct EnvState {
    float px, py, pz;
    float qx, qy, qz, qw;
    float vx, vy, vz;
    float wx, wy, wz;
    float act[FWD_NSURF];
    float thr;
    float new_dist;
    int step_count, physics_steps, tidx;
    uint32_t episode;
};

// ------------------------------------------------------------------ RNG: Philox4x32-10
__device__ __forceinline__ uint4 fw_philox(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
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
__device__ __forceinline__ float fw_u01(uint32_t x) { return ((float)(x >> 9) + 0.5f) * (1.0f / 8388608.0f); }

__device__ __forceinline__ void fw_normals4(const FwDev& p, uint32_t env, uint32_t episode, uint32_t idx, float n[4]) {
    uint4 r = fw_philox(p.seed_lo, p.seed_hi, env, episode, idx, FWD_STREAM_NOISE);
    // Box-Muller on SFU approximations (MUFU.LG2/SIN/COS): the 2e-7 absolute error is far below the
    // 2 % multiplicative motor noise this feeds
    float ra = sqrtf(-2.0f * __logf(fw_u01(r.x))), rb = sqrtf(-2.0f * __logf(fw_u01(r.z)));
    float a0 = 2.0f * FWD_PI * fw_u01(r.y) - FWD_PI, a1 = 2.0f * FWD_PI * fw_u01(r.w) - FWD_PI;   // [-pi, pi)
    float s0 = -__sinf(a0), c0 = -__cosf(a0), s1 = -__sinf(a1), c1 = -__cosf(a1);
    n[0] = ra * c0; n[1] = ra * s0; n[2] = rb * c1; n[3] = rb * s1;
}

// ------------------------------------------------------------------ math helpers
// MUFU.SIN/COS: absolute error 2^-21.4 on [-pi, pi], which is where the effective angle of attack lives.
// (The libdevice sincosf was measured to give the same parity against the fp64 oracle at 6x the instructions.)
__device__ __forceinline__ void fw_sincos(float x, float* s, float* c) { *s = __sinf(x); *c = __cosf(x); }

// Branch-free atan2 (all quadrants): odd minimax polynomial of degree 17 on [0,1] (max abs error 1.1e-7,
// checked against fp64 atan on 2e6 points) + SFU reciprocal; replaces libdevice atan2f (division slow path,
// four-way branching) in the per-surface angle-of-attack evaluation.
__device__ __forceinline__ float fw_atan2(float y, float x) {
    float ax = fabsf(x), ay = fabsf(y);
    float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    float a = mx > 0.0f ? __fdividef(mn, mx) : 0.0f;
    float q = a * a;
    float r = 0.00282363896258175373077393f;
    r = fmaf(r, q, -0.0159569028764963150024414f);
    r = fmaf(r, q, 0.0425049886107444763183594f);
    r = fmaf(r, q, -0.0748900920152664184570312f);
    r = fmaf(r, q, 0.106347933411598205566406f);
    r = fmaf(r, q, -0.142027363181114196777344f);
    r = fmaf(r, q, 0.199926957488059997558594f);
    r = fmaf(r, q, -0.333331018686294555664062f);
    r = r * q;
    r = fmaf(r, a, a);
    r = ay > ax ? FWD_HALF_PI - r : r;
    r = x < 0.0f ? FWD_PI - r : r;
    return copysignf(r, y);
}

struct Mat3 { float m[9]; };

__device__ __forceinline__ Mat3 fw_quat_mat(float x, float y, float z, float w) {
    // pybullet getMatrixFromQuaternion with s = 2/|q|^2; the state quaternion is renormalised every substep,
    // so |q|^2 = 1 to one fp32 ulp and s = 2 (no division)
    const float s = 2.0f;
    float xs = x * s, ys = y * s, zs = z * s;
    float wx = w * xs, wy = w * ys, wz = w * zs;
    float xx = x * xs, xy = x * ys, xz = x * zs;
    float yy = y * ys, yz = y * zs, zz = z * zs;
    Mat3 R;
    R.m[0] = 1.0f - (yy + zz); R.m[1] = xy - wz;          R.m[2] = xz + wy;
    R.m[3] = xy + wz;          R.m[4] = 1.0f - (xx + zz); R.m[5] = yz - wx;
    R.m[6] = xz - wy;          R.m[7] = yz + wx;          R.m[8] = 1.0f - (xx + yy);
    return R;
}

// ------------------------------------------------------------------ lifting surface (Khan & Nahon model as used by PyFlyt)
// Branch-free: the attached-flow and post-stall branches of the model share alpha_eff -> (sin, cos) ->
// Cl = CN cos - CT sin, Cd = CN sin + CT cos; only CN, CT and the |alpha_eff| in CM differ, so both are
// evaluated and selected.  That keeps all five surfaces of a thread in one straight-line block the compiler
// can interleave (ILP 5) and keeps warps convergent when only some aircraft are stalled.
// Returns the force components along the lift and forward units and the scalar pitching torque about the
// surface's torque axis (lift x fwd).
// STD (standard layout, checked on the host): forward unit = +x and lift unit = +z, or +y when LIFT_Y -- the two dot
// products are plain component picks.
__device__ __forceinline__ float fw_dot_lift(const SurfDev& sf, float vx, float vy, float vz) { return vx * sf.lift[0] + vy * sf.lift[1] + vz * sf.lift[2]; }
__device__ __forceinline__ float fw_dot_fwd(const SurfDev& sf, float vx, float vy, float vz) { return vx * sf.fwd[0] + vy * sf.fwd[1] + vz * sf.fwd[2]; }
__device__ __forceinline__ float fw_dot_lift(const SurfHot&, float, float, float) { return 0.0f; }   // standard layout: never called
__device__ __forceinline__ float fw_dot_fwd(const SurfHot&, float, float, float) { return 0.0f; }
__device__ __forceinline__ float fw_defl(const FwDev& p, const SurfDev& sf, float act) { return p.cd90_degrees ? act * sf.defl_deg : act * sf.defl_rad; }
__device__ __forceinline__ float fw_defl(const FwDev&, const SurfHot& sf, float act) { return act * sf.defl_sel; }

template <bool STD = false, bool LIFT_Y = false, class SF = SurfDev>
__device__ __forceinline__ void fw_surface(const FwDev& p, const SF& sf, float act, float vx, float vy, float vz,
                                           float& fn, float& fp, float& tq) {
    float vl = STD ? (LIFT_Y ? vy : vz) : fw_dot_lift(sf, vx, vy, vz);
    float vf = STD ? vx : fw_dot_fwd(sf, vx, vy, vz);
    float h2 = fmaf(vl, vl, vf * vf);
    float V2;
    if (STD) { const float vo = LIFT_Y ? vz : vy; V2 = p.freestream_3d ? fmaf(vo, vo, h2) : h2; }   // the third component
    else V2 = p.freestream_3d ? fmaf(vz, vz, fmaf(vy, vy, vx * vx)) : h2;
    float alpha = fw_atan2(-vl, vf);
    float inv_h = rsqrtf(fmaxf(h2, 1e-30f));

    // deflection shifts of the zero-lift and stall angles, each one FMA on the actuator state
    float a0 = fmaf(-sf.k_te, act, sf.a0_base);
    float asp = fmaf(-sf.k_shift, act, sf.asp_base);
    float asn = fmaf(-sf.k_shift, act, sf.asn_base);
    const bool nostall = (asn < alpha) && (alpha < asp);
    const bool pos = alpha > 0.0f;

    // induced angle: attached-flow value, or its stall value decaying linearly to 0 at +-pi/2
    // (numpy.interp semantics: clamped outside the two-point table)
    float aa = alpha - a0;
    float cl_lin = sf.cla * aa;
    float ast = pos ? asp : asn;
    float num = pos ? FWD_HALF_PI - alpha : alpha + FWD_HALF_PI;
    float den = pos ? FWD_HALF_PI - asp : asn + FWD_HALF_PI;
    float fac = __saturatef(__fdividef(num, den));
    float ai_stall = sf.cla_ipa * (ast - a0) * fac;
    float ai = nostall ? sf.cla_ipa * aa : ai_stall;
    float ae = aa - ai;
    float s, c;
    fw_sincos(ae, &s, &c);

    float CT_a = sf.cd0 * c;
    float CN_a = __fdividef(fmaf(CT_a, s, cl_lin), c);
    float d = fw_defl(p, sf, act);
    float cd90 = fmaf(fmaf(-4.26e-2f, d, 2.1e-1f), d, 1.98f);
    float CN_s = cd90 * s * (__fdividef(1.0f, fmaf(0.44f, fabsf(s), 0.56f)) - sf.stall_k);
    float CN = nostall ? CN_a : CN_s;
    float CT = nostall ? CT_a : 0.5f * CT_a;
    float Cl = fmaf(CN, c, -CT * s);
    float Cd = fmaf(CN, s, CT * c);
    float aem = nostall ? ae : fabsf(ae);
    // CM = -CN (0.25 - 0.175 (1 - 2 aem / pi)) = -CN (0.075 + 0.35 aem / pi); the chord is folded into the constants
    float CMc = -CN * fmaf(aem, sf.cm1c, sf.cm0c);

    // lift = Cl Q, drag = Cd Q rotated by alpha (cos = vf/h, sin = -vl/h):
    //   normal = Q (Cl vf - Cd vl) / h,  parallel = -Q (Cl vl + Cd vf) / h
    float Q = sf.qarea * V2;
    float Qi = Q * inv_h;
    fn = Qi * fmaf(Cl, vf, -Cd * vl);
    fp = -Qi * fmaf(Cl, vl, Cd * vf);
    tq = Q * CMc;
}

// ------------------------------------------------------------------ gridded wind field (wind_mode 3)
// Time: linear between slices, periodic with period nt * t_step; the stamp is the one fw_wind uses (physics step ps - 1).
__device__ __forceinline__ void fw_field_time(const FwDev& p, int ps, const float4& w0, FwFieldT& t) {
    const int stamp = ps - 1;
    t.on = stamp >= 0 && stamp >= p.wind_start_substep;
    t.sx = w0.x; t.sy = w0.y; t.sz = w0.z;
    float u = fmaf((float)stamp, p.wf_sps, w0.w * p.wf_inv_tstep);     // slices since t = 0
    u -= p.wf_nt * floorf(u * p.wf_inv_nt);
    const int nt = p.wf_n[3];
    const int i0 = min(max((int)u, 0), nt - 1);
    const int i1 = i0 + 1 < nt ? i0 + 1 : 0;
    t.wb = fminf(fmaxf(u - (float)i0, 0.0f), 1.0f);
    t.a = p.wf + (size_t)i0 * p.wf_pts;
    t.b = p.wf + (size_t)i1 * p.wf_pts;
}

// lattice coordinate along one axis: clamped to the box, cell index i0 and the step to its neighbour (0 on the last point
// or on a one-point axis: i1 = min(i0 + 1, n - 1))
__device__ __forceinline__ void fw_field_axis(float x, float org, float inv_sp, float gmax, int n, int& i0, int& di, float& f) {
    const float g = fminf(fmaxf((x - org) * inv_sp, 0.0f), gmax);
    i0 = min((int)g, n - 1);
    di = i0 + 1 < n ? 1 : 0;
    f = g - (float)i0;
}

__device__ __forceinline__ float3 fw_field_trilinear(const float4* __restrict__ s, int base, int dx, int dy, int dz, float fx,
                                                     float fy, float fz) {
    const float4 c000 = __ldg(s + base), c100 = __ldg(s + base + dx);
    const float4 c010 = __ldg(s + base + dy), c110 = __ldg(s + base + dy + dx);
    const float4 c001 = __ldg(s + base + dz), c101 = __ldg(s + base + dz + dx);
    const float4 c011 = __ldg(s + base + dz + dy), c111 = __ldg(s + base + dz + dy + dx);
    float3 r;
    {
        const float x00 = fmaf(fx, c100.x - c000.x, c000.x), x10 = fmaf(fx, c110.x - c010.x, c010.x);
        const float x01 = fmaf(fx, c101.x - c001.x, c001.x), x11 = fmaf(fx, c111.x - c011.x, c011.x);
        const float y0 = fmaf(fy, x10 - x00, x00), y1 = fmaf(fy, x11 - x01, x01);
        r.x = fmaf(fz, y1 - y0, y0);
    }
    {
        const float x00 = fmaf(fx, c100.y - c000.y, c000.y), x10 = fmaf(fx, c110.y - c010.y, c010.y);
        const float x01 = fmaf(fx, c101.y - c001.y, c001.y), x11 = fmaf(fx, c111.y - c011.y, c011.y);
        const float y0 = fmaf(fy, x10 - x00, x00), y1 = fmaf(fy, x11 - x01, x01);
        r.y = fmaf(fz, y1 - y0, y0);
    }
    {
        const float x00 = fmaf(fx, c100.z - c000.z, c000.z), x10 = fmaf(fx, c110.z - c010.z, c010.z);
        const float x01 = fmaf(fx, c101.z - c001.z, c001.z), x11 = fmaf(fx, c111.z - c011.z, c011.z);
        const float y0 = fmaf(fy, x10 - x00, x00), y1 = fmaf(fy, x11 - x01, x01);
        r.z = fmaf(fz, y1 - y0, y0);
    }
    return r;
}

// world-frame wind of the field at world point (x, y, z) for the time pair t: trilinear in space (clamped to the box) on both
// slices, linear in time -- 8 corners x 2 slices of 16-byte read-only loads
__device__ __forceinline__ float3 fw_wind_field(const FwDev& p, const FwFieldT& t, float x, float y, float z) {
    int ix, iy, iz, dx, dy, dz;
    float fx, fy, fz;
    fw_field_axis(x - t.sx, p.wf_origin[0], p.wf_inv_sp[0], p.wf_max[0], p.wf_n[0], ix, dx, fx);
    fw_field_axis(y - t.sy, p.wf_origin[1], p.wf_inv_sp[1], p.wf_max[1], p.wf_n[1], iy, dy, fy);
    fw_field_axis(z - t.sz, p.wf_origin[2], p.wf_inv_sp[2], p.wf_max[2], p.wf_n[2], iz, dz, fz);
    const int nx = p.wf_n[0], nxy = nx * p.wf_n[1];
    const int base = iz * nxy + iy * nx + ix;
    const float3 a = fw_field_trilinear(t.a, base, dx, dy * nx, dz * nxy, fx, fy, fz);
    const float3 b = fw_field_trilinear(t.b, base, dx, dy * nx, dz * nxy, fx, fy, fz);
    return make_float3(fmaf(t.wb, b.x - a.x, a.x), fmaf(t.wb, b.y - a.y, a.y), fmaf(t.wb, b.z - a.z, a.z));
}

// local airflow (body frame) of the surface with body-frame link CoM r minus the field's wind at that link CoM
__device__ __forceinline__ void fw_field_subtract(const FwDev& p, const FwFieldT& t, const EnvState& e, const float* m,
                                                  const float r[3], float& sx, float& sy, float& sz) {
    if (!t.on) return;
    const float x = e.px + m[0] * r[0] + m[1] * r[1] + m[2] * r[2];
    const float y = e.py + m[3] * r[0] + m[4] * r[1] + m[5] * r[2];
    const float z = e.pz + m[6] * r[0] + m[7] * r[1] + m[8] * r[2];
    const float3 w = fw_wind_field(p, t, x, y, z);
    sx -= m[0] * w.x + m[3] * w.y + m[6] * w.z;
    sy -= m[1] * w.x + m[4] * w.y + m[7] * w.z;
    sz -= m[2] * w.x + m[5] * w.y + m[8] * w.z;
}

// ------------------------------------------------------------------ one 240 Hz substep
// cmd: latched actuator commands [5 surfaces + motor]; wind: world-frame wind seen by the surfaces
// (already selected for this substep's time stamp); nz: N(0,1) draw for the motor noise.
//
// STD = the reference aircraft's layout, verified by derive() before a STD kernel is chosen: every surface's forward
// unit is +x; lift unit +z for surfaces 0,1,2,4 and +y for surface 3 (vertical tail); thrust along +x; the aircraft
// is symmetric about its xz plane, so the inverse spatial inertia splits into a lateral {wx, wz, vy} and a
// longitudinal {wy, vx, vz} 3x3 block.  The arithmetic is the generic path's with the structural zeros skipped.
// FIELD = gridded wind (wind_mode 3): wn* are ignored (pass 0); every surface subtracts R^T w_s from its own local airflow,
// w_s = the field at its link CoM in the world, pos + R r_s, for the time pair ft.
template <bool STD = false, bool FIELD = false>
__device__ __forceinline__ void fw_substep(const FwDev& p, EnvState& e, const float cmd[6], float wnx, float wny,
                                           float wnz, float nz, bool& contact, const FwFieldT& ft = FwFieldT()) {
    const float dt = p.dt;
    Mat3 R = fw_quat_mat(e.qx, e.qy, e.qz, e.qw);
    const float* m = R.m;
    // body-frame velocities of O (R^T v, R^T w) and the wind in the body frame
    float vbx = m[0] * (e.vx - wnx) + m[3] * (e.vy - wny) + m[6] * (e.vz - wnz);
    float vby = m[1] * (e.vx - wnx) + m[4] * (e.vy - wny) + m[7] * (e.vz - wnz);
    float vbz = m[2] * (e.vx - wnx) + m[5] * (e.vy - wny) + m[8] * (e.vz - wnz);
    float wbx = m[0] * e.wx + m[3] * e.wy + m[6] * e.wz;
    float wby = m[1] * e.wx + m[4] * e.wy + m[7] * e.wz;
    float wbz = m[2] * e.wx + m[5] * e.wy + m[8] * e.wz;

    float Fx = 0.f, Fy = 0.f, Fz = 0.f, Tx = 0.f, Ty = 0.f, Tz = 0.f;
#pragma unroll
    for (int s = 0; s < FWD_NSURF; ++s) {
        if (STD) {
            const SurfHot sf = fw_load_hot(p.hot[s]);
            e.act[s] += sf.k_act * (cmd[s] - e.act[s]);
            // local airflow at the link CoM: v_O + w x r  (wind already subtracted from v_O)
            float sx = fmaf(wby, sf.r[2], fmaf(-wbz, sf.r[1], vbx));
            float sy = fmaf(wbz, sf.r[0], fmaf(-wbx, sf.r[2], vby));
            float sz = fmaf(wbx, sf.r[1], fmaf(-wby, sf.r[0], vbz));
            if (FIELD) fw_field_subtract(p, ft, e, m, sf.r, sx, sy, sz);
            float fn, fp, tq;
            // force = lift*fn + fwd*fp at the link CoM; torque about O = fn (r x lift) + fp (r x fwd) + tq (lift x fwd)
            if (s != 3) {              // lift +z, fwd +x: ra = (ry, -rx, 0), rb = (0, rz, -ry), lift x fwd = +y
                fw_surface<true, false>(p, sf, e.act[s], sx, sy, sz, fn, fp, tq);
                Fx += fp; Fz += fn;
                Tx += sf.ra[0] * fn;
                Ty += sf.ra[1] * fn + sf.rb[1] * fp + tq;
                Tz += sf.rb[2] * fp;
            } else {                    // lift +y, fwd +x: ra = (-rz, 0, rx), rb = (0, rz, -ry), lift x fwd = -z
                fw_surface<true, true>(p, sf, e.act[s], sx, sy, sz, fn, fp, tq);
                Fx += fp; Fy += fn;
                Tx += sf.ra[0] * fn;
                Ty += sf.rb[1] * fp;
                Tz += sf.ra[2] * fn + sf.rb[2] * fp - tq;
            }
            continue;
        }
        const SurfDev& sf = p.surf[s];
        e.act[s] += sf.k_act * (cmd[s] - e.act[s]);
        float sx = fmaf(wby, sf.r[2], fmaf(-wbz, sf.r[1], vbx));
        float sy = fmaf(wbz, sf.r[0], fmaf(-wbx, sf.r[2], vby));
        float sz = fmaf(wbx, sf.r[1], fmaf(-wby, sf.r[0], vbz));
        if (FIELD) fw_field_subtract(p, ft, e, m, sf.r, sx, sy, sz);
        float fn, fp, tq;
        {
            fw_surface(p, sf, e.act[s], sx, sy, sz, fn, fp, tq);
            Fx += sf.lift[0] * fn + sf.fwd[0] * fp;
            Fy += sf.lift[1] * fn + sf.fwd[1] * fp;
            Fz += sf.lift[2] * fn + sf.fwd[2] * fp;
            Tx += sf.ra[0] * fn + sf.rb[0] * fp + sf.tq[0] * tq;
            Ty += sf.ra[1] * fn + sf.rb[1] * fp + sf.tq[1] * tq;
            Tz += sf.ra[2] * fn + sf.rb[2] * fp + sf.tq[2] * tq;
        }
    }
    // constants of the rest of the step: packed groups on the standard path, plain fields otherwise
    float k_motor_k, k_noise, k_thrust_max, k_torque_max, k_rm1, k_rm2, k_gravity, k_mass, k_com[3], k_mv, k_I[9], k_minv[18];
    if (STD) {
        const float4 q0 = p.rbk[0], q1 = p.rbk[1], q2 = p.rbk[2], q3 = p.rbk[3], q4 = p.rbk[4], q5 = p.rbk[5], q6 = p.rbk[6],
                     q7 = p.rbk[7], q8 = p.rbk[8], q9 = p.rbk[9];
        k_motor_k = q0.x; k_noise = q0.y; k_thrust_max = q0.z; k_torque_max = q0.w;
        k_rm1 = q1.x; k_rm2 = q1.y; k_gravity = q1.z; k_mass = q1.w;
        k_com[0] = q2.x; k_com[1] = q2.y; k_com[2] = q2.z; k_mv = q2.w;
        k_I[0] = q3.x; k_I[1] = q3.y; k_I[2] = q3.z; k_I[3] = q3.w; k_I[4] = q4.x; k_I[5] = q4.y; k_I[6] = q4.z; k_I[7] = q4.w;
        k_I[8] = q5.x;
        k_minv[0] = q5.y; k_minv[1] = q5.z; k_minv[2] = q5.w; k_minv[3] = q6.x; k_minv[4] = q6.y; k_minv[5] = q6.z;
        k_minv[6] = q6.w; k_minv[7] = q7.x; k_minv[8] = q7.y; k_minv[9] = q7.z; k_minv[10] = q7.w; k_minv[11] = q8.x;
        k_minv[12] = q8.y; k_minv[13] = q8.z; k_minv[14] = q8.w; k_minv[15] = q9.x; k_minv[16] = q9.y; k_minv[17] = q9.z;
    } else {
        k_motor_k = p.motor_k; k_noise = p.noise_ratio; k_thrust_max = p.thrust_max; k_torque_max = p.torque_max;
        k_rm1 = p.r_motor[1]; k_rm2 = p.r_motor[2]; k_gravity = p.gravity; k_mass = p.mass;
        k_com[0] = p.com[0]; k_com[1] = p.com[1]; k_com[2] = p.com[2]; k_mv = p.max_vel;
#pragma unroll
        for (int k = 0; k < 9; ++k) k_I[k] = p.inertia[k];
#pragma unroll
        for (int k = 0; k < 18; ++k) k_minv[k] = 0.0f;       // the generic solve below reads p.minv
    }
    {   // motor: first-order lag, multiplicative gaussian noise, thrust ~ rpm^2
        e.thr += k_motor_k * (cmd[5] - e.thr);
        e.thr += nz * e.thr * k_noise;
        float t2 = e.thr * e.thr;
        float thrust = t2 * k_thrust_max, torque = t2 * k_torque_max;
        if (STD) {                      // thrust along +x
            Fx += thrust;
            Tx += torque;
            Ty += k_rm2 * thrust;
            Tz -= k_rm1 * thrust;
        } else {
            float fx = thrust * p.thrust_unit[0], fy = thrust * p.thrust_unit[1], fz = thrust * p.thrust_unit[2];
            Fx += fx; Fy += fy; Fz += fz;
            Tx += p.r_motor[1] * fz - p.r_motor[2] * fy + torque * p.thrust_unit[0];
            Ty += p.r_motor[2] * fx - p.r_motor[0] * fz + torque * p.thrust_unit[1];
            Tz += p.r_motor[0] * fy - p.r_motor[1] * fx + torque * p.thrust_unit[2];
        }
    }
    // ground contact is detected on the pose entering the step (Bullet runs collision detection first)
    if (e.pz <= p.col_radius + p.contact_margin) {
        for (int i = 0; i < p.n_col; ++i) {
            float z = e.pz + m[6] * p.col[i][0] + m[7] * p.col[i][1] + m[8] * p.col[i][2];
            contact = contact || (z <= p.contact_margin);
        }
    }
    // gravity on every link == M g at the composite CoM; g_body = R^T (0,0,-g)
    float gx = -k_gravity * m[6], gy = -k_gravity * m[7], gz = -k_gravity * m[8];
    Fx += k_mass * gx; Fy += k_mass * gy; Fz += k_mass * gz;
    Tx += k_mass * (k_com[1] * gz - k_com[2] * gy);
    Ty += k_mass * (k_com[2] * gx - k_com[0] * gz);
    Tz += k_mass * (k_com[0] * gy - k_com[1] * gx);
    // bias terms: w x (I w) and M w x (w x c)
    float Iwx = k_I[0] * wbx + k_I[1] * wby + k_I[2] * wbz;
    float Iwy = k_I[3] * wbx + k_I[4] * wby + k_I[5] * wbz;
    float Iwz = k_I[6] * wbx + k_I[7] * wby + k_I[8] * wbz;
    float b0 = Tx - (wby * Iwz - wbz * Iwy);
    float b1 = Ty - (wbz * Iwx - wbx * Iwz);
    float b2 = Tz - (wbx * Iwy - wby * Iwx);
    float cx = wby * k_com[2] - wbz * k_com[1];
    float cy = wbz * k_com[0] - wbx * k_com[2];
    float cz = wbx * k_com[1] - wby * k_com[0];
    float b3 = Fx - k_mass * (wby * cz - wbz * cy);
    float b4 = Fy - k_mass * (wbz * cx - wbx * cz);
    float b5 = Fz - k_mass * (wbx * cy - wby * cx);
    float acc[6];
    if (STD) {
        // lateral block {0: wx, 2: wz, 4: vy} and longitudinal block {1: wy, 3: vx, 5: vz}
        acc[0] = k_minv[0] * b0 + k_minv[1] * b2 + k_minv[2] * b4;
        acc[2] = k_minv[3] * b0 + k_minv[4] * b2 + k_minv[5] * b4;
        acc[4] = k_minv[6] * b0 + k_minv[7] * b2 + k_minv[8] * b4;
        acc[1] = k_minv[9] * b1 + k_minv[10] * b3 + k_minv[11] * b5;
        acc[3] = k_minv[12] * b1 + k_minv[13] * b3 + k_minv[14] * b5;
        acc[5] = k_minv[15] * b1 + k_minv[16] * b3 + k_minv[17] * b5;
    } else {
#pragma unroll
        for (int i = 0; i < 6; ++i)
            acc[i] = p.minv[6 * i + 0] * b0 + p.minv[6 * i + 1] * b1 + p.minv[6 * i + 2] * b2 +
                     p.minv[6 * i + 3] * b3 + p.minv[6 * i + 4] * b4 + p.minv[6 * i + 5] * b5;
    }
    // to the world frame, semi-implicit Euler, Bullet's per-coordinate velocity clamp
    float awx = m[0] * acc[0] + m[1] * acc[1] + m[2] * acc[2];
    float awy = m[3] * acc[0] + m[4] * acc[1] + m[5] * acc[2];
    float awz = m[6] * acc[0] + m[7] * acc[1] + m[8] * acc[2];
    float Awx = m[0] * acc[3] + m[1] * acc[4] + m[2] * acc[5];
    float Awy = m[3] * acc[3] + m[4] * acc[4] + m[5] * acc[5];
    float Awz = m[6] * acc[3] + m[7] * acc[4] + m[8] * acc[5];
    const float mv = k_mv;
    e.wx = fminf(fmaxf(e.wx + awx * dt, -mv), mv);
    e.wy = fminf(fmaxf(e.wy + awy * dt, -mv), mv);
    e.wz = fminf(fmaxf(e.wz + awz * dt, -mv), mv);
    e.vx = fminf(fmaxf(e.vx + Awx * dt, -mv), mv);
    e.vy = fminf(fmaxf(e.vy + Awy * dt, -mv), mv);
    e.vz = fminf(fmaxf(e.vz + Awz * dt, -mv), mv);
    e.px += e.vx * dt; e.py += e.vy * dt; e.pz += e.vz * dt;
    // exponential-map quaternion update (btMultiBody::stepPositionsMultiDof).  Bullet limits the step angle to
    // pi/4; with its own +-max_vel clamp on every omega component that limiter can only fire when
    // sqrt(3)*max_vel*dt > pi/4 (quat_limiter), which the default 100 rad/s at 240 Hz never reaches.
    // Half angle h <= pi/8: sin(h)/h and cos(h) by Taylor series in h^2 (truncation < 2e-9), no SFU.
    {
        float ang2 = e.wx * e.wx + e.wy * e.wy + e.wz * e.wz;
        float scale = 1.0f;       // Bullet keeps omega unclamped in the axis but clamps the angle
        if (p.quat_limiter) {
            float ang = sqrtf(ang2);
            if (ang * dt > 0.25f * FWD_PI) {
                float lim = 0.5f * FWD_HALF_PI / dt;
                scale = ang / lim;             // axis = omega * sin(h_lim)/lim
                ang2 = lim * lim;
            }
        }
        float h2 = 0.25f * dt * dt * ang2;
        float sinc = fmaf(h2, fmaf(h2, fmaf(h2, -1.0f / 5040.0f, 1.0f / 120.0f), -1.0f / 6.0f), 1.0f);
        float cw = fmaf(h2, fmaf(h2, fmaf(h2, fmaf(h2, 1.0f / 40320.0f, -1.0f / 720.0f), 1.0f / 24.0f), -0.5f), 1.0f);
        float k = 0.5f * dt * sinc * scale;
        float ax = e.wx * k, ay = e.wy * k, az = e.wz * k;
        float nx = cw * e.qx + e.qw * ax + (ay * e.qz - az * e.qy);
        float ny = cw * e.qy + e.qw * ay + (az * e.qx - ax * e.qz);
        float nzq = cw * e.qz + e.qw * az + (ax * e.qy - ay * e.qx);
        float nw = cw * e.qw - (ax * e.qx + ay * e.qy + az * e.qz);
        float inv = rsqrtf(nx * nx + ny * ny + nzq * nzq + nw * nw);
        e.qx = nx * inv; e.qy = ny * inv; e.qz = nzq * inv; e.qw = nw * inv;
    }
    e.physics_steps += 1;
}

// wind seen by the force evaluation of physics step `ps` (cached by the state refresh of step ps-1)
__device__ __forceinline__ void fw_wind(const FwDev& p, int ps, const float4& w0, const float4& w1, float& x, float& y,
                                        float& z) {
    x = y = z = 0.0f;
    if (p.wind_mode == 0) return;
    int stamp = ps - 1;
    if (stamp < 0 || stamp < p.wind_start_substep) return;
    if (p.wind_mode == 1) { x = w0.x; y = w0.y; z = w0.z; return; }
    // sin(2 pi f t + phi) with the range reduction done on the cycle count: stamp * (f dt) cycles, minus whole turns,
    // leaves an argument in [-pi, pi] for MUFU.SIN (libdevice sinf spends ~40 instructions per substep on arguments of
    // up to 150 rad; the fp32 rounding of the argument itself, ~1e-5 rad at t = 120 s, is the same either way)
    float turns = fmaf(w0.w, 0.15915494309189535f, (float)stamp * p.gust_cyc);
    turns -= rintf(turns);
    float s = __sinf(6.283185307179586f * turns);
    x = w0.x + w1.x * s; y = w0.y + w1.y * s; z = w0.z + w1.z * s;
}

__device__ __forceinline__ void fw_map_setpoint(const FwDev& p, float roll, float pitch, float yaw, float thrust,
                                                float cmd[6]) {
    cmd[0] = p.sign_ail_l * roll;
    cmd[1] = p.sign_ail_r * roll;
    cmd[2] = p.sign_pitch * pitch;
    cmd[3] = p.sign_yaw * yaw;
    cmd[4] = 0.0f;
    cmd[5] = thrust;
}

// pybullet getEulerFromQuaternion
__device__ __forceinline__ void fw_euler(const EnvState& e, float& roll, float& pitch, float& yaw) {
    float x = e.qx, y = e.qy, z = e.qz, w = e.qw;
    float sarg = -2.0f * (x * z - w * y);
    if (sarg <= -0.99999f) { roll = 0.0f; pitch = -FWD_HALF_PI; yaw = 2.0f * atan2f(x, -y); }
    else if (sarg >= 0.99999f) { roll = 0.0f; pitch = FWD_HALF_PI; yaw = 2.0f * atan2f(-x, y); }
    else {
        roll = atan2f(2.0f * (y * z + w * x), w * w - x * x - y * y + z * z);
        pitch = asinf(sarg);
        yaw = atan2f(2.0f * (x * y + w * z), w * w + x * x - y * y - z * z);
    }
}

// flattened observation of one env into `o` (row of obs_dim floats); target rows come from the planes
__device__ __forceinline__ void fw_write_obs(const FwDev& p, const FwPlanes& pl, const EnvState& e, int i, int obs_tidx,
                                             float a0, float a1, float a2, float a3, float* o, bool duck_row = false,
                                             float dkx = 0.f, float dky = 0.f, float dkz = 0.f) {
    Mat3 R = fw_quat_mat(e.qx, e.qy, e.qz, e.qw);
    const float* m = R.m;
    float roll, pitch, yaw;
    fw_euler(e, roll, pitch, yaw);
    int k = 0;
    o[k++] = m[0] * e.wx + m[3] * e.wy + m[6] * e.wz;
    o[k++] = m[1] * e.wx + m[4] * e.wy + m[7] * e.wz;
    o[k++] = m[2] * e.wx + m[5] * e.wy + m[8] * e.wz;
    if (p.angle_repr == 0) { o[k++] = roll; o[k++] = pitch; o[k++] = yaw; }
    else {
        float sr, cr, sp, cp, sy, cy;
        sincosf(0.5f * roll, &sr, &cr); sincosf(0.5f * pitch, &sp, &cp); sincosf(0.5f * yaw, &sy, &cy);
        o[k++] = sr * cp * cy - cr * sp * sy;
        o[k++] = cr * sp * cy + sr * cp * sy;
        o[k++] = cr * cp * sy - sr * sp * cy;
        o[k++] = cr * cp * cy + sr * sp * sy;
    }
    o[k++] = m[0] * e.vx + m[3] * e.vy + m[6] * e.vz;
    o[k++] = m[1] * e.vx + m[4] * e.vy + m[7] * e.vz;
    o[k++] = m[2] * e.vx + m[5] * e.vy + m[8] * e.vz;
    o[k++] = e.px; o[k++] = e.py; o[k++] = e.pz;
    o[k++] = a0; o[k++] = a1; o[k++] = a2; o[k++] = a3;
#pragma unroll
    for (int s = 0; s < FWD_NSURF; ++s) o[k++] = e.act[s];
    o[k++] = e.thr;
    for (int r = 0; r < p.context_len; ++r) {
        int t = obs_tidx + r;
        if (t < p.num_targets) {
            float dx = pl.targets[(size_t)(t * 3 + 0) * p.n + i] - e.px;
            float dy = pl.targets[(size_t)(t * 3 + 1) * p.n + i] - e.py;
            float dz = pl.targets[(size_t)(t * 3 + 2) * p.n + i] - e.pz;
            o[k++] = m[0] * dx + m[3] * dy + m[6] * dz;
            o[k++] = m[1] * dx + m[4] * dy + m[7] * dz;
            o[k++] = m[2] * dx + m[5] * dy + m[8] * dz;
        } else if (duck_row && t == p.num_targets) {
            // ObjLock: the duck rides as one extra target row after the remaining waypoints (objlock_env.py:232-246)
            float dx = dkx - e.px, dy = dky - e.py, dz = dkz - e.pz;
            o[k++] = m[0] * dx + m[3] * dy + m[6] * dz;
            o[k++] = m[1] * dx + m[4] * dy + m[7] * dz;
            o[k++] = m[2] * dx + m[5] * dy + m[8] * dz;
        } else { o[k++] = 0.0f; o[k++] = 0.0f; o[k++] = 0.0f; }
    }
}

// FixedwingLowLevelEnv._compute_obs (fixedwing_lowlevel_env.py:143-156): Aviary.state(0) flattened
// [ang_vel_body, euler, lin_vel_body, lin_pos], the previous action (6) and the target [psi_ref, h_ref, V_ref];
// also returns yaw and the body-frame speed the reward needs
__device__ __forceinline__ void fw_write_obs_lowlevel(const FwPlanes& pl, const EnvState& e, int i, int n, const float a[6],
                                                      float* o, float& yaw_out, float& speed_out, float tref[3]) {
    Mat3 R = fw_quat_mat(e.qx, e.qy, e.qz, e.qw);
    const float* m = R.m;
    float roll, pitch, yaw;
    fw_euler(e, roll, pitch, yaw);
    const float vbx = m[0] * e.vx + m[3] * e.vy + m[6] * e.vz;
    const float vby = m[1] * e.vx + m[4] * e.vy + m[7] * e.vz;
    const float vbz = m[2] * e.vx + m[5] * e.vy + m[8] * e.vz;
    tref[0] = pl.targets[(size_t)0 * n + i]; tref[1] = pl.targets[(size_t)1 * n + i]; tref[2] = pl.targets[(size_t)2 * n + i];
    yaw_out = yaw;
    speed_out = sqrtf(vbx * vbx + vby * vby + vbz * vbz);
    if (o == nullptr) return;
    int k = 0;
    o[k++] = m[0] * e.wx + m[3] * e.wy + m[6] * e.wz;
    o[k++] = m[1] * e.wx + m[4] * e.wy + m[7] * e.wz;
    o[k++] = m[2] * e.wx + m[5] * e.wy + m[8] * e.wz;
    o[k++] = roll; o[k++] = pitch; o[k++] = yaw;
    o[k++] = vbx; o[k++] = vby; o[k++] = vbz;
    o[k++] = e.px; o[k++] = e.py; o[k++] = e.pz;
#pragma unroll
    for (int c = 0; c < 6; ++c) o[k++] = a[c];
    o[k++] = tref[0]; o[k++] = tref[1]; o[k++] = tref[2];
}

// end_reset: warmup_substeps substeps at zero setpoint.  Kept out of line: it is the rare path (only when a wind
// field acts during the warm-up, otherwise resets copy the cached result) and inlining it would duplicate
// the whole substep body and double the kernel's instruction-cache footprint.
// One substep under the wind of the env's mode: the uniform wind of fw_wind, or (FIELD) the gridded field per surface.
template <bool STD, bool FIELD>
__device__ __forceinline__ void fw_substep_wind(const FwDev& p, EnvState& e, const float cmd[6], const float4& w0,
                                                const float4& w1, float nz, bool& contact) {
    if (FIELD) {
        FwFieldT ft;
        fw_field_time(p, e.physics_steps, w0, ft);
        fw_substep<STD, true>(p, e, cmd, 0.0f, 0.0f, 0.0f, nz, contact, ft);
    } else {
        float wx, wy, wz;
        fw_wind(p, e.physics_steps, w0, w1, wx, wy, wz);
        fw_substep<STD>(p, e, cmd, wx, wy, wz, nz, contact);
    }
}

template <bool FIELD = false>
static __device__ __noinline__ void fw_warmup_loop(const FwDev& p, EnvState& e, float4 w0, float4 w1, int nsub) {
    float cmd[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    bool contact = false;
    if (FIELD) {
        if (p.std_geom) {
            for (int k = 0; k < nsub; ++k) fw_substep_wind<true, true>(p, e, cmd, w0, w1, 0.0f, contact);
            return;
        }
        for (int k = 0; k < nsub; ++k) fw_substep_wind<false, true>(p, e, cmd, w0, w1, 0.0f, contact);
        return;
    }
    if (p.std_geom) {                // same choice of physics path as the step kernels (uniform branch)
        for (int k = 0; k < nsub; ++k) {
            float wx, wy, wz;
            fw_wind(p, e.physics_steps, w0, w1, wx, wy, wz);
            fw_substep<true>(p, e, cmd, wx, wy, wz, 0.0f, contact);   // throttle is 0 during warm-up: noise term is 0
        }
        return;
    }
    for (int k = 0; k < nsub; ++k) {
        float wx, wy, wz;
        fw_wind(p, e.physics_steps, w0, w1, wx, wy, wz);
        fw_substep(p, e, cmd, wx, wy, wz, 0.0f, contact);
    }
}

// ---- reset pieces (begin_reset / WaypointHandler.reset / end_reset), composed per task by the kernels
// FIELD: w0 = (spatial shift xyz ~ U(shift_lo, shift_hi), time offset ~ U(0, nt t_step) when randomize_time), w1 = 0; both
// zero without wind_randomize.  Same Philox stream and counter as the uniform modes' draws.
template <bool FIELD = false>
__device__ __forceinline__ void fw_reset_begin(const FwDev& p, const FwPlanes& pl, EnvState& e, int i, uint32_t gid,
                                               uint32_t episode, float4& w0, float4& w1) {
    e.episode = episode;
    e.step_count = 0;
    e.tidx = 0;
    if (FIELD) {
        w0 = make_float4(0.f, 0.f, 0.f, 0.f);
        w1 = w0;
        if (p.wind_randomize) {
            const uint4 r0 = fw_philox(p.seed_lo, p.seed_hi, gid, episode, 0u, FWD_STREAM_WIND);
            w0.x = p.wf_shift_lo[0] + fw_u01(r0.x) * (p.wf_shift_hi[0] - p.wf_shift_lo[0]);
            w0.y = p.wf_shift_lo[1] + fw_u01(r0.y) * (p.wf_shift_hi[1] - p.wf_shift_lo[1]);
            w0.z = p.wf_shift_lo[2] + fw_u01(r0.z) * (p.wf_shift_hi[2] - p.wf_shift_lo[2]);
            if (p.wf_rand_time) w0.w = fw_u01(r0.w) * p.wf_period;
        }
        pl.w0[i] = w0; pl.w1[i] = w1;
    }
    w0 = FIELD ? w0 : make_float4(p.wind_base[0], p.wind_base[1], p.wind_base[2], p.gust_phase);
    w1 = FIELD ? w1 : make_float4(p.gust_amp[0], p.gust_amp[1], p.gust_amp[2], 0.0f);
    if (!FIELD && p.wind_mode != 0) {
        if (p.wind_randomize) {
            uint4 r0 = fw_philox(p.seed_lo, p.seed_hi, gid, episode, 0u, FWD_STREAM_WIND);
            uint4 r1 = fw_philox(p.seed_lo, p.seed_hi, gid, episode, 1u, FWD_STREAM_WIND);
            w0.x = p.wind_base_lo[0] + fw_u01(r0.x) * (p.wind_base_hi[0] - p.wind_base_lo[0]);
            w0.y = p.wind_base_lo[1] + fw_u01(r0.y) * (p.wind_base_hi[1] - p.wind_base_lo[1]);
            w0.z = p.wind_base_lo[2] + fw_u01(r0.z) * (p.wind_base_hi[2] - p.wind_base_lo[2]);
            if (p.wind_mode == 2) {
                w1.x = p.gust_amp_lo[0] + fw_u01(r1.x) * (p.gust_amp_hi[0] - p.gust_amp_lo[0]);
                w1.y = p.gust_amp_lo[1] + fw_u01(r1.y) * (p.gust_amp_hi[1] - p.gust_amp_lo[1]);
                w1.z = p.gust_amp_lo[2] + fw_u01(r1.z) * (p.gust_amp_hi[2] - p.gust_amp_lo[2]);
                if (p.wind_rand_phase) w0.w = 2.0f * FWD_PI * fw_u01(r0.w);
            }
        }
        pl.w0[i] = w0; pl.w1[i] = w1;
    }
    e.px = p.start_pos[0]; e.py = p.start_pos[1]; e.pz = p.start_pos[2];
    e.qx = 0.f; e.qy = 0.f; e.qz = 0.f; e.qw = 1.f;
    e.vx = p.start_vel[0]; e.vy = p.start_vel[1]; e.vz = p.start_vel[2];
    e.wx = e.wy = e.wz = 0.f;
#pragma unroll
    for (int s = 0; s < FWD_NSURF; ++s) e.act[s] = 0.f;
    e.thr = 0.f;
    e.physics_steps = 0;
    e.new_dist = 0.0f;
}

// WaypointHandler.reset: polar sampling of every target into the planes
__device__ __forceinline__ void fw_sample_targets(const FwDev& p, const FwPlanes& pl, int i, uint32_t gid, uint32_t episode) {
    if (p.task == 3) {
        // FixedwingLowLevelEnv.reset (fixedwing_lowlevel_env.py:87-91): psi_ref ~ U(-pi, pi), h_ref ~ U(5, 20),
        // V_ref ~ U(10, 20); the tracked reference rides in target slot 0
        uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid, episode, 0u, FWD_STREAM_TARGETS);
        pl.targets[(size_t)0 * p.n + i] = -FWD_PI + 2.0f * FWD_PI * fw_u01(r.x);
        pl.targets[(size_t)1 * p.n + i] = 5.0f + 15.0f * fw_u01(r.y);
        pl.targets[(size_t)2 * p.n + i] = 10.0f + 10.0f * fw_u01(r.z);
        return;
    }
    for (int t = 0; t < p.num_targets; ++t) {
        uint4 r = fw_philox(p.seed_lo, p.seed_hi, gid, episode, (uint32_t)t, FWD_STREAM_TARGETS);
        float st, ct, sp, cp;
        sincospif(2.0f * fw_u01(r.x), &st, &ct);
        sincospif(2.0f * fw_u01(r.y), &sp, &cp);
        float dist = 1.0f + fw_u01(r.z) * (p.spawn_size * 0.9f - 1.0f);
        float x = dist * sp * ct, y = dist * sp * st, z = fabsf(dist * cp);
        z = z > p.min_height ? z : p.min_height;
        pl.targets[(size_t)(t * 3 + 0) * p.n + i] = x;
        pl.targets[(size_t)(t * 3 + 1) * p.n + i] = y;
        pl.targets[(size_t)(t * 3 + 2) * p.n + i] = z;
    }
}

// nsub warm-up substeps at zero setpoint (end_reset); copies the cached result when it is valid
template <bool FIELD = false>
__device__ __forceinline__ void fw_warm(const FwDev& p, EnvState& e, const float4& w0, const float4& w1, int nsub,
                                        bool allow_cache) {
    if (allow_cache && p.warm_cached && nsub == p.warmup_substeps) {
        e.px = p.warm[0]; e.py = p.warm[1]; e.pz = p.warm[2];
        e.qx = p.warm[3]; e.qy = p.warm[4]; e.qz = p.warm[5]; e.qw = p.warm[6];
        e.vx = p.warm[7]; e.vy = p.warm[8]; e.vz = p.warm[9];
        e.wx = p.warm[10]; e.wy = p.warm[11]; e.wz = p.warm[12];
#pragma unroll
        for (int s = 0; s < FWD_NSURF; ++s) e.act[s] = p.warm[13 + s];
        e.thr = p.warm[18];
        e.physics_steps = p.warmup_substeps;
    } else if (nsub > 0) {
        EnvState tmp = e;          // only this copy is address-taken (local memory); `e` stays in registers
        fw_warmup_loop<FIELD>(p, tmp, w0, w1, nsub);
        e = tmp;
    }
}

__device__ __forceinline__ void fw_reset_finish(const FwDev& p, const FwPlanes& pl, EnvState& e, int i) {
    e.new_dist = 0.0f;
    if (p.task != 0 && p.task != 3 && p.num_targets > 0) {
        float dx = pl.targets[(size_t)0 * p.n + i] - e.px;
        float dy = pl.targets[(size_t)1 * p.n + i] - e.py;
        float dz = pl.targets[(size_t)2 * p.n + i] - e.pz;
        e.new_dist = sqrtf(dx * dx + dy * dy + dz * dz);
    }
}

// begin_reset/end_reset for the physics-only and Waypoints tasks
template <bool FIELD = false>
__device__ __forceinline__ void fw_reset_env(const FwDev& p, const FwPlanes& pl, EnvState& e, int i, uint32_t gid,
                                             uint32_t episode) {
    float4 w0, w1;
    fw_reset_begin<FIELD>(p, pl, e, i, gid, episode, w0, w1);
    if (p.task != 0) fw_sample_targets(p, pl, i, gid, episode);
    fw_warm<FIELD>(p, e, w0, w1, p.warmup_substeps, true);
    fw_reset_finish(p, pl, e, i);
}

// Non-finite-state guard (SURVEY section 5, failure detection): true when every state float is finite.  The reference
// swallows simulator exceptions (fixedwing_waypoint_objlock_env.py:401,449,502) and has no such check; here a poisoned
// env is flagged (FW_FLAG_FAULT), counted in stats[8] and force-reset instead of spreading NaNs into the running
// observation moments of the PPO loop.  One add chain + one compare per agent step.
__device__ __forceinline__ bool fw_state_finite(const EnvState& e) {
    float s = ((e.px + e.py) + (e.pz + e.qx)) + ((e.qy + e.qz) + (e.qw + e.vx)) + ((e.vy + e.vz) + (e.wx + e.wy)) +
              ((e.wz + e.thr) + (e.act[0] + e.act[1])) + ((e.act[2] + e.act[3]) + e.act[4]);
    return fabsf(s) < 3.0e38f;            // false for NaN and +-inf
}

__device__ __forceinline__ void fw_load(const FwPlanes& pl, int i, EnvState& e) {
    float4 a = pl.s0[i], b = pl.s1[i], c = pl.s2[i], d = pl.s3[i], f = pl.s4[i];
    int4 g = pl.s5[i];
    e.px = a.x; e.py = a.y; e.pz = a.z; e.thr = a.w;
    e.qx = b.x; e.qy = b.y; e.qz = b.z; e.qw = b.w;
    e.vx = c.x; e.vy = c.y; e.vz = c.z; e.act[0] = c.w;
    e.wx = d.x; e.wy = d.y; e.wz = d.z; e.act[1] = d.w;
    e.act[2] = f.x; e.act[3] = f.y; e.act[4] = f.z; e.new_dist = f.w;
    e.step_count = g.x; e.physics_steps = g.y; e.episode = (uint32_t)g.z; e.tidx = g.w;
}

__device__ __forceinline__ void fw_store(const FwPlanes& pl, int i, const EnvState& e) {
    pl.s0[i] = make_float4(e.px, e.py, e.pz, e.thr);
    pl.s1[i] = make_float4(e.qx, e.qy, e.qz, e.qw);
    pl.s2[i] = make_float4(e.vx, e.vy, e.vz, e.act[0]);
    pl.s3[i] = make_float4(e.wx, e.wy, e.wz, e.act[1]);
    pl.s4[i] = make_float4(e.act[2], e.act[3], e.act[4], e.new_dist);
    pl.s5[i] = make_int4(e.step_count, e.physics_steps, (int)e.episode, e.tidx);
}
