/*
 * fwsim.h -- C ABI of libfwsim.so, the B200-native batched fixed-wing simulator.
 *
 * The reference (WdBlink/pyflyt-drone) is pure Python and has no FFI: its replaceable seams for this path are
 *   - stable_baselines3 SubprocVecEnv([make_env(i) ...])   train/train_Fixedwing_Waypoints_v3.py:251
 *                                                          train/train_Fixedwing_Waypoints_ObjLock.py:306
 *   - gymnasium Env reset()/step()                         envs/fixedwing_envs/fixedwing_base_env.py:175-195,314-348
 * This header is the boundary added beneath those seams; each entry point names the reference interface it
 * replaces.  The Python host side (pyflyt_drone_b200/vec_env.py, gym_env.py) binds it with ctypes; the stub a
 * reference maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions: every function returns 0 on success and a negative FW_E* code on failure (never throws);
 * fw_last_error() gives a thread-local message.  The caller owns every I/O buffer; the library owns the
 * per-env SoA state in HBM and frees it in fw_destroy().  All device work is enqueued on the caller's
 * stream (`stream` is a cudaStream_t passed as void*, NULL = legacy default stream) with no implicit
 * device synchronisation, except the *_host entry points which are synchronous by contract.
 * A handle is not thread-safe; distinct handles (one per GPU) are independent.
 */
#ifndef FWSIM_H
#define FWSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FW_ABI_VERSION 11

#define FW_NSURF 5            /* cmd order: left aileron, right aileron, h-tail, v-tail, main wing */
#define FW_MAX_TARGETS 16
#define FW_MAX_COL 16
#define FW_MAX_OBST 32
#define FW_MAX_HIST 4            /* duck-only task: frames of vision history in the observation */

/* error codes */
#define FW_OK 0
#define FW_EINVAL (-1)
#define FW_ECUDA (-2)
#define FW_ENOMEM (-3)
#define FW_ESTATE (-4)

/* per-env flag byte written by fw_step: info dict of the reference env packed into bits
 * (fixedwing_base_env.py:212-215,296-312; fixedwing_waypoint_objlock_env.py:180-181,336-337) */
#define FW_FLAG_TERM      1   /* termination */
#define FW_FLAG_TRUNC     2   /* truncation */
#define FW_FLAG_COLLISION 4   /* info["collision"] */
#define FW_FLAG_OOB       8   /* info["out_of_bounds"] */
#define FW_FLAG_COMPLETE  16  /* info["env_complete"] */
#define FW_FLAG_STRIKE    32  /* info["duck_strike"] */
#define FW_FLAG_FAULT     64  /* no reference counterpart: the env's state went non-finite; it was terminated with reward 0,
                               * counted (fw_fault_count) and reset, and its terminal observation is the first observation
                               * of the new episode.  The reference swallows simulator exceptions instead
                               * (fixedwing_waypoint_objlock_env.py:401,449,502). */

#define FW_TASK_PHYSICS   0   /* dynamics + ground/dome termination, no observation (BASELINE config 2) */
#define FW_TASK_WAYPOINTS 1   /* PyFlyt/Fixedwing-Waypoints-v3 + FlattenWaypointEnv */
#define FW_TASK_OBJLOCK   2   /* FixedwingWaypointObjLockEnv + FlattenWaypointEnv */
#define FW_TASK_LOWLEVEL  3   /* FixedwingLowLevelEnv (envs/fixedwing_envs/fixedwing_lowlevel_env.py) */
#define FW_TASK_DUCK      4   /* FixedwingObjLockEnv + FlattenObjLockEnv (envs/fixedwing_objlock_env.py, flatten_objlock_env.py) */
#define FW_TASK_HIGHLEVEL 5   /* the Waypoints episode of task 1 flown through a frozen low-level tracker (fw_set_tracker) */

/* Everything the kernels need to know about the aircraft and the task.  Raw physical parameters only;
 * derived constants are computed inside fw_create. */
typedef struct FwConfig {
    /* lifting surfaces -- my_models/fixedwing/fixewing.yaml:8-71 */
    double cl_alpha_2d[FW_NSURF], chord[FW_NSURF], span[FW_NSURF], flap_to_chord[FW_NSURF], eta[FW_NSURF];
    double alpha0_base_deg[FW_NSURF], stall_p_base_deg[FW_NSURF], stall_n_base_deg[FW_NSURF];
    double cd0[FW_NSURF], defl_limit_deg[FW_NSURF], surf_tau[FW_NSURF];
    double lift_unit[FW_NSURF][3], fwd_unit[FW_NSURF][3], r_surf[FW_NSURF][3];
    /* motor -- fixewing.yaml:1-6 */
    double total_thrust, thrust_coef, torque_coef, noise_ratio, motor_tau;
    double r_motor[3], thrust_unit[3];
    /* composite rigid body at the base-link CoM (from the URDF; see pyflyt_drone_b200/aircraft.py) */
    double mass, com[3], inertia_o[9];
    double col_pts[FW_MAX_COL][3];
    double contact_margin;
    /* simulator rates (PyFlyt Aviary: physics 240 Hz, control 120 Hz; env: agent_hz 30) */
    double dt, gravity, rho, max_coord_vel;
    /* upstream conventions that cannot be verified offline (SURVEY.md appendix B) */
    double ail_left_sign, ail_right_sign, pitch_sign, yaw_sign;
    /* env */
    double goal_reach, dome, spawn_size, min_height;
    double start_pos[3], start_vel[3];
    /* wind -- fixedwing_base_env.py:108-173, envs/utils.py:141-218 */
    double wind_base[3], wind_base_lo[3], wind_base_hi[3];
    double gust_amp[3], gust_amp_lo[3], gust_amp_hi[3];
    double gust_freq, gust_phase;
    /* objlock -- fixedwing_waypoint_objlock_env.py:42-168 */
    double obst_radius, obst_h_lo, obst_h_hi, obst_safe, obst_scale, obst_max_pen;
    double strike_dist, strike_reward, lock_step_reward, approach_scale, switch_min_area;
    double duck_radius, cam_offset[3], cam_near, cam_far;
    /* duck-only task -- envs/fixedwing_objlock_env.py:37-118.  cam_tilt_deg = camera_angle_degrees ([UP-RECALL] rotation
     * about body +y, positive = nose-down); the rest are the visual-shaping reward constants of :71-79 */
    double cam_tilt_deg, duck_dist_scale, lock_center_radius, centering_scale, visible_step_reward, area_reward_scale;
    double lock_lost_penalty, approach_clip;

    int32_t n_col;
    int32_t physics_per_control, substeps_per_inner, inner_per_step, warmup_inner;
    int32_t freestream_3d, cd90_degrees;
    int32_t task;   /* 0 physics only, 1 Waypoints-v3, 2 Waypoint+ObjLock, 3 low-level tracking (FixedwingLowLevelEnv:
                     * 21-float obs, 6-channel action, one Aviary.step per env step, truncation at step_count >= max_steps),
                     * 4 duck-only lock/strike (FixedwingObjLockEnv: attitude + target_vector + 9*history (+4 deltas) obs),
                     * 5 high-level waypoints (task 1 through a frozen low-level tracker, fw_set_tracker) */
    int32_t num_targets, sparse_reward, angle_repr, max_steps, context_len;
    int32_t early_return_on_crash, complete_truncates;
    int32_t wind_mode, wind_randomize, wind_rand_phase, wind_start_substep;   /* wind_mode: 0 off, 1 constant, 2 gust_sine,
                                                                              * 3 gridded field (fw_set_wind_field) */
    int32_t num_obstacles, cam_interval_substeps, lock_hold_steps, switch_min_seen, cam_res;
    int32_t force_generic_kernel;   /* 1 = never pick the kernels specialised for the standard aircraft layout (testing) */
    int32_t cam_mode;               /* 0 tracking chase camera (looks at the aircraft from cam_offset), 1 fixed camera at
                                     * cam_offset looking along body x tilted by cam_tilt_deg (is_tracking_camera = False) */
    int32_t vision_hist_len;        /* duck_vision_history_len, 1..FW_MAX_HIST (task 4) */
    int32_t vision_use_deltas;      /* duck_vision_use_deltas (task 4) */
    int32_t lock_decay_steps;       /* duck_lock_decay_steps (task 4) */
    int32_t packed_pairs;           /* 1 = tasks 0/1/3 on the standard layout step TWO envs per thread on the packed fp32x2
                                     * instructions of sm_100a (csrc/fw_pack.cuh).  Opt-in: measured slower than the one-env
                                     * kernels on B200 (profiles/r2_k1_packed.md); results agree to fp32 rounding. */
} FwConfig;

/* Host-side view of the per-env state for parity injection / inspection.  Any pointer may be NULL
 * (that field is skipped).  Arrays are row-major [n_envs, k] in HOST memory. */
typedef struct FwStateHost {
    float* pos;          /* [N,3] world */
    float* quat;         /* [N,4] x,y,z,w body->world */
    float* vel;          /* [N,3] world */
    float* omega;        /* [N,3] world */
    float* act;          /* [N,6] five surface actuations + throttle */
    float* targets;      /* [N,num_targets,3] full original list */
    int32_t* target_idx; /* [N] index of the current target (== num reached) */
    int32_t* step_count; /* [N] */
    int32_t* physics_steps; /* [N] */
    uint32_t* episode;   /* [N] */
    float* new_dist;     /* [N] WaypointHandler.new_distance */
    float* wind;         /* [N,7] base xyz, gust amp xyz, phase.  wind_mode 3 (gridded field): the episode's spatial shift xyz
                          * (metres; the field is sampled at position - shift), 0, 0, 0, time offset (seconds) */
    /* ObjLock tasks (2 and 4) only (ignored otherwise) */
    float* duck;         /* [N,3] duck position */
    float* obst;         /* [N,FW_MAX_OBST,3] cylinders x, y, height (first n_obst rows valid) */
    float* ol_f;         /* [N,12] last cx,cy,area,depth | frame cx,cy,area,depth | frame dL,dC,dR | prev_est_dist */
    int32_t* ol_i;       /* [N,9] duck_phase, has_prev, post_waypoints, cam_valid, frame_visible,
                                  seen_consecutive (task 4: _vision_history_filled), lock_steps, steps_since_seen, n_obst */
    float* vis_hist;     /* task 4: [N, FW_MAX_HIST*9 + 4] vision history rows (newest first; rows >= vision_hist_len unused)
                                  followed by the four delta features */
} FwStateHost;

typedef struct FwSim* fw_handle;

/* Gridded wind field (FwConfig.wind_mode = 3): a regular lattice of world-frame (ENU) wind vectors, nx * ny * nz points from
 * `origin` with `spacing` metres along world x, y, z, and nt time slices t_step seconds apart.  The step kernels evaluate it at
 * every lifting surface's link CoM in the world (pos + R r_surf[s]) on every physics substep: trilinear in space with
 * coordinates clamped to the box (a one-point axis is constant), linear in time and periodic with period nt * t_step (nt = 1 is
 * a static field).  Time and gating are those of the uniform modes: physics step ps sees t = (ps - 1) dt + the episode's time
 * offset, from wind_start_substep on.  With FwConfig.wind_randomize every reset draws a spatial shift ~ U(shift_lo, shift_hi)
 * (the field is sampled at position - shift) and, when randomize_time is set, a time offset ~ U(0, nt * t_step); both come
 * from the Philox stream of the other modes' wind draws (index 0), so they do not depend on how envs are sharded.
 * Replaces: Aviary.register_wind_field_function(f) with f(time_s, positions[n,3]) -> [n,3], sampled on the lattice. */
typedef struct FwWindField {
    const float* values;     /* HOST [nt][nz][ny][nx][3] float32, m/s; copied by fw_set_wind_field */
    int32_t nx, ny, nz, nt;  /* each >= 1; nx * ny * nz * nt < 2^31 */
    double origin[3];        /* world position of lattice point (0, 0, 0), metres */
    double spacing[3];       /* > 0, metres */
    double t_step;           /* > 0, seconds between slices (any positive value when nt = 1) */
    double shift_lo[3], shift_hi[3];   /* per-episode spatial shift range (wind_randomize), metres */
    int32_t randomize_time;  /* 1: per-episode time offset ~ U(0, nt * t_step) (wind_randomize) */
    int32_t _pad;
} FwWindField;

int fw_abi_version(void);
const char* fw_last_error(void);
int fw_config_size(void);

/* Replaces: SubprocVecEnv([make_env(rank, seed) ...]) construction + the Aviary/URDF load of every worker
 * (train_Fixedwing_Waypoints_v3.py:82-121,251).  env_id0 is the global id of env 0 (multi-GPU sharding:
 * rank r owns [r*N, (r+1)*N); the RNG is keyed by the global id so results do not depend on the split). */
int fw_create(const FwConfig* cfg, int32_t n_envs, int32_t device, uint64_t seed, uint32_t env_id0, fw_handle* out);
int fw_destroy(fw_handle h);
/* Install the gridded wind field of a wind_mode 3 handle (see FwWindField).  fw_create with wind_mode 3 allocates the batch but
 * defers its first reset to this call; step, reset and rollout entry points return FW_ESTATE until it has run.  Synchronous and
 * one-shot: the values are validated (finite), uploaded to handle-owned device memory and the batch is reset; a second call
 * returns FW_ESTATE, a handle of another wind mode FW_EINVAL.  The field stays fixed for the handle's lifetime (fw_destroy frees
 * it), so every launch and CUDA graph sees the same field. */
int fw_set_wind_field(fw_handle h, const FwWindField* field);

/* High-level waypoints (FwConfig.task = 5): the hierarchical flow the reference starts in train/train_highlevel_cmd.py and
 * examples/lowlevel.py.  Everything is task 1 (Waypoints: targets, reward, termination, flags, the 28/29-float observation
 * with the agent's action in slots 12-15, reset and wind) except how the action reaches the aircraft.  The agent's action
 * a in R^4 is a command
 *     psi_ref = atan2(a1, a0)       (a direction vector: no wrap at +-pi; atan2(0, 0) = 0)
 *     h_ref   = h_lo + (clamp(a2, -1, 1) + 1) / 2 * (h_hi - h_lo)
 *     V_ref   = v_lo + (clamp(a3, -1, 1) + 1) / 2 * (v_hi - v_lo)
 * and each of the inner_per_step inner iterations (120 Hz) is one decision of a frozen low-level tracker followed by one
 * Aviary.step: the tracker sees task 3's 21-float observation with [psi_ref, h_ref, V_ref] as its target and its own
 * previous action (per-env state, zero after a reset, carried across agent steps), normalised by its frozen VecNormalize
 * statistics ((x - mean) / sqrt(var + 1e-8) clipped to +-clip_obs); its policy tower's mean, clipped to [-1, 1], is the
 * six-channel mode -1 command (the arithmetic of ppo_policy_forward_a with deterministic = 1, bit for bit).
 * The ranges default to task 3's reference distribution: h in [5, 20] m, V in [10, 20] m/s. */
typedef struct FwTracker {
    const float* params;      /* HOST: the flat parameter vector of include/fwppo.h for (obs 21, action 6),
                               * ppo_param_count_a(21, 6) floats; only the policy tower is read */
    const double* obs_mean;   /* HOST [21] VecNormalize obs_rms.mean, or NULL (un-normalised tracker) */
    const double* obs_var;    /* HOST [21] obs_rms.var (>= 0), NULL exactly when obs_mean is */
    double clip_obs;          /* > 0 */
    double h_range[2];        /* altitude command range, metres, lo < hi */
    double v_range[2];        /* airspeed command range, m/s, lo < hi */
} FwTracker;

/* Install the tracker of a task 5 handle.  fw_create with task 5 allocates the batch but defers its first reset to this call
 * (after fw_set_wind_field as well, for a wind_mode 3 handle: whichever of the two comes last runs it); step, reset and
 * observe entry points return FW_ESTATE until then.  Synchronous and one-shot: the descriptor is validated (finite values,
 * var >= 0, lo < hi, clip_obs > 0) before the device is touched, then copied to handle-owned device memory; a second call
 * returns FW_ESTATE, a handle of another task FW_EINVAL.  fw_rollout_random and fw_render return FW_EINVAL for task 5. */
int fw_set_tracker(fw_handle h, const FwTracker* tracker);
/* The tracker's previous action of every env, HOST [N, 6] (parity injection / inspection; synchronous). */
int fw_get_tracker_state(fw_handle h, float* prev_host);
int fw_set_tracker_state(fw_handle h, const float* prev_host);
/* Opt-in: obs_dev = device [N, 21] floats (NULL clears it).  Every step enqueued while it is set writes the raw (un-normalised)
 * tracker observation of each env's last tracker decision of that step; nothing is written while it is NULL. */
int fw_set_tracker_obs_buffer(fw_handle h, float* obs_dev);
int fw_num_envs(fw_handle h);
int fw_obs_dim(fw_handle h);
/* action width: 4 ([roll, pitch, yaw, thrust], Fixedwing mode 0) or 6 for task 3, the low-level env
 * ([left ail, right ail, h-tail, v-tail, main wing, thrust], mode -1; envs/fixedwing_envs/fixedwing_lowlevel_env.py) */
int fw_act_dim(fw_handle h);

/* Replaces: VecEnv.reset() -> env.reset(seed=seed+rank) of every worker (fixedwing_base_env.py:193-257).
 * mask_dev: optional device bytes [N], non-zero = reset that env; NULL = all.  obs_dev: [N, obs_dim] f32 or NULL. */
int fw_reset(fw_handle h, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* Replaces: VecEnv.step_async/step_wait -> FlattenWaypointEnv.step -> FixedwingBaseEnv.step
 * (fixedwing_base_env.py:314-348, flatten_waypoint_env.py:52-72) plus the SubprocVecEnv worker's
 * reset-on-done.  act_dev [N,fw_act_dim] f32 in [-1,1]; obs_dev [N,obs_dim]; rew_dev [N]; flags_dev [N] bytes;
 * term_obs_dev [N,obs_dim] or NULL (rows of done envs receive info["terminal_observation"]). */
int fw_step(fw_handle h, const float* act_dev, float* obs_dev, float* rew_dev, uint8_t* flags_dev,
            float* term_obs_dev, void* stream);

/* Random-action workload (BASELINE config 2/5): actions U(-1,1)^4 drawn in-kernel from Philox keyed by
 * (seed, global env id, episode, step_count); n_steps env-steps, one kernel launch per env-step.
 * rew_dev / flags_dev may be NULL. */
int fw_step_random(fw_handle h, int32_t n_steps, float* rew_dev, uint8_t* flags_dev, void* stream);

/* Random-action sweep over a list of env batches on one device: launch j advances batch hs[j % n_handles] by
 * steps_per_launch env-steps (state stays in registers between the fused steps; no observation is emitted).
 * use_graph != 0 replays a cached CUDA graph of one round-robin pass so launches are issued back to back
 * without host involvement.  Results are identical to fw_step_random step by step.  The graph cache is process-global:
 * do not call this entry point from two host threads at once. */
int fw_rollout_random(const fw_handle* hs, int32_t n_handles, int32_t n_launches, int32_t steps_per_launch,
                      int32_t use_graph, void* stream);

/* Synchronous host-buffer variant of fw_step: the call SB3's VecEnv.step() makes (numpy in, numpy out).
 * Copies actions H2D, steps, copies obs/reward/flags (and terminal obs when requested) D2H through
 * internal pinned staging buffers on an internal stream, then waits. */
int fw_step_host(fw_handle h, const float* act_host, float* obs_host, float* rew_host, uint8_t* flags_host,
                 float* term_obs_host);
int fw_reset_host(fw_handle h, float* obs_host);
/* Observation of the CURRENT state of every env without resetting anything (last action unknown -> zeros in the action
 * slots): what a single-env gymnasium view returns from reset() right after a finished episode, when the batch has
 * already auto-reset itself (the SubprocVecEnv worker's obs = env.reset()). */
int fw_observe_host(fw_handle h, float* obs_host);

/* info["num_targets_reached"] (fixedwing_waypoint_objlock_env.py:296, upstream FixedwingWaypointsEnv) of the last step,
 * per env, taken BEFORE the auto-reset of a finished episode -- what WaypointEvalCallback._log_success_callback reads
 * on every done (train_Fixedwing_Waypoints_v3.py:136-138, train_Fixedwing_Waypoints_ObjLock.py:181-185).
 * Host lane: a pinned [N] byte buffer owned by the handle that every fw_step_host fills (tasks 1 and 2).
 * Device lane: an asynchronous device-to-device copy of the same plane as written by the last fw_step. */
int fw_host_info_buffer(fw_handle h, uint8_t** targets_reached);
int fw_targets_reached(fw_handle h, uint8_t* dst_dev, void* stream);

/* Camera tasks (2, 4): how the in-step auto-resets were served since fw_create -- out[0] from a pre-warmed spare episode
 * (prepared ahead of time by dedicated blocks of the previous step launch, DESIGN.md section 4.4), out[1] inline in the
 * step kernel (no valid spare: e.g. after fw_set_state, or FWSIM_SPARE=0).  Both give the same state.  Synchronous. */
int fw_spare_stats(fw_handle h, int64_t out[2]);

/* Running-moment accumulation fused into the step kernels' epilogue (VecNormalize's obs_rms.update of the observations a
 * step returns, train_Fixedwing_Waypoints_v3.py:254-270): acc_dev = device doubles, FW_OBS_ACC_SLOTS x 2 x obs_dim, zeroed by
 * the caller; slot s holds [column sums | column sums of squares] added by the blocks with index = s mod FW_OBS_ACC_SLOTS of
 * every fw_step enqueued while the accumulator is set (NULL clears it).  ppo_moments_finalize folds the slots into the
 * running statistics and zeroes them.  Launches already enqueued (or captured in a CUDA graph) keep the pointer they were
 * launched with. */
#define FW_OBS_ACC_SLOTS 64
int fw_set_obs_accumulator(fw_handle h, double* acc_dev);

/* Debug / evaluation frame of ONE env: FixedwingBaseEnv.render() -> pybullet getCameraImage
 * [REF envs/fixedwing_envs/fixedwing_base_env.py:350-369; eval/eval_objlock.py:120-162 keeps seg and depth too].
 * Device buffers, any may be NULL: rgba uint8 [height,width,4]; seg int32 [height,width] (-1 sky, 0 ground, 1 duck,
 * 2+k obstacle k, 64+t waypoint t); depth float [height,width] = OpenGL depth-buffer values (1.0 = far plane).  The camera
 * is the task's own (FwConfig cam_*; vertical field of view 90 degrees), the scene the analytic one the vision features
 * are computed from (ground plane, obstacle cylinders, duck sphere, a goal_reach sphere per remaining waypoint) -- not
 * pybullet's meshes.  Reads the state as of the last enqueued step on `stream`. */
int fw_render(fw_handle h, int32_t env, int32_t width, int32_t height, uint8_t* rgba_dev, int32_t* seg_dev, float* depth_dev,
              void* stream);

/* number of envs force-reset because their state went non-finite (FW_FLAG_FAULT) since fw_create (synchronous) */
int fw_fault_count(fw_handle h, int64_t* nonfinite_resets);
/* The library's pinned staging buffers ([N,4] actions, [N,obs_dim] obs, [N] rewards, [N] flag bytes,
 * [N,obs_dim] terminal obs).  Passing these very pointers to fw_step_host / fw_reset_host makes the call
 * zero-copy on the host side (DMA straight from/to the caller-visible memory).  Owned by the handle. */
int fw_host_buffers(fw_handle h, float** act, float** obs, float** rew, uint8_t** flags, float** term_obs);

/* parity injection / inspection (synchronous) */
int fw_set_state(fw_handle h, const FwStateHost* s);
int fw_get_state(fw_handle h, FwStateHost* s);

/* device-side episode accumulators: sums since the last call (synchronous, resets the counters).
 * out[0]=episodes finished, [1]=sum return, [2]=sum length, [3]=sum targets reached,
 * [4]=collisions, [5]=out-of-bounds, [6]=completed, [7]=strikes */
int fw_episode_stats(fw_handle h, double out[8]);

/* number of kernel launches issued through this handle so far (bench.py's gpu_launches) */
int64_t fw_launch_count(fw_handle h);

/* FP32 FMA-chain peak (TFLOP/s, best of 5) of `device`, with its SM count and nominal clock: the roofline
 * denominator for the FP32-bound env-step kernel (MEASURED_PEAKS.json has only HBM and bf16 tensor peaks). */
int fw_measure_fp32_peak(int32_t device, double* tflops, int32_t* sm_count, int32_t* sm_clock_khz);

#ifdef __cplusplus
}
#endif
#endif
