// fw_api.cu -- C ABI of libfwsim.so (include/fwsim.h): handle lifetime, constant folding, host<->device plumbing.
// No torch types cross this boundary; the Python host binds it with ctypes (pyflyt_drone_b200/_lib.py).
#include "../../include/fwsim.h"
#include "fw_device.cuh"
#include "fw_kernels.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess) return fail(FW_ECUDA, "%s: %s", #call, cudaGetErrorString(_e)); \
    } while (0)

#define FW_HOST_CHUNKS 2      // host lane: chunks per step, alternating between two streams (measured best of 1..16)

struct FwSim {
    FwConfig cfg;
    FwDev dev;
    FwPlanes pl;
    int n, device, obs_dim;
    char* plane_mem;
    size_t plane_bytes;
    cudaStream_t io_stream;
    cudaStream_t io_streams[2];   // host lane: io_stream and a second stream, chunks alternate between them
    // *_host staging: pinned host + device mirrors
    float *h_act, *h_obs, *h_rew, *h_term;
    uint8_t* h_flg;
    float *d_act, *d_obs, *d_rew, *d_term;
    uint8_t* d_flg;
    uint8_t* h_tidx;   // host lane: info["num_targets_reached"] per env, written by the step kernel (pinned, device-mapped)
    // pre-warmed spare episodes of the camera tasks (FwPlanes::sp_*): second plane arena, two request lists used alternately
    // (ctl[0], ctl[1] = their entry counts, ctl[2], ctl[3] = finished-block counters of the refill kernels), and the
    // low-priority side stream the refill runs on beside the next step
    char* spare_mem;
    int2* refill_list[2];
    int* refill_ctl;
    int parity;
    bool spare_on;
    cudaStream_t side;
    cudaEvent_t ev_fork, ev_join;
    int64_t launches;
    bool fresh;   // true until the state created by fw_create has been stepped or overwritten
    // Lane ordering: the device lane enqueues on the caller's stream, the host lane on private non-blocking streams, and
    // both touch the same state planes.  The host lane is synchronous (it waits for its own streams before returning), so
    // the only hazard is device-lane work still in flight when a host-lane call starts: the flag makes that call wait
    // for the device first.  Pure-host and pure-device users never pay for it.
    bool dev_lane_dirty;
    // gridded wind field (wind_mode 3): device lattice, and whether the batch still waits for it (fw_set_wind_field)
    float4* wf_mem;
    bool field_pending;
    // high-level waypoint task (task 5): the frozen tracker's device copies (one allocation: policy tower, statistics, the
    // previous-action plane) and whether the batch still waits for it (fw_set_tracker)
    char* trk_mem;
    FwTrk trk;
    bool tracker_pending;
};

// step / reset / rollout entry points on a handle whose wind field (wind_mode 3) or tracker (task 5) is not installed yet
static int need_field(const FwSim* h) {
    if (h->field_pending) return fail(FW_ESTATE, "wind_mode 3: install the wind field with fw_set_wind_field first");
    if (h->tracker_pending) return fail(FW_ESTATE, "task 5: install the low-level tracker with fw_set_tracker first");
    return FW_OK;
}

// host-lane entry: wait for device-lane launches that may still be running on the caller's streams
static int host_lane_enter(FwSim* h) {
    if (h->dev_lane_dirty) {
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) return fail(FW_ECUDA, "cudaDeviceSynchronize: %s", cudaGetErrorString(e));
        h->dev_lane_dirty = false;
    }
    return FW_OK;
}

// shared with ppo_api.cu so that fw_last_error() reports PPO kernel errors too
extern "C" void fw_set_last_error_(const char* msg) { g_err = msg ? msg : ""; }

extern "C" int fw_abi_version(void) { return FW_ABI_VERSION; }
extern "C" const char* fw_last_error(void) { return g_err.c_str(); }
extern "C" int fw_config_size(void) { return (int)sizeof(FwConfig); }

static bool invert6(const double A[36], double out[36]) {
    double m[6][12];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) { m[i][j] = A[6 * i + j]; m[i][6 + j] = i == j ? 1.0 : 0.0; }
    for (int i = 0; i < 6; ++i) {
        int p = i;
        for (int r = i + 1; r < 6; ++r) if (fabs(m[r][i]) > fabs(m[p][i])) p = r;
        if (fabs(m[p][i]) < 1e-300) return false;
        if (p != i) for (int k = 0; k < 12; ++k) std::swap(m[i][k], m[p][k]);
        double inv = 1.0 / m[i][i];
        for (int k = 0; k < 12; ++k) m[i][k] *= inv;
        for (int r = 0; r < 6; ++r) {
            if (r == i) continue;
            double f = m[r][i];
            if (f == 0.0) continue;
            for (int k = 0; k < 12; ++k) m[r][k] -= f * m[i][k];
        }
    }
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) out[6 * i + j] = m[i][6 + j];
    return true;
}

static int derive(const FwConfig& c, int n, uint64_t seed, uint32_t env_id0, FwDev& d) {
    memset(&d, 0, sizeof(d));
    const double PI = 3.14159265358979323846, DEG = PI / 180.0;
    if (!(c.dt > 0) || !(c.mass > 0)) return fail(FW_EINVAL, "dt and mass must be positive");
    if (c.wind_mode < 0 || c.wind_mode > 3) return fail(FW_EINVAL, "wind_mode %d unknown (0 off, 1 constant, 2 gust_sine, 3 gridded field)", c.wind_mode);
    if (c.task < 0 || c.task > 5)
        return fail(FW_EINVAL, "task %d unknown (0 physics, 1 waypoints, 2 waypoint+objlock, 3 low-level, 4 duck-only objlock, "
                    "5 high-level waypoints)", c.task);
    const bool cam_task = c.task == 2 || c.task == 4;
    if (cam_task && (c.num_obstacles < 0 || c.num_obstacles > FW_MAX_OBST)) return fail(FW_EINVAL, "num_obstacles out of range");
    if (cam_task && (c.cam_res < 3 || c.cam_res > 1024)) return fail(FW_EINVAL, "cam_res out of range");
    if (cam_task && c.cam_mode != 0 && c.cam_mode != 1) return fail(FW_EINVAL, "cam_mode must be 0 (tracking) or 1 (fixed)");
    if (cam_task && c.cam_mode == 0 && c.cam_offset[0] == 0 && c.cam_offset[1] == 0 && c.cam_offset[2] == 0)
        return fail(FW_EINVAL, "a tracking camera needs a non-zero cam_offset");
    if (c.task == 4 && (c.vision_hist_len < 1 || c.vision_hist_len > FW_MAX_HIST)) return fail(FW_EINVAL, "vision_hist_len out of range (1..%d)", FW_MAX_HIST);
    if (c.task == 4 && c.lock_decay_steps < 1) return fail(FW_EINVAL, "lock_decay_steps must be >= 1");
    if (c.task == 4 && c.context_len != 0) return fail(FW_EINVAL, "the duck-only task has no waypoint context (context_len must be 0)");
    if (c.num_targets < 0 || c.num_targets > FW_MAX_TARGETS) return fail(FW_EINVAL, "num_targets out of range");
    if (c.task != 0 && c.task != 4 && c.num_targets < 1) return fail(FW_EINVAL, "waypoint task needs num_targets >= 1");
    if (c.task == 4 && c.num_targets != 0) return fail(FW_EINVAL, "the duck-only task has no waypoints (num_targets must be 0)");
    if (c.context_len < 0 || c.context_len > 4) return fail(FW_EINVAL, "context_len out of range");
    if (c.n_col < 0 || c.n_col > FW_MAX_COL) return fail(FW_EINVAL, "n_col out of range");
    if (c.physics_per_control < 1 || c.substeps_per_inner < 1 || c.inner_per_step < 1 || c.warmup_inner < 0)
        return fail(FW_EINVAL, "bad step ratios");
    if (c.substeps_per_inner % c.physics_per_control != 0)
        return fail(FW_EINVAL, "substeps_per_inner must be a multiple of physics_per_control (control latch alignment)");
    for (int s = 0; s < FW_NSURF; ++s) {
        SurfDev& o = d.surf[s];
        if (!(c.chord[s] > 0) || !(c.span[s] > 0) || !(c.surf_tau[s] > 0)) return fail(FW_EINVAL, "surface %d: bad geometry", s);
        double ar = c.span[s] / c.chord[s];
        double cla = c.cl_alpha_2d[s] * (ar / (ar + ((2.0 * (ar + 4.0)) / (ar + 2.0))));
        double theta_f = acos(2.0 * c.flap_to_chord[s] - 1.0);
        double aero_tau = 1.0 - ((theta_f - sin(theta_f)) / PI);
        o.k_act = (float)(c.dt / c.surf_tau[s]);
        o.defl_rad = (float)(c.defl_limit_deg[s] * DEG);
        o.defl_deg = (float)c.defl_limit_deg[s];
        o.cla = (float)cla;
        o.tau_eta = (float)(aero_tau * c.eta[s]);
        o.omf = (float)(1.0 - c.flap_to_chord[s]);
        o.a0_base = (float)(c.alpha0_base_deg[s] * DEG);
        o.asp_base = (float)(c.stall_p_base_deg[s] * DEG);
        o.asn_base = (float)(c.stall_n_base_deg[s] * DEG);
        o.inv_pi_ar = (float)(1.0 / (PI * ar));
        o.cd0 = (float)c.cd0[s];
        o.stall_k = (float)(0.41 * (1.0 - exp(-17.0 / ar)));
        o.qarea = (float)(0.5 * c.rho * c.chord[s] * c.span[s]);
        o.chord = (float)c.chord[s];
        o.k_te = (float)(aero_tau * c.eta[s] * c.defl_limit_deg[s] * DEG);
        o.k_shift = (float)((1.0 - c.flap_to_chord[s]) * aero_tau * c.eta[s] * c.defl_limit_deg[s] * DEG);
        o.cm0c = (float)(0.075 * c.chord[s]);
        o.cm1c = (float)(0.175 * 2.0 / PI * c.chord[s]);
        o.cla_ipa = (float)(cla / (PI * ar));
        const double* l = c.lift_unit[s];
        const double* f = c.fwd_unit[s];
        double t[3] = {l[1] * f[2] - l[2] * f[1], l[2] * f[0] - l[0] * f[2], l[0] * f[1] - l[1] * f[0]};
        const double* r = c.r_surf[s];
        double ra[3] = {r[1] * l[2] - r[2] * l[1], r[2] * l[0] - r[0] * l[2], r[0] * l[1] - r[1] * l[0]};
        double rb[3] = {r[1] * f[2] - r[2] * f[1], r[2] * f[0] - r[0] * f[2], r[0] * f[1] - r[1] * f[0]};
        for (int k = 0; k < 3; ++k) {
            o.lift[k] = (float)l[k]; o.fwd[k] = (float)f[k]; o.tq[k] = (float)t[k]; o.r[k] = (float)r[k];
            o.ra[k] = (float)ra[k]; o.rb[k] = (float)rb[k];
        }
        // the same numbers packed for the standard-layout kernels (SurfHot, fw_device.cuh)
        float4* g = d.hot[s];
        g[0] = make_float4(o.k_act, o.r[0], o.r[1], o.r[2]);
        g[1] = make_float4(o.a0_base, o.k_te, o.asp_base, o.asn_base);
        g[2] = make_float4(o.k_shift, o.cla, o.cla_ipa, o.cd0);
        g[3] = make_float4(c.cd90_degrees ? o.defl_deg : o.defl_rad, o.stall_k, o.cm1c, o.cm0c);
        g[4] = make_float4(o.qarea, o.ra[0], o.ra[1], o.ra[2]);
        g[5] = make_float4(o.rb[0], o.rb[1], o.rb[2], 0.0f);
    }
    if (!(c.motor_tau > 0) || !(c.thrust_coef > 0)) return fail(FW_EINVAL, "bad motor constants");
    d.motor_k = (float)(c.dt / c.motor_tau);
    d.noise_ratio = (float)c.noise_ratio;
    double max_rpm = sqrt(c.total_thrust / c.thrust_coef);
    d.thrust_max = (float)(max_rpm * max_rpm * c.thrust_coef);
    d.torque_max = (float)(max_rpm * max_rpm * c.torque_coef);
    for (int k = 0; k < 3; ++k) { d.r_motor[k] = (float)c.r_motor[k]; d.thrust_unit[k] = (float)c.thrust_unit[k]; d.com[k] = (float)c.com[k]; }
    d.mass = (float)c.mass;
    for (int k = 0; k < 9; ++k) d.inertia[k] = (float)c.inertia_o[k];
    {
        double A[36] = {0}, Ai[36];
        const double M = c.mass, cx = c.com[0], cy = c.com[1], cz = c.com[2];
        const double Cx[3][3] = {{0, -cz, cy}, {cz, 0, -cx}, {-cy, cx, 0}};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                A[6 * i + j] = c.inertia_o[3 * i + j];
                A[6 * i + 3 + j] = M * Cx[i][j];
                A[6 * (3 + i) + j] = -M * Cx[i][j];
            }
        for (int i = 0; i < 3; ++i) A[6 * (3 + i) + 3 + i] = M;
        if (!invert6(A, Ai)) return fail(FW_EINVAL, "singular spatial inertia");
        for (int k = 0; k < 36; ++k) d.minv[k] = (float)Ai[k];
        // Standard layout (fw_substep<STD>): +x forward units, lift +z (+y for the vertical tail, surface 3), thrust
        // along +x, and an inverse spatial inertia that splits into the lateral {wx, wz, vy} / longitudinal
        // {wy, vx, vz} blocks of an aircraft symmetric about its xz plane.  Anything else runs the generic kernels.
        bool std_ok = true;
        for (int s = 0; s < FWD_NSURF; ++s) {
            const double* l = c.lift_unit[s];
            const double* f = c.fwd_unit[s];
            const bool lift_ok = s == 3 ? (l[0] == 0 && l[1] == 1 && l[2] == 0) : (l[0] == 0 && l[1] == 0 && l[2] == 1);
            std_ok = std_ok && lift_ok && f[0] == 1 && f[1] == 0 && f[2] == 0;
        }
        std_ok = std_ok && c.thrust_unit[0] == 1 && c.thrust_unit[1] == 0 && c.thrust_unit[2] == 0;
        double amax = 0;
        for (int k = 0; k < 36; ++k) amax = fmax(amax, fabs(Ai[k]));
        for (int i = 0; i < 6; ++i)
            for (int j = 0; j < 6; ++j) {
                const bool lat_i = (i == 0 || i == 2 || i == 4), lat_j = (j == 0 || j == 2 || j == 4);
                if (lat_i != lat_j && fabs(Ai[6 * i + j]) > 1e-12 * amax) std_ok = false;
            }
        d.std_geom = (std_ok && c.force_generic_kernel == 0) ? 1 : 0;
        // packed rigid-body / motor constants of the standard-layout substep (FwDev::rbk)
        const int lat[9] = {0, 2, 4, 12, 14, 16, 24, 26, 28}, lon[9] = {7, 9, 11, 19, 21, 23, 31, 33, 35};
        float k[FWD_RBK * 4] = {0};
        k[0] = d.motor_k; k[1] = d.noise_ratio; k[2] = d.thrust_max; k[3] = d.torque_max;
        k[4] = d.r_motor[1]; k[5] = d.r_motor[2]; k[6] = (float)c.gravity; k[7] = d.mass;
        k[8] = d.com[0]; k[9] = d.com[1]; k[10] = d.com[2]; k[11] = (float)c.max_coord_vel;
        for (int q = 0; q < 9; ++q) k[12 + q] = d.inertia[q];
        for (int q = 0; q < 9; ++q) { k[21 + q] = d.minv[lat[q]]; k[30 + q] = d.minv[lon[q]]; }
        for (int q = 0; q < FWD_RBK; ++q) d.rbk[q] = make_float4(k[4 * q], k[4 * q + 1], k[4 * q + 2], k[4 * q + 3]);
    }
    double rad = 0.0;
    for (int i = 0; i < c.n_col; ++i) {
        double r2 = 0;
        for (int k = 0; k < 3; ++k) { d.col[i][k] = (float)c.col_pts[i][k]; r2 += c.col_pts[i][k] * c.col_pts[i][k]; }
        rad = fmax(rad, sqrt(r2));
    }
    d.col_radius = (float)(rad * 1.0001 + 1e-6);
    d.contact_margin = (float)c.contact_margin;
    d.n_col = c.n_col;
    d.dt = (float)c.dt; d.gravity = (float)c.gravity; d.max_vel = (float)c.max_coord_vel;
    d.sign_ail_l = (float)c.ail_left_sign; d.sign_ail_r = (float)c.ail_right_sign;
    d.sign_pitch = (float)c.pitch_sign; d.sign_yaw = (float)c.yaw_sign;
    d.substeps_per_inner = c.substeps_per_inner; d.inner_per_step = c.inner_per_step;
    d.warmup_substeps = c.warmup_inner * c.substeps_per_inner;
    d.freestream_3d = c.freestream_3d; d.cd90_degrees = c.cd90_degrees;
    d.quat_limiter = (sqrt(3.0) * c.max_coord_vel * c.dt > 0.25 * PI) ? 1 : 0;
    d.task = c.task; d.num_targets = c.num_targets; d.sparse_reward = c.sparse_reward; d.angle_repr = c.angle_repr;
    d.max_steps = c.max_steps; d.context_len = c.context_len;
    d.obs_dim = c.task == 0 ? 0 : (c.task == 3 ? 21 : ((c.angle_repr == 0 ? 12 : 13) + 4 + 6 + 3 * c.context_len));
    if (c.task == 4) d.obs_dim += 3 + 9 * c.vision_hist_len + (c.vision_use_deltas ? 4 : 0);   // flatten_objlock_env.py:20-31
    d.act_dim = c.task == 3 ? 6 : 4;
    d.early_return_on_crash = c.early_return_on_crash; d.complete_truncates = c.complete_truncates;
    d.goal_reach = (float)c.goal_reach; d.dome = (float)c.dome; d.dome2 = (float)(c.dome * c.dome); d.spawn_size = (float)c.spawn_size; d.min_height = (float)c.min_height;
    for (int k = 0; k < 3; ++k) {
        d.start_pos[k] = (float)c.start_pos[k]; d.start_vel[k] = (float)c.start_vel[k];
        d.wind_base[k] = (float)c.wind_base[k]; d.wind_base_lo[k] = (float)c.wind_base_lo[k]; d.wind_base_hi[k] = (float)c.wind_base_hi[k];
        d.gust_amp[k] = (float)c.gust_amp[k]; d.gust_amp_lo[k] = (float)c.gust_amp_lo[k]; d.gust_amp_hi[k] = (float)c.gust_amp_hi[k];
    }
    d.wind_mode = c.wind_mode; d.wind_randomize = c.wind_randomize; d.wind_rand_phase = c.wind_rand_phase;
    d.wind_start_substep = c.wind_start_substep;
    d.gust_omega = (float)(2.0 * PI * c.gust_freq); d.gust_phase = (float)c.gust_phase;
    d.gust_cyc = (float)(c.gust_freq * c.dt);
    d.num_obstacles = c.num_obstacles; d.cam_interval = c.cam_interval_substeps; d.lock_hold = c.lock_hold_steps;
    d.switch_min_seen = c.switch_min_seen; d.cam_res = c.cam_res;
    d.obst_radius = (float)c.obst_radius; d.obst_h_lo = (float)c.obst_h_lo; d.obst_h_hi = (float)c.obst_h_hi;
    d.obst_safe = (float)c.obst_safe; d.obst_scale = (float)c.obst_scale; d.obst_max_pen = (float)c.obst_max_pen;
    d.strike_dist = (float)c.strike_dist; d.strike_reward = (float)c.strike_reward; d.lock_step_reward = (float)c.lock_step_reward;
    d.approach_scale = (float)c.approach_scale; d.switch_min_area = (float)c.switch_min_area;
    d.duck_radius = (float)c.duck_radius; d.cam_near = (float)c.cam_near; d.cam_far = (float)c.cam_far;
    for (int k = 0; k < 3; ++k) d.cam_offset[k] = (float)c.cam_offset[k];
    d.cam_mode = c.cam_mode;
    {   // fixed camera: forward and up hint = body x and z rotated about body +y by the tilt (positive = nose-down)
        const double t = c.cam_tilt_deg * DEG;
        d.cam_fb[0] = (float)cos(t); d.cam_fb[1] = 0.0f; d.cam_fb[2] = (float)(-sin(t));
        d.cam_ub[0] = (float)sin(t); d.cam_ub[1] = 0.0f; d.cam_ub[2] = (float)cos(t);
    }
    d.hist_len = c.task == 4 ? c.vision_hist_len : 0; d.use_deltas = c.vision_use_deltas; d.lock_decay = c.lock_decay_steps;
    d.hist_slots = c.task == 4 ? 9 * c.vision_hist_len + 4 : 0;
    d.duck_dist_scale = (float)c.duck_dist_scale; d.lock_center_radius = (float)c.lock_center_radius;
    d.centering_scale = (float)c.centering_scale; d.visible_step_reward = (float)c.visible_step_reward;
    d.area_reward_scale = (float)c.area_reward_scale; d.lock_lost_penalty = (float)c.lock_lost_penalty;
    d.approach_clip = (float)c.approach_clip;
    d.warm_cached = 0;
    d.packed = (c.packed_pairs != 0 && c.wind_mode != 3) ? 1 : 0;    // the packed path has no gridded field
    d.seed_lo = (uint32_t)(seed & 0xffffffffu); d.seed_hi = (uint32_t)(seed >> 32); d.env_id0 = env_id0;
    d.n = n;
    d.i_begin = 0; d.i_end = n;
    return FW_OK;
}

// cached CUDA graph of one round-robin pass over a handle list
struct MultiGraph {
    std::vector<FwSim*> hs;
    int spl = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
};
// Process-global (not per handle): fw_rollout_random takes a LIST of handles, so the cache belongs to the call site, keyed by
// the list.  Consequence for the "handles are independent" contract: fw_rollout_random itself is not re-entrant -- two host
// threads must not call it concurrently, even on disjoint handle lists (every other entry point only touches its handle);
// fw_destroy drops a cached graph that names the handle.
static MultiGraph g_multi;     // one full round-robin pass over the handle list
static MultiGraph g_rem;       // the launches left over after the full passes (a prefix of the list)

// (re)build `mg` as a chain of `count` random-step launches over hs[0], hs[1], ... (wrapping), unless it already is
static int multi_graph_get(MultiGraph& mg, const fw_handle* hs, int n_handles, int count, int spl) {
    bool hit = mg.exec && mg.spl == spl && (int)mg.hs.size() == count;
    for (int k = 0; hit && k < count; ++k) hit = mg.hs[k] == hs[k % n_handles];
    if (hit) return FW_OK;
    if (mg.exec) { cudaGraphExecDestroy(mg.exec); mg.exec = nullptr; }
    if (mg.graph) { cudaGraphDestroy(mg.graph); mg.graph = nullptr; }
    mg.hs.clear();
    CU(cudaGraphCreate(&mg.graph, 0));
    // Step launches form one chain.  With spare episodes, handle h's refill (serving the list its step of the PREVIOUS pass
    // filled -- list 0 for every graph launch) is a branch that forks off three launches ahead of h's step and joins at it:
    // it runs beside other handles' steps and nothing dangles at the end of the graph.  (count <= n_handles: every handle
    // appears at most once per graph; successive graph launches of one stream do not overlap.)
    std::vector<cudaGraphNode_t> steps((size_t)count);
    for (int k = 0; k < count; ++k) {
        FwSim* h = hs[k % n_handles];
        cudaGraphNode_t deps[2];
        int nd = 0;
        if (k > 0) deps[nd++] = steps[(size_t)k - 1];
        FwPlanes plc = h->pl;
        if (h->spare_on) {
            cudaGraphNode_t rf;
            const int fork = k - 3;
            CU(fwk_graph_add_refill(mg.graph, fork >= 0 ? &steps[(size_t)fork] : nullptr, fork >= 0 ? 1 : 0, h->dev, h->pl,
                                    h->refill_list[0], h->refill_ctl, h->refill_ctl + 2, h->n, &rf));
            deps[nd++] = rf;
            plc.refill_list = h->refill_list[0]; plc.refill_count = h->refill_ctl;
        }
        // programmatic dependent launch along the chain: the next step launch places its blocks while this one drains.  A
        // launch touches the state of its own handle only, and the one before it in the chain belongs to another handle
        // whenever the list has several (mode 2: no wait); a handle stepping itself waits for its predecessor (mode 1).
        // FWSIM_PDL=0 turns it off.
        static const bool pdl_on = [] { const char* e = getenv("FWSIM_PDL"); return !(e && atoi(e) == 0); }();
        // Every (n_handles / 2)-th edge stays an ordinary one: two launches on the same handle are n_handles apart, so they can
        // never be in flight together whatever the block scheduler does.
        const int period = n_handles / 2;
        const int pdl = (pdl_on && !h->spare_on && !(n_handles >= 4 && k % period == 0)) ? (n_handles >= 4 ? 2 : 1) : 0;
        CU(fwk_graph_add_random_step(mg.graph, nd ? deps : nullptr, nd, h->dev, plc, spl, &steps[(size_t)k], pdl));
    }
    CU(cudaGraphInstantiate(&mg.exec, mg.graph, 0));
    for (int k = 0; k < count; ++k) mg.hs.push_back(hs[k % n_handles]);
    mg.spl = spl;
    return FW_OK;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Lay the per-env planes out in one arena (256-byte aligned sub-ranges); base == nullptr only measures.
static size_t carve_planes(const FwConfig& cfg, const FwDev& dev, size_t N, char* base, FwPlanes& pl) {
    const size_t T = (size_t)(cfg.num_targets > 0 ? cfg.num_targets : 1);
    const bool cam_task = cfg.task == 2 || cfg.task == 4;
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off = align_up(off + bytes, 256); return p; };
    memset(&pl, 0, sizeof(pl));
    pl.s0 = (float4*)take(N * 16); pl.s1 = (float4*)take(N * 16); pl.s2 = (float4*)take(N * 16);
    pl.s3 = (float4*)take(N * 16); pl.s4 = (float4*)take(N * 16); pl.s5 = (int4*)take(N * 16);
    pl.w0 = (float4*)take(N * 16); pl.w1 = (float4*)take(N * 16);
    pl.targets = (float*)take(T * 3 * N * 4);
    pl.ep_ret = (float*)take(N * 4);
    pl.stats = (double*)take(16 * sizeof(double));
    pl.tidx_out = (uint8_t*)take(N);
    if (cam_task) {
        pl.dk = (float4*)take(N * 16); pl.v0 = (float4*)take(N * 16); pl.v1 = (float4*)take(N * 16);
        pl.v2 = (float4*)take(N * 16); pl.v3 = (int4*)take(N * 16);
        pl.obst = (float*)take((size_t)FW_MAX_OBST * 3 * N * 4);
    }
    if (cfg.task == 4) pl.hist = (float*)take((size_t)dev.hist_slots * N * 4);
    return off;
}

static int fw_create_impl(const FwConfig* cfg, int32_t n_envs, int32_t device, uint64_t seed, uint32_t env_id0, FwSim* h);
static int initial_episodes(FwSim* h);

extern "C" int fw_create(const FwConfig* cfg, int32_t n_envs, int32_t device, uint64_t seed, uint32_t env_id0, fw_handle* out) {
    if (!cfg || !out) return fail(FW_EINVAL, "null argument");
    if (n_envs <= 0) return fail(FW_EINVAL, "n_envs must be positive");
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0)
        return fail(FW_ECUDA, "no CUDA device available (%s): libfwsim has no CPU fallback", cudaGetErrorString(ce));
    if (device < 0 || device >= ndev) return fail(FW_EINVAL, "device %d out of range (%d visible)", device, ndev);
    CU(cudaSetDevice(device));
    FwSim* h = new FwSim();
    memset(h, 0, sizeof(*h));
    const int rc = fw_create_impl(cfg, n_envs, device, seed, env_id0, h);
    if (rc != FW_OK) {                       // every early return of the body lands here: nothing leaks
        const std::string keep = g_err;
        fw_destroy(h);
        g_err = keep;
        return rc;
    }
    *out = h;
    return FW_OK;
}

static int fw_create_impl(const FwConfig* cfg, int32_t n_envs, int32_t device, uint64_t seed, uint32_t env_id0, FwSim* h) {
    cudaError_t ce;
    h->cfg = *cfg; h->n = n_envs; h->device = device;
    int rc = derive(*cfg, n_envs, seed, env_id0, h->dev);
    if (rc != FW_OK) return rc;
    h->obs_dim = h->dev.obs_dim;
    const size_t N = (size_t)n_envs;
    h->plane_bytes = carve_planes(*cfg, h->dev, N, nullptr, h->pl);
    ce = cudaMalloc((void**)&h->plane_mem, h->plane_bytes);
    if (ce != cudaSuccess) return fail(FW_ENOMEM, "cudaMalloc(%zu): %s", h->plane_bytes, cudaGetErrorString(ce));
    cudaMemset(h->plane_mem, 0, h->plane_bytes);
    carve_planes(*cfg, h->dev, N, h->plane_mem, h->pl);
    FwPlanes& pl = h->pl;
    // episode counter starts at -1 so that the first reset opens episode 0
    cudaMemset(pl.s5, 0xff, N * 16);
    CU(cudaStreamCreateWithFlags(&h->io_stream, cudaStreamNonBlocking));
    h->io_streams[0] = h->io_stream;
    CU(cudaStreamCreateWithFlags(&h->io_streams[1], cudaStreamNonBlocking));
    // the first reset needs the field and the tracker: the last of fw_set_wind_field / fw_set_tracker runs the set-up
    h->field_pending = h->dev.wind_mode == 3;
    h->tracker_pending = h->dev.task == 5;
    if (h->field_pending || h->tracker_pending) return FW_OK;
    return initial_episodes(h);
}

// The warm-up cache decision, the first reset of every env and the spare episodes of the camera tasks: the tail of fw_create,
// or of whichever of fw_set_wind_field (wind_mode 3) and fw_set_tracker (task 5) completes the handle.
static int initial_episodes(FwSim* h) {
    cudaError_t ce;
    const FwConfig* cfg = &h->cfg;
    const int32_t n_envs = h->n;
    const size_t N = (size_t)n_envs;
    const bool cam_task = cfg->task == 2 || cfg->task == 4;
    // cache the deterministic warm-up result when no wind acts during it
    if (!cam_task && (h->dev.wind_mode == 0 || h->dev.wind_start_substep >= h->dev.warmup_substeps)) {
        float* d_warm = nullptr;
        CU(cudaMalloc((void**)&d_warm, 20 * sizeof(float)));
        CU(fwk_launch_warm(h->dev, h->pl, d_warm, h->io_stream));
        h->launches++;
        CU(cudaMemcpyAsync(h->dev.warm, d_warm, 20 * sizeof(float), cudaMemcpyDeviceToHost, h->io_stream));
        CU(cudaStreamSynchronize(h->io_stream));
        cudaFree(d_warm);
        h->dev.warm_cached = 1;
    }
    CU(fwk_launch_reset(h->dev, h->pl, nullptr, nullptr, false, h->io_stream));
    h->launches++;
    CU(cudaStreamSynchronize(h->io_stream));
    h->fresh = true;
    // Spare episodes for the camera tasks, whose reset cannot be cached (per-episode wind during the warm-up, a camera frame
    // inside it).  FWSIM_SPARE=0 turns the feature off (inline resets only; the results are the same).
    const char* sp_env = getenv("FWSIM_SPARE");
    if (cam_task && !(sp_env && atoi(sp_env) == 0)) {
        FwPlanes sv;
        const size_t bytes = carve_planes(*cfg, h->dev, N, nullptr, sv);
        ce = cudaMalloc((void**)&h->spare_mem, bytes);
        if (ce != cudaSuccess) return fail(FW_ENOMEM, "cudaMalloc(%zu) for the spare episodes: %s", bytes, cudaGetErrorString(ce));
        CU(cudaMemset(h->spare_mem, 0, bytes));
        carve_planes(*cfg, h->dev, N, h->spare_mem, sv);
        for (int k = 0; k < 2; ++k) CU(cudaMalloc((void**)&h->refill_list[k], N * sizeof(int2)));
        CU(cudaMalloc((void**)&h->refill_ctl, 4 * sizeof(int)));
        CU(cudaMemset(h->refill_ctl, 0, 4 * sizeof(int)));
        {
            int lo = 0, hi = 0;
            CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CU(cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, lo));   // lowest: the step's blocks are placed first
        }
        CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
        FwPlanes& l = h->pl;
        l.sp_s0 = sv.s0; l.sp_s1 = sv.s1; l.sp_s2 = sv.s2; l.sp_s3 = sv.s3; l.sp_s4 = sv.s4; l.sp_s5 = sv.s5;
        l.sp_w0 = sv.w0; l.sp_w1 = sv.w1; l.sp_targets = sv.targets;
        l.sp_dk = sv.dk; l.sp_v0 = sv.v0; l.sp_v1 = sv.v1; l.sp_v2 = sv.v2; l.sp_v3 = sv.v3; l.sp_obst = sv.obst; l.sp_hist = sv.hist;
        l.refill_cap = n_envs;
        CU(cudaMemset(sv.s5, 0xff, N * 16));                              // tag -1: no spare yet
        CU(fwk_launch_refill(h->dev, h->pl, nullptr, nullptr, nullptr, n_envs, n_envs, h->io_stream));   // episode 1 of every env
        h->launches++;
        CU(cudaStreamSynchronize(h->io_stream));
        h->spare_on = true;
    }
    return FW_OK;
}

// One step launch with the spare-episode traffic around it: the refill of the PREVIOUS launch's request list runs on the
// low-priority side stream beside this step's kernel (fork / join through events, so a stream capture of the caller's
// stream records a two-branch graph); this step appends to the other list, which the refill that served it last has
// left empty.
static int launch_step(FwSim* h, const FwDev& dev, FwPlanes pl, const float* act, float* obs, float* rew, uint8_t* flg,
                       float* term_obs, bool random_act, int spl, cudaStream_t st) {
    if (!h->spare_on) {
        CU(fwk_launch_step(dev, pl, act, obs, rew, flg, term_obs, random_act, spl, st, &h->trk));
        h->launches++;
        return FW_OK;
    }
    const int par = h->parity, prev = par ^ 1;
    CU(cudaEventRecord(h->ev_fork, st));
    CU(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
    pl.refill_list = h->refill_list[par];
    pl.refill_count = h->refill_ctl + par;
    CU(fwk_launch_step(dev, pl, act, obs, rew, flg, term_obs, random_act, spl, st));     // first: its blocks are placed first
    CU(fwk_launch_refill(dev, h->pl, h->refill_list[prev], h->refill_ctl + prev, h->refill_ctl + 2 + prev, h->n, 0, h->side));
    CU(cudaEventRecord(h->ev_join, h->side));
    CU(cudaStreamWaitEvent(st, h->ev_join, 0));
    h->launches += 2;
    h->parity ^= 1;
    return FW_OK;
}

extern "C" int fw_destroy(fw_handle h) {
    if (!h) return FW_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (MultiGraph* mg : {&g_multi, &g_rem})          // a cached launch graph that names this handle dies with it
        for (FwSim* g : mg->hs)
            if (g == h) {
                if (mg->exec) cudaGraphExecDestroy(mg->exec);
                if (mg->graph) cudaGraphDestroy(mg->graph);
                *mg = MultiGraph();
                break;
            }
    if (h->plane_mem) cudaFree(h->plane_mem);
    if (h->wf_mem) cudaFree(h->wf_mem);
    if (h->trk_mem) cudaFree(h->trk_mem);
    if (h->d_act) cudaFree(h->d_act);
    if (h->d_obs) cudaFree(h->d_obs);
    if (h->d_rew) cudaFree(h->d_rew);
    if (h->d_term) cudaFree(h->d_term);
    if (h->d_flg) cudaFree(h->d_flg);
    if (h->h_act) cudaFreeHost(h->h_act);
    if (h->h_obs) cudaFreeHost(h->h_obs);
    if (h->h_rew) cudaFreeHost(h->h_rew);
    if (h->h_term) cudaFreeHost(h->h_term);
    if (h->h_flg) cudaFreeHost(h->h_flg);
    if (h->h_tidx) cudaFreeHost(h->h_tidx);
    if (h->spare_mem) cudaFree(h->spare_mem);
    if (h->refill_list[0]) cudaFree(h->refill_list[0]);
    if (h->refill_list[1]) cudaFree(h->refill_list[1]);
    if (h->refill_ctl) cudaFree(h->refill_ctl);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->io_stream) cudaStreamDestroy(h->io_stream);
    if (h->io_streams[1]) cudaStreamDestroy(h->io_streams[1]);
    delete h;
    return FW_OK;
}

extern "C" int fw_set_wind_field(fw_handle h, const FwWindField* f) {
    // argument checks first, without touching the device
    if (!f) return fail(FW_EINVAL, "null wind field");
    if (!f->values) return fail(FW_EINVAL, "wind field: values is null");
    if (f->nx < 1 || f->ny < 1 || f->nz < 1 || f->nt < 1) return fail(FW_EINVAL, "wind field: every dimension must be >= 1");
    const int64_t pts = (int64_t)f->nx * f->ny * f->nz;
    if (pts * f->nt >= ((int64_t)1 << 31)) return fail(FW_EINVAL, "wind field: nx * ny * nz * nt must be < 2^31");
    for (int k = 0; k < 3; ++k) {
        if (!(f->spacing[k] > 0) || !std::isfinite(f->spacing[k])) return fail(FW_EINVAL, "wind field: spacing must be finite and > 0");
        if (!std::isfinite(f->origin[k])) return fail(FW_EINVAL, "wind field: origin must be finite");
        if (!std::isfinite(f->shift_lo[k]) || !std::isfinite(f->shift_hi[k]) || f->shift_lo[k] > f->shift_hi[k])
            return fail(FW_EINVAL, "wind field: shift range must be finite with shift_lo <= shift_hi");
    }
    if (!(f->t_step > 0) || !std::isfinite(f->t_step)) return fail(FW_EINVAL, "wind field: t_step must be finite and > 0");
    const size_t nval = (size_t)(pts * f->nt) * 3;
    for (size_t k = 0; k < nval; ++k)
        if (!std::isfinite(f->values[k])) return fail(FW_EINVAL, "wind field: value %zu is not finite", k);
    if (!h) return fail(FW_EINVAL, "null handle");
    if (h->dev.wind_mode != 3) return fail(FW_EINVAL, "fw_set_wind_field needs a handle created with wind_mode 3 (has %d)", h->dev.wind_mode);
    if (!h->field_pending) return fail(FW_ESTATE, "the wind field of this handle is already set (one field per handle)");
    CU(cudaSetDevice(h->device));
    // float4 lattice points: one 16-byte load per corner
    const size_t npts = (size_t)(pts * f->nt);
    std::vector<float4> host(npts);
    for (size_t k = 0; k < npts; ++k) host[k] = make_float4(f->values[3 * k], f->values[3 * k + 1], f->values[3 * k + 2], 0.0f);
    cudaError_t ce = cudaMalloc((void**)&h->wf_mem, npts * sizeof(float4));
    if (ce != cudaSuccess) { h->wf_mem = nullptr; return fail(FW_ENOMEM, "cudaMalloc(%zu) for the wind field: %s", npts * sizeof(float4), cudaGetErrorString(ce)); }
    ce = cudaMemcpyAsync(h->wf_mem, host.data(), npts * sizeof(float4), cudaMemcpyHostToDevice, h->io_stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->io_stream);
    if (ce != cudaSuccess) {                  // the handle stays pending: a later call may try again
        cudaFree(h->wf_mem);
        h->wf_mem = nullptr;
        return fail(FW_ECUDA, "uploading the wind field: %s", cudaGetErrorString(ce));
    }
    FwDev& d = h->dev;
    d.wf = h->wf_mem;
    d.wf_n[0] = f->nx; d.wf_n[1] = f->ny; d.wf_n[2] = f->nz; d.wf_n[3] = f->nt;
    d.wf_pts = (int)pts;
    for (int k = 0; k < 3; ++k) {
        d.wf_origin[k] = (float)f->origin[k];
        d.wf_inv_sp[k] = (float)(1.0 / f->spacing[k]);
        d.wf_max[k] = (float)((k == 0 ? f->nx : (k == 1 ? f->ny : f->nz)) - 1);
        d.wf_shift_lo[k] = (float)f->shift_lo[k]; d.wf_shift_hi[k] = (float)f->shift_hi[k];
    }
    d.wf_sps = (float)(h->cfg.dt / f->t_step);
    d.wf_inv_tstep = (float)(1.0 / f->t_step);
    d.wf_nt = (float)f->nt;
    d.wf_inv_nt = (float)(1.0 / f->nt);
    d.wf_period = (float)(f->nt * f->t_step);
    d.wf_rand_time = f->randomize_time != 0;
    h->field_pending = false;
    return h->tracker_pending ? FW_OK : initial_episodes(h);
}

// floats of the policy tower at the head of the flat (21, 6) parameter vector (include/fwppo.h)
static const size_t TRK_TOWER = (size_t)64 * FW_TRK_OBS + 64 + 64 * 64 + 64 + FW_TRK_ACT * 64 + FW_TRK_ACT;

static bool finite_range(const double r[2]) { return std::isfinite(r[0]) && std::isfinite(r[1]) && r[0] < r[1]; }

extern "C" int fw_set_tracker(fw_handle h, const FwTracker* t) {
    // argument checks first, without touching the device
    if (!t) return fail(FW_EINVAL, "null tracker");
    if (!t->params) return fail(FW_EINVAL, "tracker: params is null");
    if ((t->obs_mean == nullptr) != (t->obs_var == nullptr))
        return fail(FW_EINVAL, "tracker: obs_mean and obs_var are both set (normalised tracker) or both null");
    for (size_t k = 0; k < TRK_TOWER; ++k)
        if (!std::isfinite(t->params[k])) return fail(FW_EINVAL, "tracker: policy parameter %zu is not finite", k);
    if (t->obs_mean)
        for (int k = 0; k < FW_TRK_OBS; ++k) {
            if (!std::isfinite(t->obs_mean[k])) return fail(FW_EINVAL, "tracker: obs_mean[%d] is not finite", k);
            if (!std::isfinite(t->obs_var[k]) || t->obs_var[k] < 0) return fail(FW_EINVAL, "tracker: obs_var[%d] must be finite and >= 0", k);
        }
    if (!(t->clip_obs > 0) || !std::isfinite(t->clip_obs)) return fail(FW_EINVAL, "tracker: clip_obs must be finite and > 0");
    if (!finite_range(t->h_range)) return fail(FW_EINVAL, "tracker: h_range must be finite with lo < hi");
    if (!finite_range(t->v_range)) return fail(FW_EINVAL, "tracker: v_range must be finite with lo < hi");
    if (!h) return fail(FW_EINVAL, "null handle");
    if (h->dev.task != 5) return fail(FW_EINVAL, "fw_set_tracker needs a handle created with task 5 (has %d)", h->dev.task);
    if (!h->tracker_pending) return fail(FW_ESTATE, "the tracker of this handle is already set (one tracker per handle)");
    CU(cudaSetDevice(h->device));
    // one allocation: tower | statistics (mean 21 | var 21, doubles) | previous-action plane [6][N], zeroed
    const size_t N = (size_t)h->n;
    const size_t off_stats = align_up(TRK_TOWER * sizeof(float), 256), off_prev = off_stats + align_up(2 * FW_TRK_OBS * sizeof(double), 256);
    const size_t bytes = off_prev + (size_t)FW_TRK_ACT * N * sizeof(float);
    std::vector<double> stats(2 * FW_TRK_OBS);
    if (t->obs_mean)
        for (int k = 0; k < FW_TRK_OBS; ++k) { stats[k] = t->obs_mean[k]; stats[FW_TRK_OBS + k] = t->obs_var[k]; }
    cudaError_t ce = cudaMalloc((void**)&h->trk_mem, bytes);
    if (ce != cudaSuccess) { h->trk_mem = nullptr; return fail(FW_ENOMEM, "cudaMalloc(%zu) for the tracker: %s", bytes, cudaGetErrorString(ce)); }
    ce = cudaMemcpyAsync(h->trk_mem, t->params, TRK_TOWER * sizeof(float), cudaMemcpyHostToDevice, h->io_stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(h->trk_mem + off_stats, stats.data(), stats.size() * sizeof(double), cudaMemcpyHostToDevice, h->io_stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(h->trk_mem + off_prev, 0, (size_t)FW_TRK_ACT * N * sizeof(float), h->io_stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->io_stream);
    if (ce != cudaSuccess) {                  // the handle stays pending: a later call may try again
        cudaFree(h->trk_mem);
        h->trk_mem = nullptr;
        return fail(FW_ECUDA, "uploading the tracker: %s", cudaGetErrorString(ce));
    }
    FwTrk& k = h->trk;
    k.params = reinterpret_cast<const float*>(h->trk_mem);
    k.stats = t->obs_mean ? reinterpret_cast<const double*>(h->trk_mem + off_stats) : nullptr;
    k.clip = (float)t->clip_obs;
    k.h_lo = (float)t->h_range[0]; k.h_hi = (float)t->h_range[1];
    k.v_lo = (float)t->v_range[0]; k.v_hi = (float)t->v_range[1];
    k.prev = reinterpret_cast<float*>(h->trk_mem + off_prev);
    h->tracker_pending = false;
    return h->field_pending ? FW_OK : initial_episodes(h);
}

// the tracker entry points below need an installed tracker
static int need_tracker(const FwSim* h) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (h->dev.task != 5) return fail(FW_EINVAL, "the tracker entry points need a task 5 handle (has %d)", h->dev.task);
    if (h->tracker_pending) return fail(FW_ESTATE, "task 5: install the low-level tracker with fw_set_tracker first");
    return FW_OK;
}

extern "C" int fw_get_tracker_state(fw_handle h, float* prev_host) {
    if (!prev_host) return fail(FW_EINVAL, "null argument");
    int rc = need_tracker(h);
    if (rc != FW_OK) return rc;
    CU(cudaSetDevice(h->device));
    const size_t N = (size_t)h->n;
    std::vector<float> soa((size_t)FW_TRK_ACT * N);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(soa.data(), h->trk.prev, soa.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < N; ++i)
        for (int c = 0; c < FW_TRK_ACT; ++c) prev_host[i * FW_TRK_ACT + c] = soa[(size_t)c * N + i];
    return FW_OK;
}

extern "C" int fw_set_tracker_state(fw_handle h, const float* prev_host) {
    if (!prev_host) return fail(FW_EINVAL, "null argument");
    int rc = need_tracker(h);
    if (rc != FW_OK) return rc;
    CU(cudaSetDevice(h->device));
    const size_t N = (size_t)h->n;
    std::vector<float> soa((size_t)FW_TRK_ACT * N);
    for (size_t i = 0; i < N; ++i)
        for (int c = 0; c < FW_TRK_ACT; ++c) soa[(size_t)c * N + i] = prev_host[i * FW_TRK_ACT + c];
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(h->trk.prev, soa.data(), soa.size() * sizeof(float), cudaMemcpyHostToDevice));
    h->fresh = false;
    return FW_OK;
}

extern "C" int fw_set_tracker_obs_buffer(fw_handle h, float* obs_dev) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (h->dev.task != 5) return fail(FW_EINVAL, "fw_set_tracker_obs_buffer needs a task 5 handle (has %d)", h->dev.task);
    h->trk.obs_out = obs_dev;         // read by the step launches enqueued from now on (by value, at launch time)
    return FW_OK;
}

extern "C" int fw_num_envs(fw_handle h) { return h ? h->n : fail(FW_EINVAL, "null handle"); }
extern "C" int fw_obs_dim(fw_handle h) { return h ? h->obs_dim : fail(FW_EINVAL, "null handle"); }
extern "C" int fw_act_dim(fw_handle h) { return h ? h->dev.act_dim : fail(FW_EINVAL, "null handle"); }
extern "C" int64_t fw_launch_count(fw_handle h) { return h ? h->launches : 0; }

extern "C" int fw_reset(fw_handle h, const uint8_t* mask_dev, float* obs_dev, void* stream) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (need_field(h) != FW_OK) return FW_ESTATE;
    CU(cudaSetDevice(h->device));
    // the first whole-batch reset after fw_create only emits the observation of the episode-0 state
    const bool emit_only = h->fresh && mask_dev == nullptr;
    CU(fwk_launch_reset(h->dev, h->pl, mask_dev, obs_dev, emit_only, (cudaStream_t)stream));
    h->launches++;
    if (h->dev.task == 5 && !emit_only) {       // a reset episode starts with the tracker's previous action at zero
        CU(fwk_launch_tracker_clear(mask_dev, h->trk.prev, h->n, (cudaStream_t)stream));
        h->launches++;
    }
    h->fresh = false;
    h->dev_lane_dirty = true;
    return FW_OK;
}

extern "C" int fw_step(fw_handle h, const float* act_dev, float* obs_dev, float* rew_dev, uint8_t* flags_dev,
                       float* term_obs_dev, void* stream) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (!act_dev) return fail(FW_EINVAL, "act_dev is null");
    if ((reinterpret_cast<uintptr_t>(act_dev) & 15u) != 0) return fail(FW_EINVAL, "act_dev must be 16-byte aligned");
    if (need_field(h) != FW_OK) return FW_ESTATE;
    CU(cudaSetDevice(h->device));
    int rc = launch_step(h, h->dev, h->pl, act_dev, obs_dev, rew_dev, flags_dev, term_obs_dev, false, 1, (cudaStream_t)stream);
    if (rc != FW_OK) return rc;
    h->fresh = false;
    h->dev_lane_dirty = true;
    return FW_OK;
}

extern "C" int fw_step_random(fw_handle h, int32_t n_steps, float* rew_dev, uint8_t* flags_dev, void* stream) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (n_steps < 0) return fail(FW_EINVAL, "n_steps < 0");
    if (need_field(h) != FW_OK) return FW_ESTATE;
    CU(cudaSetDevice(h->device));
    h->fresh = false;
    h->dev_lane_dirty = true;
    for (int s = 0; s < n_steps; ++s) {
        int rc = launch_step(h, h->dev, h->pl, nullptr, nullptr, rew_dev, flags_dev, nullptr, true, 1, (cudaStream_t)stream);
        if (rc != FW_OK) return rc;
    }
    return FW_OK;
}

extern "C" int fw_rollout_random(const fw_handle* hs, int32_t n_handles, int32_t n_launches, int32_t steps_per_launch,
                                 int32_t use_graph, void* stream) {
    if (!hs || n_handles <= 0) return fail(FW_EINVAL, "empty handle list");
    if (n_launches < 0 || steps_per_launch < 1) return fail(FW_EINVAL, "bad launch counts");
    for (int k = 0; k < n_handles; ++k) {
        if (!hs[k]) return fail(FW_EINVAL, "null handle in list");
        if (hs[k]->device != hs[0]->device) return fail(FW_EINVAL, "handles of one rollout must share a device");
        if (hs[k]->dev.task == 5) return fail(FW_EINVAL, "fw_rollout_random does not run task 5 (high-level waypoints): use fw_step_random");
        if (need_field(hs[k]) != FW_OK) return FW_ESTATE;
        hs[k]->fresh = false;
        hs[k]->dev_lane_dirty = true;
    }
    CU(cudaSetDevice(hs[0]->device));
    cudaStream_t st = (cudaStream_t)stream;
    int done = 0;
    if (use_graph) {
        const int rounds = n_launches / n_handles, rem = n_launches % n_handles;
        if (rounds > 0) {
            int rc = multi_graph_get(g_multi, hs, n_handles, n_handles, steps_per_launch);
            if (rc != FW_OK) return rc;
            for (int r = 0; r < rounds; ++r) CU(cudaGraphLaunch(g_multi.exec, st));
            for (int k = 0; k < n_handles; ++k) hs[k]->launches += rounds * (hs[k]->spare_on ? 2 : 1);
        }
        if (rem > 0) {       // the tail of a launch count that is not a multiple of the list: one more (shorter) graph
            int rc = multi_graph_get(g_rem, hs, n_handles, rem, steps_per_launch);
            if (rc != FW_OK) return rc;
            CU(cudaGraphLaunch(g_rem.exec, st));
            for (int k = 0; k < rem; ++k) hs[k]->launches += hs[k]->spare_on ? 2 : 1;
        }
        done = n_launches;
    }
    for (int j = done; j < n_launches; ++j) {
        FwSim* h = hs[j % n_handles];
        int rc = launch_step(h, h->dev, h->pl, nullptr, nullptr, nullptr, nullptr, nullptr, true, steps_per_launch, st);
        if (rc != FW_OK) return rc;
    }
    return FW_OK;
}

static int ensure_host_io(FwSim* h) {
    if (h->h_act) return FW_OK;
    const size_t N = (size_t)h->n, D = (size_t)(h->obs_dim > 0 ? h->obs_dim : 1);
    const size_t Aw = (size_t)h->dev.act_dim;
    CU(cudaMallocHost((void**)&h->h_act, N * Aw * sizeof(float)));
    CU(cudaMallocHost((void**)&h->h_obs, N * D * sizeof(float)));
    CU(cudaMallocHost((void**)&h->h_rew, N * sizeof(float)));
    CU(cudaMallocHost((void**)&h->h_term, N * D * sizeof(float)));
    CU(cudaMallocHost((void**)&h->h_flg, N));
    CU(cudaMallocHost((void**)&h->h_tidx, N));
    memset(h->h_tidx, 0, N);
    CU(cudaMalloc((void**)&h->d_act, N * Aw * sizeof(float)));
    CU(cudaMalloc((void**)&h->d_obs, N * D * sizeof(float)));
    CU(cudaMalloc((void**)&h->d_rew, N * sizeof(float)));
    CU(cudaMalloc((void**)&h->d_term, N * D * sizeof(float)));
    CU(cudaMalloc((void**)&h->d_flg, N));
    CU(cudaMemset(h->d_term, 0, N * D * sizeof(float)));
    return FW_OK;
}

extern "C" int fw_step_host(fw_handle h, const float* act_host, float* obs_host, float* rew_host, uint8_t* flags_host,
                            float* term_obs_host) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (!act_host) return fail(FW_EINVAL, "act_host is null");
    if (need_field(h) != FW_OK) return FW_ESTATE;
    CU(cudaSetDevice(h->device));
    int rc = ensure_host_io(h);
    if (rc != FW_OK) return rc;
    rc = host_lane_enter(h);
    if (rc != FW_OK) return rc;
    const size_t N = (size_t)h->n, D = (size_t)h->obs_dim;
    // The batch is cut into chunks that alternate between two streams, so that the staging of caller-owned (pageable)
    // actions for chunk c+1 runs under the kernel of chunk c.  No DMA operation is issued at all (each costs several
    // microseconds of fixed latency, see the chunk sweep in DESIGN.md): the kernel reads the actions from and writes every
    // output to pinned host memory directly (unified addressing; posted PCIe writes, complete when the kernel is).
    const bool want_term = term_obs_host && D;
    // A caller buffer that is itself page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) is read by the
    // kernel in place, like the library's own staging buffer: no host-side copy at all.
    const float* act_dev_view = nullptr;
    if (act_host != h->h_act && (reinterpret_cast<uintptr_t>(act_host) & 15u) == 0) {
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, act_host) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer != nullptr)
            act_dev_view = static_cast<const float*>(pa.devicePointer);
        else
            (void)cudaGetLastError();
    }
    static const int tuned_chunks = [] {               // FWSIM_HOST_CHUNKS=<n> overrides the default (tuning aid)
        const char* e = getenv("FWSIM_HOST_CHUNKS");
        const int v = e ? atoi(e) : 0;
        return v >= 1 && v <= 64 ? v : FW_HOST_CHUNKS;
    }();
    const int chunks = h->n >= 16384 ? tuned_chunks : 1;
    const int per = (((h->n + chunks - 1) / chunks) + 63) / 64 * 64;
    // spare episodes: the previous step's request list is served on the side stream beside this step's chunk kernels, which
    // all append to the other list
    const int par = h->parity, prev = par ^ 1;
    if (h->spare_on) {
        CU(cudaEventRecord(h->ev_fork, h->io_streams[0]));
        CU(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
    }
    for (int c = 0; c < chunks; ++c) {
        const int c0 = c * per, c1 = (c + 1) * per < h->n ? (c + 1) * per : h->n;
        if (c0 >= c1) break;
        const size_t n0 = (size_t)c0, cn = (size_t)(c1 - c0);
        cudaStream_t st = h->io_streams[c & 1];
        const size_t Aw = (size_t)h->dev.act_dim;
        if (act_host != h->h_act && act_dev_view == nullptr) memcpy(h->h_act + n0 * Aw, act_host + n0 * Aw, cn * Aw * sizeof(float));
        FwDev pc = h->dev;
        pc.i_begin = c0; pc.i_end = c1;
        // Observations, rewards, flags and terminal observations are written by the kernel straight into the pinned
        // host buffers (unified addressing; the observation rows leave each CTA as one bulk store, so the PCIe writes
        // are 7 KB bursts).  Measured at 65,536 envs: 188 us per step against 200-212 us with a device buffer and a
        // D2H copy per chunk, and the terminal observations (rows of finished episodes only) cost nothing instead of
        // a second 7.3 MB copy.  FWSIM_HOST_ZEROCOPY_OBS=0 restores the copy-engine route.
        static const bool zc_obs = [] { const char* e = getenv("FWSIM_HOST_ZEROCOPY_OBS"); return !(e && atoi(e) == 0); }();
        float* obs_dst = D ? (zc_obs ? h->h_obs : h->d_obs) : nullptr;
        float* term_dst = want_term ? (zc_obs ? h->h_term : h->d_term) : nullptr;
        FwPlanes plh = h->pl;
        plh.tidx_out = h->h_tidx;          // info["num_targets_reached"] goes straight to the host like the flags
        if (h->spare_on) { plh.refill_list = h->refill_list[par]; plh.refill_count = h->refill_ctl + par; }
        CU(fwk_launch_step(pc, plh, act_dev_view ? act_dev_view : h->h_act, obs_dst, h->h_rew, h->h_flg, term_dst, false, 1, st,
                           &h->trk));
        h->launches++;
        if (!zc_obs) {
            if (obs_host && D) CU(cudaMemcpyAsync(h->h_obs + n0 * D, h->d_obs + n0 * D, cn * D * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (want_term) CU(cudaMemcpyAsync(h->h_term + n0 * D, h->d_term + n0 * D, cn * D * sizeof(float), cudaMemcpyDeviceToHost, st));
        }
    }
    h->fresh = false;
    if (h->spare_on) {
        CU(fwk_launch_refill(h->dev, h->pl, h->refill_list[prev], h->refill_ctl + prev, h->refill_ctl + 2 + prev, h->n, 0, h->side));
        h->launches++;
    }
    CU(cudaStreamSynchronize(h->io_streams[0]));
    if (chunks > 1) CU(cudaStreamSynchronize(h->io_streams[1]));
    if (h->spare_on) { CU(cudaStreamSynchronize(h->side)); h->parity ^= 1; }
    // buffers obtained from fw_host_buffers are the pinned staging itself: nothing left to copy
    if (obs_host && D && obs_host != h->h_obs) memcpy(obs_host, h->h_obs, N * D * sizeof(float));
    if (rew_host && rew_host != h->h_rew) memcpy(rew_host, h->h_rew, N * sizeof(float));
    if (flags_host && flags_host != h->h_flg) memcpy(flags_host, h->h_flg, N);
    if (term_obs_host && D && term_obs_host != h->h_term) memcpy(term_obs_host, h->h_term, N * D * sizeof(float));
    return FW_OK;
}

extern "C" int fw_host_buffers(fw_handle h, float** act, float** obs, float** rew, uint8_t** flags, float** term_obs) {
    if (!h) return fail(FW_EINVAL, "null handle");
    CU(cudaSetDevice(h->device));
    int rc = ensure_host_io(h);
    if (rc != FW_OK) return rc;
    if (act) *act = h->h_act;
    if (obs) *obs = h->h_obs;
    if (rew) *rew = h->h_rew;
    if (flags) *flags = h->h_flg;
    if (term_obs) *term_obs = h->h_term;
    return FW_OK;
}

extern "C" int fw_host_info_buffer(fw_handle h, uint8_t** targets_reached) {
    if (!h) return fail(FW_EINVAL, "null handle");
    CU(cudaSetDevice(h->device));
    int rc = ensure_host_io(h);
    if (rc != FW_OK) return rc;
    if (targets_reached) *targets_reached = h->h_tidx;
    return FW_OK;
}

extern "C" int fw_targets_reached(fw_handle h, uint8_t* dst_dev, void* stream) {
    if (!h || !dst_dev) return fail(FW_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    CU(cudaMemcpyAsync(dst_dev, h->pl.tidx_out, (size_t)h->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return FW_OK;
}

extern "C" int fw_set_obs_accumulator(fw_handle h, double* acc_dev) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (h->obs_dim <= 0 && acc_dev) return fail(FW_EINVAL, "this task has no observation");
    h->pl.obs_acc = acc_dev;          // read by the step launches enqueued from now on (by value, at launch time)
    return FW_OK;
}

extern "C" int fw_render(fw_handle h, int32_t env, int32_t width, int32_t height, uint8_t* rgba_dev, int32_t* seg_dev,
                         float* depth_dev, void* stream) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (env < 0 || env >= h->n) return fail(FW_EINVAL, "env index %d out of range [0,%d)", env, h->n);
    if (width <= 0 || height <= 0 || width > 4096 || height > 4096) return fail(FW_EINVAL, "frame size must be in [1,4096]");
    if (!rgba_dev && !seg_dev && !depth_dev) return fail(FW_EINVAL, "no output buffer");
    if (h->dev.task == 5) return fail(FW_EINVAL, "fw_render does not draw task 5 (high-level waypoints)");
    CU(cudaSetDevice(h->device));
    CU(fwk_render(h->dev, h->pl, env, width, height, rgba_dev, seg_dev, depth_dev, (cudaStream_t)stream));
    h->launches++;
    return FW_OK;
}

extern "C" int fw_fault_count(fw_handle h, int64_t* nonfinite_resets) {
    if (!h || !nonfinite_resets) return fail(FW_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    CU(cudaDeviceSynchronize());
    double v = 0.0;
    CU(cudaMemcpy(&v, h->pl.stats + 8, sizeof(double), cudaMemcpyDeviceToHost));
    *nonfinite_resets = (int64_t)v;
    return FW_OK;
}

static int reset_host_impl(fw_handle h, float* obs_host, bool observe_only);

extern "C" int fw_spare_stats(fw_handle h, int64_t out[2]) {
    if (!h || !out) return fail(FW_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    CU(cudaDeviceSynchronize());
    double v[2] = {0.0, 0.0};
    CU(cudaMemcpy(v, h->pl.stats + 9, 2 * sizeof(double), cudaMemcpyDeviceToHost));
    out[0] = (int64_t)v[0]; out[1] = (int64_t)v[1];
    return FW_OK;
}

extern "C" int fw_reset_host(fw_handle h, float* obs_host) { return reset_host_impl(h, obs_host, false); }
extern "C" int fw_observe_host(fw_handle h, float* obs_host) { return reset_host_impl(h, obs_host, true); }

static int reset_host_impl(fw_handle h, float* obs_host, bool observe_only) {
    if (!h) return fail(FW_EINVAL, "null handle");
    if (need_field(h) != FW_OK) return FW_ESTATE;
    CU(cudaSetDevice(h->device));
    int rc = ensure_host_io(h);
    if (rc != FW_OK) return rc;
    rc = host_lane_enter(h);
    if (rc != FW_OK) return rc;
    if (!observe_only) memset(h->h_tidx, 0, (size_t)h->n);
    const size_t N = (size_t)h->n, D = (size_t)h->obs_dim;
    cudaStream_t st = h->io_stream;
    CU(fwk_launch_reset(h->dev, h->pl, nullptr, D ? h->d_obs : nullptr, h->fresh || observe_only, st));
    h->launches++;
    if (h->dev.task == 5 && !(h->fresh || observe_only)) {
        CU(cudaMemsetAsync(h->trk.prev, 0, (size_t)FW_TRK_ACT * h->n * sizeof(float), st));
    }
    if (!observe_only) h->fresh = false;
    if (obs_host && D) CU(cudaMemcpyAsync(h->h_obs, h->d_obs, N * D * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (obs_host && D && obs_host != h->h_obs) memcpy(obs_host, h->h_obs, N * D * sizeof(float));
    return FW_OK;
}

// ------------------------------------------------------------------ state injection / inspection
struct HostPlanes {
    std::vector<float4> s[5];
    std::vector<int4> s5;
    std::vector<float4> w0, w1;
    std::vector<float> targets;
    std::vector<float4> dk, v0, v1, v2;
    std::vector<int4> v3;
    std::vector<float> obst;
    std::vector<float> hist;
};

static int pull(FwSim* h, HostPlanes& hp) {
    const size_t N = (size_t)h->n, T = (size_t)(h->cfg.num_targets > 0 ? h->cfg.num_targets : 1);
    float4* src[5] = {h->pl.s0, h->pl.s1, h->pl.s2, h->pl.s3, h->pl.s4};
    CU(cudaDeviceSynchronize());
    for (int k = 0; k < 5; ++k) { hp.s[k].resize(N); CU(cudaMemcpy(hp.s[k].data(), src[k], N * 16, cudaMemcpyDeviceToHost)); }
    hp.s5.resize(N); CU(cudaMemcpy(hp.s5.data(), h->pl.s5, N * 16, cudaMemcpyDeviceToHost));
    hp.w0.resize(N); CU(cudaMemcpy(hp.w0.data(), h->pl.w0, N * 16, cudaMemcpyDeviceToHost));
    hp.w1.resize(N); CU(cudaMemcpy(hp.w1.data(), h->pl.w1, N * 16, cudaMemcpyDeviceToHost));
    hp.targets.resize(T * 3 * N); CU(cudaMemcpy(hp.targets.data(), h->pl.targets, T * 3 * N * 4, cudaMemcpyDeviceToHost));
    if (h->cfg.task == 4) {
        hp.hist.resize((size_t)h->dev.hist_slots * N);
        CU(cudaMemcpy(hp.hist.data(), h->pl.hist, hp.hist.size() * 4, cudaMemcpyDeviceToHost));
    }
    if (h->cfg.task == 2 || h->cfg.task == 4) {
        hp.dk.resize(N); hp.v0.resize(N); hp.v1.resize(N); hp.v2.resize(N); hp.v3.resize(N);
        CU(cudaMemcpy(hp.dk.data(), h->pl.dk, N * 16, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(hp.v0.data(), h->pl.v0, N * 16, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(hp.v1.data(), h->pl.v1, N * 16, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(hp.v2.data(), h->pl.v2, N * 16, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(hp.v3.data(), h->pl.v3, N * 16, cudaMemcpyDeviceToHost));
        hp.obst.resize((size_t)FW_MAX_OBST * 3 * N);
        CU(cudaMemcpy(hp.obst.data(), h->pl.obst, (size_t)FW_MAX_OBST * 3 * N * 4, cudaMemcpyDeviceToHost));
    }
    return FW_OK;
}

static int push(FwSim* h, const HostPlanes& hp) {
    const size_t N = (size_t)h->n, T = (size_t)(h->cfg.num_targets > 0 ? h->cfg.num_targets : 1);
    float4* dst[5] = {h->pl.s0, h->pl.s1, h->pl.s2, h->pl.s3, h->pl.s4};
    for (int k = 0; k < 5; ++k) CU(cudaMemcpy(dst[k], hp.s[k].data(), N * 16, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->pl.s5, hp.s5.data(), N * 16, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->pl.w0, hp.w0.data(), N * 16, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->pl.w1, hp.w1.data(), N * 16, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->pl.targets, hp.targets.data(), T * 3 * N * 4, cudaMemcpyHostToDevice));
    if (h->cfg.task == 4) CU(cudaMemcpy(h->pl.hist, hp.hist.data(), hp.hist.size() * 4, cudaMemcpyHostToDevice));
    if (h->cfg.task == 2 || h->cfg.task == 4) {
        CU(cudaMemcpy(h->pl.dk, hp.dk.data(), N * 16, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(h->pl.v0, hp.v0.data(), N * 16, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(h->pl.v1, hp.v1.data(), N * 16, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(h->pl.v2, hp.v2.data(), N * 16, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(h->pl.v3, hp.v3.data(), N * 16, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(h->pl.obst, hp.obst.data(), (size_t)FW_MAX_OBST * 3 * N * 4, cudaMemcpyHostToDevice));
    }
    CU(cudaDeviceSynchronize());
    return FW_OK;
}

extern "C" int fw_get_state(fw_handle h, FwStateHost* s) {
    if (!h || !s) return fail(FW_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    HostPlanes hp;
    int rc = pull(h, hp);
    if (rc != FW_OK) return rc;
    const size_t N = (size_t)h->n;
    const int T = h->cfg.num_targets;
    for (size_t i = 0; i < N; ++i) {
        const float4 &a = hp.s[0][i], &b = hp.s[1][i], &c = hp.s[2][i], &d = hp.s[3][i], &f = hp.s[4][i];
        const int4& g = hp.s5[i];
        if (s->pos) { s->pos[3 * i] = a.x; s->pos[3 * i + 1] = a.y; s->pos[3 * i + 2] = a.z; }
        if (s->quat) { s->quat[4 * i] = b.x; s->quat[4 * i + 1] = b.y; s->quat[4 * i + 2] = b.z; s->quat[4 * i + 3] = b.w; }
        if (s->vel) { s->vel[3 * i] = c.x; s->vel[3 * i + 1] = c.y; s->vel[3 * i + 2] = c.z; }
        if (s->omega) { s->omega[3 * i] = d.x; s->omega[3 * i + 1] = d.y; s->omega[3 * i + 2] = d.z; }
        if (s->act) {
            float* o = s->act + 6 * i;
            o[0] = c.w; o[1] = d.w; o[2] = f.x; o[3] = f.y; o[4] = f.z; o[5] = a.w;
        }
        if (s->new_dist) s->new_dist[i] = f.w;
        if (s->step_count) s->step_count[i] = g.x;
        if (s->physics_steps) s->physics_steps[i] = g.y;
        if (s->episode) s->episode[i] = (uint32_t)g.z;
        if (s->target_idx) s->target_idx[i] = g.w;
        if (s->wind) {
            float* o = s->wind + 7 * i;
            o[0] = hp.w0[i].x; o[1] = hp.w0[i].y; o[2] = hp.w0[i].z;
            o[3] = hp.w1[i].x; o[4] = hp.w1[i].y; o[5] = hp.w1[i].z; o[6] = hp.w0[i].w;
        }
        if (s->targets)
            for (int t = 0; t < T; ++t)
                for (int k = 0; k < 3; ++k) s->targets[(i * T + t) * 3 + k] = hp.targets[(size_t)(t * 3 + k) * N + i];
        if (h->cfg.task == 4 && s->vis_hist) {
            // device slots: hist_len rows of 9, then 4 deltas; host layout: FW_MAX_HIST rows of 9, then 4 deltas
            float* o = s->vis_hist + (size_t)(FW_MAX_HIST * 9 + 4) * i;
            const int H = h->dev.hist_len;
            for (int k = 0; k < FW_MAX_HIST * 9 + 4; ++k) o[k] = 0.0f;
            for (int k = 0; k < 9 * H; ++k) o[k] = hp.hist[(size_t)k * N + i];
            for (int k = 0; k < 4; ++k) o[FW_MAX_HIST * 9 + k] = hp.hist[(size_t)(9 * H + k) * N + i];
        }
        if (h->cfg.task == 2 || h->cfg.task == 4) {
            const float4 &dk = hp.dk[i], &v0 = hp.v0[i], &v1 = hp.v1[i], &v2 = hp.v2[i];
            const int4& v3 = hp.v3[i];
            if (s->duck) { s->duck[3 * i] = dk.x; s->duck[3 * i + 1] = dk.y; s->duck[3 * i + 2] = dk.z; }
            if (s->ol_f) {
                float* o = s->ol_f + 12 * i;
                o[0] = v0.x; o[1] = v0.y; o[2] = v0.z; o[3] = v0.w; o[4] = v1.x; o[5] = v1.y; o[6] = v1.z; o[7] = v1.w;
                o[8] = v2.x; o[9] = v2.y; o[10] = v2.z; o[11] = v2.w;
            }
            if (s->ol_i) {
                int32_t* o = s->ol_i + 9 * i;
                o[0] = v3.x & 1; o[1] = (v3.x >> 1) & 1; o[2] = (v3.x >> 2) & 1; o[3] = (v3.x >> 3) & 1; o[4] = (v3.x >> 4) & 1;
                o[5] = v3.y; o[6] = v3.z; o[7] = v3.w; o[8] = (v3.x >> 8) & 0xff;
            }
            if (s->obst)
                for (int k = 0; k < FW_MAX_OBST; ++k)
                    for (int c = 0; c < 3; ++c) s->obst[(i * FW_MAX_OBST + k) * 3 + c] = hp.obst[(size_t)(k * 3 + c) * N + i];
        }
    }
    return FW_OK;
}

extern "C" int fw_set_state(fw_handle h, const FwStateHost* s) {
    if (!h || !s) return fail(FW_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    HostPlanes hp;
    int rc = pull(h, hp);
    if (rc != FW_OK) return rc;
    const size_t N = (size_t)h->n;
    const int T = h->cfg.num_targets;
    for (size_t i = 0; i < N; ++i) {
        float4 &a = hp.s[0][i], &b = hp.s[1][i], &c = hp.s[2][i], &d = hp.s[3][i], &f = hp.s[4][i];
        int4& g = hp.s5[i];
        if (s->pos) { a.x = s->pos[3 * i]; a.y = s->pos[3 * i + 1]; a.z = s->pos[3 * i + 2]; }
        if (s->quat) { b.x = s->quat[4 * i]; b.y = s->quat[4 * i + 1]; b.z = s->quat[4 * i + 2]; b.w = s->quat[4 * i + 3]; }
        if (s->vel) { c.x = s->vel[3 * i]; c.y = s->vel[3 * i + 1]; c.z = s->vel[3 * i + 2]; }
        if (s->omega) { d.x = s->omega[3 * i]; d.y = s->omega[3 * i + 1]; d.z = s->omega[3 * i + 2]; }
        if (s->act) {
            const float* o = s->act + 6 * i;
            c.w = o[0]; d.w = o[1]; f.x = o[2]; f.y = o[3]; f.z = o[4]; a.w = o[5];
        }
        if (s->new_dist) f.w = s->new_dist[i];
        if (s->step_count) g.x = s->step_count[i];
        if (s->physics_steps) g.y = s->physics_steps[i];
        if (s->episode) g.z = (int)s->episode[i];
        if (s->target_idx) g.w = s->target_idx[i];
        if (s->wind) {
            const float* o = s->wind + 7 * i;
            hp.w0[i] = make_float4(o[0], o[1], o[2], o[6]);
            hp.w1[i] = make_float4(o[3], o[4], o[5], 0.0f);
        }
        if (s->targets)
            for (int t = 0; t < T; ++t)
                for (int k = 0; k < 3; ++k) hp.targets[(size_t)(t * 3 + k) * N + i] = s->targets[(i * T + t) * 3 + k];
        if (h->cfg.task == 4 && s->vis_hist) {
            const float* o = s->vis_hist + (size_t)(FW_MAX_HIST * 9 + 4) * i;
            const int H = h->dev.hist_len;
            for (int k = 0; k < 9 * H; ++k) hp.hist[(size_t)k * N + i] = o[k];
            for (int k = 0; k < 4; ++k) hp.hist[(size_t)(9 * H + k) * N + i] = o[FW_MAX_HIST * 9 + k];
        }
        if (h->cfg.task == 2 || h->cfg.task == 4) {
            float4 &dk = hp.dk[i], &v0 = hp.v0[i], &v1 = hp.v1[i], &v2 = hp.v2[i];
            int4& v3 = hp.v3[i];
            if (s->duck) dk = make_float4(s->duck[3 * i], s->duck[3 * i + 1], s->duck[3 * i + 2], 0.0f);
            if (s->ol_f) {
                const float* o = s->ol_f + 12 * i;
                v0 = make_float4(o[0], o[1], o[2], o[3]); v1 = make_float4(o[4], o[5], o[6], o[7]);
                v2 = make_float4(o[8], o[9], o[10], o[11]);
            }
            if (s->ol_i) {
                const int32_t* o = s->ol_i + 9 * i;
                v3.x = (o[0] & 1) | ((o[1] & 1) << 1) | ((o[2] & 1) << 2) | ((o[3] & 1) << 3) | ((o[4] & 1) << 4) | ((o[8] & 0xff) << 8);
                v3.y = o[5]; v3.z = o[6]; v3.w = o[7];
            }
            if (s->obst)
                for (int k = 0; k < FW_MAX_OBST; ++k)
                    for (int c = 0; c < 3; ++c) hp.obst[(size_t)(k * 3 + c) * N + i] = s->obst[(i * FW_MAX_OBST + k) * 3 + c];
        }
    }
    h->fresh = false;
    return push(h, hp);
}

extern "C" int fw_episode_stats(fw_handle h, double out[8]) {
    if (!h || !out) return fail(FW_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, h->pl.stats, 8 * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemset(h->pl.stats, 0, 8 * sizeof(double)));
    return FW_OK;
}

// FP32 FMA-chain peak of the device, for the roofline denominator of the (FP32-bound) env-step kernel.
extern "C" int fw_measure_fp32_peak(int32_t device, double* tflops, int32_t* sm_count, int32_t* sm_clock_khz) {
    if (!tflops) return fail(FW_EINVAL, "null argument");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0) return fail(FW_ECUDA, "no CUDA device available (%s)", cudaGetErrorString(ce));
    if (device < 0 || device >= ndev) return fail(FW_EINVAL, "device out of range");
    CU(cudaSetDevice(device));
    int sms = 0, khz = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CU(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
    if (sm_count) *sm_count = sms;
    if (sm_clock_khz) *sm_clock_khz = khz;
    float* scratch = nullptr;
    CU(cudaMalloc((void**)&scratch, 64));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double flops = 0, best = 0;
    CU(fwk_fma_peak(sms, 2000, scratch, &flops, 0));   // warm-up
    CU(cudaDeviceSynchronize());
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0, 0));
        CU(fwk_fma_peak(sms, 20000, scratch, &flops, 0));
        CU(cudaEventRecord(e1, 0));
        CU(cudaEventSynchronize(e1));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        double tf = flops / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(scratch);
    *tflops = best;
    return FW_OK;
}
