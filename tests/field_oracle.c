/*
 * field_oracle.c -- fp64 reference of the gridded wind field (wind_mode 3), TEST INFRASTRUCTURE ONLY.
 *
 * Compiled by tests/field_oracle.py together with an unmodified copy of oracle/fw_oracle.c, whose two wind entry points are
 * renamed there (fwo_refresh_surface_vel -> fwo_refresh_surface_vel_uniform, sample_wind -> sample_wind_uniform): this file
 * provides the originals' names, delegating every other wind mode to them unchanged.  It restates the semantics of
 * include/fwsim.h FwWindField independently of the CUDA code: world-frame wind at lattice points origin + (i, j, k) * spacing,
 * values[nt][nz][ny][nx][3] float32, trilinear in space with coordinates clamped to the box, linear in time between slices
 * t_step apart and periodic over nt * t_step, evaluated in double at every surface's link CoM pos + R r_surf[s] minus the
 * episode's shift.  Per env, wind_base holds the shift, gust_phase the time offset (seconds) and gust_amp is zero.
 */

typedef struct {
    const float* values;
    int32_t nx, ny, nz, nt;
    double origin[3], spacing[3], t_step;
    double shift_lo[3], shift_hi[3];
    int32_t randomize_time, _pad;
} fwf_field;

/* the field of the wind_mode 3 configs this library is called with (set by the Python side before every call) */
static const fwf_field* g_field = NULL;

void fwf_set_field(const fwf_field* f) { g_field = f; }

static int fwf_axis(double x, double org, double sp, int n, double* f) {
    double g = (x - org) / sp;
    if (g < 0.0) g = 0.0;
    if (g > (double)(n - 1)) g = (double)(n - 1);
    int i0 = (int)floor(g);
    if (i0 > n - 1) i0 = n - 1;
    *f = g - (double)i0;
    return i0;
}

/* wind of field f at time t (seconds, offset included) and field-frame point x (shift already removed) */
void fwf_wind_at(const fwf_field* f, double t, const double x[3], double w[3]) {
    const int n[3] = {f->nx, f->ny, f->nz};
    int i0[3], i1[3];
    double fr[3];
    for (int k = 0; k < 3; ++k) {
        i0[k] = fwf_axis(x[k], f->origin[k], f->spacing[k], n[k], &fr[k]);
        i1[k] = i0[k] + 1 < n[k] ? i0[k] + 1 : n[k] - 1;
    }
    double u = t / f->t_step;
    u -= (double)f->nt * floor(u / (double)f->nt);
    int s0 = (int)floor(u);
    if (s0 > f->nt - 1) s0 = f->nt - 1;
    if (s0 < 0) s0 = 0;
    const int s1 = s0 + 1 < f->nt ? s0 + 1 : 0;
    const double ft = u - (double)s0;
    const size_t pts = (size_t)f->nx * f->ny * f->nz;
    for (int k = 0; k < 3; ++k) w[k] = 0.0;
    for (int sl = 0; sl < 2; ++sl) {
        const double ws = sl ? ft : 1.0 - ft;
        const float* base = f->values + (size_t)(sl ? s1 : s0) * pts * 3;
        for (int cz = 0; cz < 2; ++cz)
            for (int cy = 0; cy < 2; ++cy)
                for (int cx = 0; cx < 2; ++cx) {
                    const double wc = ws * (cx ? fr[0] : 1.0 - fr[0]) * (cy ? fr[1] : 1.0 - fr[1]) * (cz ? fr[2] : 1.0 - fr[2]);
                    const size_t idx = ((size_t)(cz ? i1[2] : i0[2]) * f->ny + (size_t)(cy ? i1[1] : i0[1])) * f->nx +
                                       (size_t)(cx ? i1[0] : i0[0]);
                    for (int k = 0; k < 3; ++k) w[k] += wc * (double)base[idx * 3 + k];
                }
    }
}

/* Fixedwing.update_state with the gridded field: each surface's local airflow minus the field at its own link CoM */
void fwo_refresh_surface_vel(const fwo_config* c, fwo_env* e, int stamp) {
    if (c->wind_mode != 3) {
        fwo_refresh_surface_vel_uniform(c, e, stamp);
        return;
    }
    double R[9];
    fwo_quat_to_mat(e->quat, R);
    const int on = g_field != NULL && stamp >= 0 && stamp >= c->wind_start_substep;
    for (int s = 0; s < FWO_NSURF; ++s) {
        double rw[3], wxr[3], vw[3], w[3] = {0.0, 0.0, 0.0};
        mat_vec(R, c->r_surf[s], rw);
        cross3(e->omega, rw, wxr);
        if (on) {
            double x[3];
            for (int k = 0; k < 3; ++k) x[k] = e->pos[k] + rw[k] - e->wind_base[k];
            fwf_wind_at(g_field, (double)stamp * c->dt + e->gust_phase, x, w);
        }
        for (int k = 0; k < 3; ++k) vw[k] = e->vel[k] + wxr[k] - w[k];
        matT_vec(R, vw, e->surf_vel[s]);
    }
}

/* per-episode draws of the field: shift ~ U(shift_lo, shift_hi), time offset ~ U(0, nt t_step); wind Philox stream, index 0 */
static void sample_wind(const fwo_config* c, fwo_env* e, uint64_t seed) {
    if (c->wind_mode != 3) {
        sample_wind_uniform(c, e, seed);
        return;
    }
    for (int k = 0; k < 3; ++k) { e->wind_base[k] = 0.0; e->gust_amp[k] = 0.0; }
    e->gust_phase = 0.0;
    if (!c->wind_randomize || g_field == NULL) return;
    uint32_t r[4];
    fwo_philox(seed, e->env_id, e->episode, 0u, STREAM_WIND, r);
    for (int k = 0; k < 3; ++k) e->wind_base[k] = g_field->shift_lo[k] + fwo_u01(r[k]) * (g_field->shift_hi[k] - g_field->shift_lo[k]);
    if (g_field->randomize_time) e->gust_phase = fwo_u01(r[3]) * (double)g_field->nt * g_field->t_step;
}
