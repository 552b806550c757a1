// glg_kernels.cuh -- sm_100a kernels of the env-step path.  One thread = one greenhouse env.
//
//   glg_step_kernel   : fused TomatoEnv.step (tomato_env.py:115-146): action->control (S1), parametric noise (S2),
//                       weather row fetch (TMA bulk copy of the block's rows k..k+Np into shared memory when the
//                       block is in lock-step), hoisting of the (u,d,p)-only work, n_sub RK4 substeps with the stage
//                       state in registers (R1-R3), time update (S3), observation (S4), reward + info (S5,S7),
//                       termination (S6), episode statistics (warp-shuffle reduction) and auto-reset (S8).
//   glg_reset_kernel  : TomatoEnv.reset (tomato_env.py:231-270) for a masked subset.
//   glg_evalf_kernel  : batched GreenLight::evalF (greenlight_model.cpp:96-120) as a pure function.
//   glg_fma_peak_*    : FMA throughput micro-benchmarks used as roofline denominators.
//
// HBM layout (all per-env data structure-of-arrays, index [field][env], so a warp's loads are 256-B contiguous):
//   x[28][B] f64, u[6][B] f64, timestep[B] i32, table[B] i32, time[2][B] f64, step_ctr[B] u32,
//   ep_return[B] f64, ep_len[B] i32, ep_info[11][B] f64 ; outputs obs[B][obs_dim] f32 (row-major: the layout SB3 /
//   torch policies consume), term_obs same, reward[B] f64, done[B] u8, info[11][B] f64.
//   Weather bank W[n_tables][rows][10] f64: row stride 80 B (16-B aligned => legal cp.async.bulk source).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "glg_controller.h"
#include "glg_model.h"
#include "glg_philox.h"
#include "glg_rk4.h"

#define GLG_NOBS_FIXED 23
// observation modules (observations.py:35-182); ids as in glg_config.obs_modules
#define GLG_MAXOBSMOD 8
#define GLG_OBS_STATE 1     // StateObservations: 27 uniform random numbers (observations.py:57)
#define GLG_OBS_CLIMATE 2   // IndoorClimateObservations (4)
#define GLG_OBS_CROP 3      // BasicCropObservations (3)
#define GLG_OBS_CONTROL 4   // ControlObservations (6)
#define GLG_OBS_WEATHER 5   // WeatherObservations (5)
#define GLG_OBS_TIME 6      // TimeObservations (5)
#define GLG_OBS_FORECAST 7  // WeatherForecastObservations (5 Np)
#define GLG_NOBS_STATE 27
#define GLG_NINFO 11
#define GLG_NSTATS 16

struct GlgUniform {  // passed as a __grid_constant__ kernel parameter: lives in the constant bank, no global state
    double P[GLG_NP];
    double K[K_COUNT];
    double C[C_COUNT];
    float Kf[K_COUNT];  // fp32 copies for the throughput mode (precision = 1)
    float Cf[C_COUNT];
};

struct GlgStepArgs {
    int B, n_sub, N, Np, rows, n_tables, obs_dim, auto_reset, raw_control, n_reset_tables;
    int integrator;  // 0 fixed-step, 1 graded (kernel B's guarded loop)
    // observation row layout (tomato_env.py:77-96,193-198): ordered module list, offset of each module in the row
    int obs_nmod, obs_mod[GLG_MAXOBSMOD], obs_off[GLG_MAXOBSMOD];
    int fc_off;      // offset of the forecast block in the row, -1 if the stack has no WeatherForecastObservations
    int role_lanes;  // kernel B: envs per CTA (<= 32); fewer envs per CTA = more CTAs = more resident warps for small batches
    // raw_control: 0 = actions through S1, 1 = caller's controls as-is, 2 = rule-based controller evaluated in the prologue
    double ctrl[GLG_NCTRL];  // rule-based controller settings (glg_controller.h)
    double dt;
    double u_min[GLG_NU], u_max[GLG_NU];
    float delta_u_max_f32;
    double con_low[3], con_high[3];
    double elec_price, heating_price, co2_price, fruit_price, dmfm, fixed_costs;
    double uncertainty_scale;
    unsigned long long seed;
    long long env_id_offset;
    const float *actions;     // [B][6]
    const double *controls;   // [B][6] (raw control mode)
    const double *noise;      // [B][34] or null
    const double *weather;    // [n_tables][rows][10]
    const double *start_day;  // [n_tables]
    const int *reset_tables;  // [n_reset_tables]
    double *x, *u, *time, *ep_return, *ep_info;
    int *timestep, *table, *ep_len;
    unsigned int *step_ctr;
    float *obs, *term_obs;
    float *obs_head;  // [B][obs_dim - 5 Np]: the row without its forecast block, packed (host path glg_step_host_split)
    double *reward, *info, *stats;
    unsigned char *done;
};

// ---------------------------------------------------------------------------------------------------------
// shared-memory column views: element i of thread t lives at base[i*NT + t]  (conflict-free for 8-byte words)
// ---------------------------------------------------------------------------------------------------------
template <int NT>
struct GlgCol {
    double *b;
    __device__ __forceinline__ double &operator[](int i) { return b[i * NT]; }
    __device__ __forceinline__ double operator[](int i) const { return b[i * NT]; }
};
template <int NT>
struct GlgSmemStore {
    double *b;  // x at rows [0,28), acc at rows [28,56)
    __device__ __forceinline__ double &x(int i) { return b[i * NT]; }
    __device__ __forceinline__ double &acc(int i) { return b[(GLG_NX + i) * NT]; }
};
struct GlgConstView {  // read-only view of a constant-bank array
    const double *b;
    __device__ __forceinline__ double operator[](int i) const { return b[i]; }
};
struct GlgConstViewF {
    const float *b;
    __device__ __forceinline__ float operator[](int i) const { return b[i]; }
};
template <class T, int NT>
struct GlgColT {  // shared-memory column of scalar type T
    T *b;
    __device__ __forceinline__ T &operator[](int i) { return b[i * NT]; }
    __device__ __forceinline__ T operator[](int i) const { return b[i * NT]; }
};

// ---------------------------------------------------------------------------------------------------------
// TMA (1-D bulk async copy) + mbarrier wrappers, sm_90+ PTX
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t glg_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void glg_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(glg_smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void glg_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(glg_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void glg_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     glg_smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(glg_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void glg_mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok = 0;
    const uint32_t a = glg_smem_u32(bar);
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// env-step semantics shared by the step and reset kernels
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double glg_dens2ppm(double t, double dens) {  // utils.py:352-361
    return 1e6 * 8.3144598 * (t + 273.15) * dens / (101325 * 44.01e-3);
}
__device__ __forceinline__ double glg_clamp(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }
__device__ __forceinline__ double glg_rh(double t, double vp) {  // utils.py:363-364
    return glg_clamp(100 * vp / glg_satvp(t), 0., 100.);
}

// init_state(): environments/utils.py:13-46 (rhMax=90, time 0)
__device__ __forceinline__ void glg_init_state(const double *w0, double *x) {
    const double t0 = 16.5;
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) x[i] = t0;
    x[0] = w0[3];
    x[1] = x[0];
    x[4] = t0 + 4;
    x[11] = 0.25 * (3. * t0 + w0[6]);
    x[12] = 0.25 * (2. * t0 + 2 * w0[6]);
    x[13] = 0.25 * (t0 + 3 * w0[6]);
    x[14] = w0[6];
    x[15] = 90 / 100. * glg_satvp(t0);
    x[16] = x[15];
    x[21] = x[4];
    x[22] = 0.;
    x[23] = 9.5283e4;
    x[24] = 2.5107e5;
    x[25] = 5.5338e4;
    x[26] = 3.0978e3;
    x[27] = 0.;
}

// The 7 state-dependent observation entries: co2_air [ppm], temp_air, rh_air, pipe_temp (IndoorClimateObservations), 24CanTemp,
// cFruit, tSum (BasicCropObservations).  Also the state estimator's measurement function h(x) (glg_est.cuh).
__device__ __forceinline__ void glg_obs_state7(const double *x, double *hd) {
    hd[0] = glg_dens2ppm(x[2], x[0] * 1e-6);
    hd[1] = x[2];
    hd[2] = glg_rh(x[2], x[15]);
    hd[3] = x[9];
    hd[4] = x[21];
    hd[5] = x[25];
    hd[6] = x[26];
}

// The 23 entries of the five per-env modules (observations.py:59-161) for state x, controls u, weather row w, timestep k
// (pre-increment), day_of_year, hour_of_day, in the canonical order climate(4) crop(3) control(6) weather(5) time(5), fp64.
__device__ __forceinline__ void glg_obs_head(const double *x, const double *u, const double *w, int k, double doy,
                                             double hod, double *hd) {
    const double two_pi = 2 * 3.14159265358979323846;
    glg_obs_state7(x, hd);
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) hd[7 + i] = u[i];
    hd[13] = w[0];
    hd[14] = w[1];
    hd[15] = glg_rh(w[1], w[2]);
    hd[16] = glg_dens2ppm(w[1], w[3] * 1e-6);
    hd[17] = w[4];
    hd[18] = (double)k;
    double s, c;
    sincos(two_pi * doy / 365.0, &s, &c);
    hd[19] = s;
    hd[20] = c;
    sincos(two_pi * hod / 24.0, &s, &c);
    hd[21] = s;
    hd[22] = c;
}
// Writes the per-env part of one observation row in the configured module order (everything but the forecast block, which
// the whole CTA writes cooperatively) and returns the row's first three entries in fp64: the reward's constraint terms
// read obs[[0, 1, 2]] whatever the stack puts there (rewards.py:191-198).  wnext = weather row k+1 (first forecast row).
// StateObservations is `np.random.rand(27)` in the reference (global numpy RNG, observations.py:57): here 27 Philox uniforms
// keyed by (seed, global env id, step counter), draw blocks 96.. (disjoint from the noise and reset-table blocks).
// hrow (may be NULL): the same row without the forecast block, packed.
__device__ __forceinline__ void glg_write_obs_row(const GlgStepArgs &A, const double *hd, const double *wnext, unsigned long long env_id,
                                                  unsigned int ctr, float *orow, float *hrow, double *o3) {
    const int seg0[5] = {0, 4, 7, 13, 18}, segn[5] = {4, 3, 6, 5, 5};
#pragma unroll 1
    for (int m = 0; m < A.obs_nmod; ++m) {
        const int id = A.obs_mod[m], off = A.obs_off[m];
        const int hoff = (A.fc_off >= 0 && off > A.fc_off) ? off - 5 * A.Np : off;
        if (id >= GLG_OBS_CLIMATE && id <= GLG_OBS_TIME) {
            const int s0 = seg0[id - GLG_OBS_CLIMATE], n = segn[id - GLG_OBS_CLIMATE];
#pragma unroll 1
            for (int i = 0; i < n; ++i) {
                const double v = hd[s0 + i];
                orow[off + i] = (float)v;
                if (hrow) hrow[hoff + i] = (float)v;
                if (off + i < 3) o3[off + i] = v;
            }
        } else if (id == GLG_OBS_STATE) {
#pragma unroll 1
            for (int b = 0; b < (GLG_NOBS_STATE + 1) / 2; ++b) {
                const GlgPhilox4 r = glg_philox4x32_10(96u + (uint32_t)b, ctr, (uint32_t)env_id, (uint32_t)(env_id >> 32),
                                                       (uint32_t)A.seed, (uint32_t)(A.seed >> 32));
                const double v0 = glg_u01(r.v[0], r.v[1]), v1 = glg_u01(r.v[2], r.v[3]);
                orow[off + 2 * b] = (float)v0;
                if (hrow) hrow[hoff + 2 * b] = (float)v0;
                if (off + 2 * b < 3) o3[off + 2 * b] = v0;
                if (2 * b + 1 < GLG_NOBS_STATE) {
                    orow[off + 2 * b + 1] = (float)v1;
                    if (hrow) hrow[hoff + 2 * b + 1] = (float)v1;
                    if (off + 2 * b + 1 < 3) o3[off + 2 * b + 1] = v1;
                }
            }
        } else if (id == GLG_OBS_FORECAST) {
#pragma unroll 1
            for (int i = 0; off + i < 3 && i < 5 * A.Np; ++i) o3[off + i] = wnext[(i / 5) * GLG_ND + (i % 5)];
        }
    }
}

__device__ __forceinline__ double glg_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------------------
// building blocks shared by the two step kernels
// ---------------------------------------------------------------------------------------------------------

// Stages the block's weather rows kw..kw+Np of table tbl with ONE TMA bulk copy when every env of the block is in
// lock-step (same table, same timestep).  Returns 1 and the common (bk, bt) in that case; all threads must call it.
__device__ __forceinline__ int glg_stage_weather(const GlgStepArgs &A, double *s_wtile, uint64_t *s_bar, int *s_misc,
                                                 bool active, int kw, int tbl, int &bk, int &bt) {
    if (threadIdx.x == 0) {
        s_misc[0] = kw;
        s_misc[1] = tbl;
        glg_mbar_init(s_bar, 1);
    }
    __syncthreads();
    bk = s_misc[0];
    bt = s_misc[1];
    const int uniform = __syncthreads_and(!active || (kw == bk && tbl == bt));
    if (uniform) {
        const uint32_t tile_bytes = (uint32_t)((A.Np + 1) * GLG_ND * sizeof(double));
        if (threadIdx.x == 0) {
            glg_mbar_expect_tx(s_bar, tile_bytes);
            glg_bulk_g2s(s_wtile, A.weather + ((size_t)bt * A.rows + (size_t)bk) * GLG_ND, tile_bytes, s_bar);
        }
        glg_mbar_wait(s_bar, 0);
    }
    return uniform;
}

// S1 (action -> control), state load, S2 (parametric noise) and hoisting for env e.  Fills x[28], u[6], d[7..],
// the H column and (NOISY) the per-env crop-constant column.
template <bool NOISY, class HC, class CC>
__device__ __forceinline__ void glg_env_prologue(const GlgUniform &U, const GlgStepArgs &A, int e, const double *wrow,
                                                 unsigned int ctr, HC &Hc, CC &Cc, double *x, double *u, double *d) {
    const int B = A.B;
#pragma unroll
    for (int i = 0; i < 7; ++i) d[i] = wrow[i];
    // S1: tomato_env.py:109-113 (float32 action * float32 delta, then float64 add and clip) or raw control :148-149
    if (A.raw_control == 2) {
        // baseline.py:68-227 on the state before the step, the full weather row and the pre-step clock
        // (experiments/evaluate_baseline.py:21-23), then used as-is like step_raw_control
        double xc[GLG_NX], dc[GLG_ND];
#pragma unroll
        for (int i = 0; i < GLG_NX; ++i) xc[i] = (i == 0 || i == 2 || i == 15) ? A.x[(size_t)i * B + e] : 0.0;
#pragma unroll
        for (int i = 0; i < GLG_ND; ++i) dc[i] = wrow[i];
        glg_rule_control(A.ctrl, xc, dc, A.time[(size_t)B + e], A.time[e], u);
    } else if (A.raw_control) {
#pragma unroll
        for (int i = 0; i < GLG_NU; ++i) u[i] = A.controls[(size_t)e * GLG_NU + i];
    } else {
#pragma unroll
        for (int i = 0; i < GLG_NU; ++i) {
            const float prod = __fmul_rn(A.actions[(size_t)e * GLG_NU + i], A.delta_u_max_f32);
            u[i] = glg_clamp(A.u[(size_t)i * B + e] + (double)prod, A.u_min[i], A.u_max[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) A.u[(size_t)i * B + e] = u[i];
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) x[i] = A.x[(size_t)i * B + e];
    if (NOISY) {
        // noise.py:16-22: p'[i] = f32(p[i] + n_i p[i]), i in 128..161 ; p'[144] = f32(p'[141] / p'[142])
        double pl[GLG_NP];
        double n34[34];
        if (A.noise) {
#pragma unroll 1
            for (int i = 0; i < 34; ++i) n34[i] = A.noise[(size_t)e * 34 + i];
        } else {
            glg_noise34(A.seed, (unsigned long long)(A.env_id_offset + e), ctr, A.uncertainty_scale, n34);
        }
#pragma unroll 1
        for (int i = 0; i < GLG_NP; ++i) pl[i] = U.P[i];
#pragma unroll 1
        for (int i = 0; i < 34; ++i) {
            const double pv = U.P[128 + i];
            pl[128 + i] = (double)__double2float_rn(pv + n34[i] * pv);
        }
        pl[144] = (double)__fdiv_rn(__double2float_rn(pl[141]), __double2float_rn(pl[142]));
        double Cl[C_COUNT];
        glg_make_c(pl, Cl);
#pragma unroll
        for (int i = 0; i < C_COUNT; ++i) Cc[i] = Cl[i];
        glg_hoist(pl, u, d, Hc);
    } else {
        glg_hoist(GlgConstView{U.P}, u, d, Hc);
    }
}

struct GlgEnvOut {  // what the per-env epilogue hands to the block-level phases
    int done, k_obs, tbl_obs, k_term, tbl_term;
    double fin_ret, fin_len, fin_info[GLG_NINFO];
};

// S3..S8 for env e after the integration: time update, observation head, termination, reward/info, episode
// accumulators, SB3-style auto-reset, state write-back.  x holds the integrated state (restored if bad).
__device__ __forceinline__ void glg_env_epilogue(const GlgUniform &U, const GlgStepArgs &A, int e, int k, int kw, int tbl,
                                                 const double *wrow, double *x, double fruit_prev, int bad,
                                                 unsigned int ctr, GlgEnvOut &o) {
    const int B = A.B;
    const size_t table_stride = (size_t)A.rows * GLG_ND;
    int done = 0;
    if (bad) {
        // reference: evalF raised -> x unchanged, terminated (tomato_env.py:119-123)
#pragma unroll
        for (int i = 0; i < GLG_NX; ++i) x[i] = A.x[(size_t)i * B + e];
        done = 1;
    }
    // S3: time update (tomato_env.py:126-128)
    double doy = A.time[e], hod = A.time[(size_t)B + e];
    doy += fmod(A.dt / 86400.0, 365.0);
    hod = fmod(hod + A.dt / 3600.0, 24.0);
    // S4: observation head with the pre-increment timestep
    double u[GLG_NU], d[GLG_ND];
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) u[i] = A.u[(size_t)i * B + e];
#pragma unroll
    for (int i = 0; i < 5; ++i) d[i] = wrow[i];
    double hd[GLG_NOBS_FIXED];
    double o3[3] = {0.0, 0.0, 0.0};
    glg_obs_head(x, u, d, k, doy, hod, hd);
    float *orow = A.obs + (size_t)e * A.obs_dim;
    const unsigned long long env_gid = (unsigned long long)(A.env_id_offset + e);
    // the row of this step: written to obs, or (when the env terminates and resets in place) to the terminal observation
    float *step_row = orow;
    float *hrow = A.obs_head + (size_t)e * (A.obs_dim - (A.fc_off >= 0 ? 5 * A.Np : 0));
    // S6: termination (tomato_env.py:68-75,131-132)
    if (k >= A.N) done = 1;
    if (done && A.auto_reset) step_row = A.term_obs + (size_t)e * A.obs_dim;
    glg_write_obs_row(A, hd, wrow + GLG_ND, env_gid, ctr, step_row, step_row == orow ? hrow : nullptr, o3);
    // S5/S7: reward and info with the nominal parameters (rewards.py:156-231), same operation order
    double reward, info[GLG_NINFO];
    {
        const double dt = A.dt;
        const double heat_costs = u[0] * U.P[108] / U.P[46] * dt / 3600 * 1e-3 * A.heating_price;
        const double elec_costs = u[4] * U.P[172] * dt / 3600 * 1e-3 * A.elec_price;
        const double co2_costs = u[1] * U.P[109] / U.P[46] * dt * 1e-6 * A.co2_price;
        const double variable_costs = 0 + heat_costs + co2_costs + elec_costs;
        const double gains = (x[25] - fruit_prev) * 1e-6 / A.dmfm * A.fruit_price;
        const double profit = gains - variable_costs;
        const double max_profit = U.P[154] * dt * 1e-6 / A.dmfm * A.fruit_price;
        const double max_heating = U.P[108] / U.P[46] * dt / 3600 * 1e-3 * A.heating_price;
        const double max_elec = U.P[172] * dt / 3600 * 1e-3 * A.elec_price;
        const double max_co2 = U.P[109] / U.P[46] * dt * 1e-6 * A.co2_price;
        const double min_profit = -(0 + max_heating + max_elec + max_co2);
        const double max_viol[3] = {2500, 15, 15};
        double viol[3], pen = 0.0;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double lo = fmax(A.con_low[j] - o3[j], 0.0), hi = fmax(o3[j] - A.con_high[j], 0.0);
            viol[j] = lo + hi;
            pen += viol[j] / max_viol[j];
        }
        reward = (profit - min_profit) / (max_profit - min_profit) - pen - 0.0;  // lamp penalty is 0: rewards.py:203-216
        info[0] = profit; info[1] = gains; info[2] = variable_costs; info[3] = A.fixed_costs;
        info[4] = co2_costs; info[5] = heat_costs; info[6] = elec_costs;
        info[7] = viol[1]; info[8] = viol[0]; info[9] = viol[2]; info[10] = 0.0;
    }
    A.reward[e] = reward;
    A.done[e] = (unsigned char)done;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) A.info[(size_t)j * B + e] = info[j];
    // episode accumulators
    const double ep_ret = A.ep_return[e] + reward;
    const int ep_len = A.ep_len[e] + 1;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) info[j] += A.ep_info[(size_t)j * B + e];

    k += 1;
    o.k_obs = kw;
    o.tbl_obs = tbl;
    o.k_term = -1;
    o.tbl_term = 0;
    if (done && A.auto_reset) {
        // SB3 VecEnv semantics: keep the terminal observation (written above), then reset in place (tomato_env.py:231-270)
        o.k_term = kw;
        o.tbl_term = tbl;
        tbl = A.n_reset_tables > 1
                  ? A.reset_tables[glg_rand_below(A.seed, (unsigned long long)(A.env_id_offset + e), ctr, (uint32_t)A.n_reset_tables)]
                  : A.reset_tables[0];
        const double *w0 = A.weather + (size_t)tbl * table_stride;
#pragma unroll
        for (int i = 0; i < 7; ++i) d[i] = w0[i];
        glg_init_state(d, x);
#pragma unroll
        for (int i = 0; i < GLG_NU; ++i) {
            u[i] = 0.0;
            A.u[(size_t)i * B + e] = 0.0;
        }
        k = 0;
        doy = A.start_day[tbl];
        hod = 0.0;
        glg_obs_head(x, u, d, 0, doy, hod, hd);
        double o3r[3];
        glg_write_obs_row(A, hd, w0 + GLG_ND, env_gid, ctr + 0x80000000u, orow, hrow, o3r);
        o.k_obs = 0;
        o.tbl_obs = tbl;
    }
    // state out
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) A.x[(size_t)i * B + e] = x[i];
    A.timestep[e] = k;
    A.table[e] = tbl;
    A.time[e] = doy;
    A.time[(size_t)B + e] = hod;
    A.step_ctr[e] = ctr + 1u;
    A.ep_return[e] = done ? 0.0 : ep_ret;
    A.ep_len[e] = done ? 0 : ep_len;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) A.ep_info[(size_t)j * B + e] = done ? 0.0 : info[j];
    o.done = done;
    o.fin_ret = done ? ep_ret : 0.0;
    o.fin_len = done ? (double)ep_len : 0.0;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) o.fin_info[j] = done ? info[j] : 0.0;
}

// Finished-episode statistics: warp-shuffle reduction, one atomic per warp and entry.  Full-warp call.
__device__ __forceinline__ void glg_stats_reduce(const GlgStepArgs &A, bool active, int bad, const GlgEnvOut &o) {
    const unsigned any_done = __ballot_sync(0xffffffffu, active && o.done);
    if (!any_done) return;
    const double cnt = glg_warp_sum((active && o.done) ? 1.0 : 0.0);
    const double ret = glg_warp_sum(o.fin_ret);
    const double len = glg_warp_sum(o.fin_len);
    const double nbad = glg_warp_sum((active && bad) ? 1.0 : 0.0);
    double isum[GLG_NINFO];
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) isum[j] = glg_warp_sum(o.fin_info[j]);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(A.stats + 0, cnt);
        atomicAdd(A.stats + 1, ret);
        atomicAdd(A.stats + 2, len);
#pragma unroll
        for (int j = 0; j < GLG_NINFO; ++j) atomicAdd(A.stats + 3 + j, isum[j]);
        atomicAdd(A.stats + 14, nbad);
    }
}

// S4 forecast block: obs[23 + 5*(i-1) + c] = weather[k+i][c], i=1..Np, c<5 (observations.py:179-182), written
// cooperatively by the whole block so each row's 5*Np floats are stored with coalesced accesses.  NR rows/block.
__device__ __forceinline__ void glg_write_forecast(const GlgStepArgs &A, int NR, const int *s_tbl, const int *s_k,
                                                   const int *s_tbl_t, const int *s_k_t, const double *s_wtile,
                                                   int uniform, int bk, int bt) {
    if (A.fc_off < 0) return;  // the observation stack has no forecast block
    const size_t table_stride = (size_t)A.rows * GLG_ND;
    const int nf = 5 * A.Np;
    const int row0 = blockIdx.x * NR;
#pragma unroll 1
    for (int r = 0; r < NR; ++r) {
        const int kk = s_k[r];
        if (kk < 0) continue;
        const int tb = s_tbl[r];
        const double *src = (uniform && tb == bt && kk == bk) ? s_wtile : (A.weather + (size_t)tb * table_stride + (size_t)kk * GLG_ND);
        float *orow = A.obs + (size_t)(row0 + r) * A.obs_dim + A.fc_off;
        for (int j = threadIdx.x; j < nf; j += blockDim.x) {
            const int i = j / 5, c = j - 5 * i;
            orow[j] = (float)src[(size_t)(1 + i) * GLG_ND + c];
        }
        const int kt = s_k_t[r];
        if (kt >= 0) {
            const double *srct = A.weather + (size_t)s_tbl_t[r] * table_stride + (size_t)kt * GLG_ND;
            float *trow = A.term_obs + (size_t)(row0 + r) * A.obs_dim + A.fc_off;
            for (int j = threadIdx.x; j < nf; j += blockDim.x) {
                const int i = j / 5, c = j - 5 * i;
                trow[j] = (float)srct[(size_t)(1 + i) * GLG_ND + c];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// step kernel A: one thread = one env, the whole RHS in one instruction stream (large batches)
// ---------------------------------------------------------------------------------------------------------
template <int NT, bool NOISY>
struct GlgStepSmem {
    static constexpr int kColRows = 2 * GLG_NX + H_COUNT + (NOISY ? C_COUNT : 0);
    __host__ __device__ static size_t bytes(int Np) {
        return sizeof(double) * ((size_t)kColRows * NT + (size_t)(Np + 1) * GLG_ND) + 16 /*mbarrier*/ + sizeof(int) * (4 * NT + 4);
    }
};

template <bool GENERAL, bool NOISY, int NT>
__global__ void __launch_bounds__(NT) glg_step_kernel(const __grid_constant__ GlgUniform U, const __grid_constant__ GlgStepArgs A) {
    glg_exp_tbl_fill();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *s_wtile = reinterpret_cast<double *>(smem_raw);                         // [(Np+1)][10], 16-B aligned
    double *s_cols = s_wtile + (size_t)(A.Np + 1) * GLG_ND;                          // [kColRows][NT]
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_cols + (size_t)GlgStepSmem<NT, NOISY>::kColRows * NT);
    int *s_tbl = reinterpret_cast<int *>(s_bar + 2);  // obs source table per row
    int *s_k = s_tbl + NT;                            // obs source timestep per row (-1: no env)
    int *s_tbl_t = s_k + NT;                          // terminal-obs source (done rows)
    int *s_k_t = s_tbl_t + NT;                        // -1: not done
    int *s_misc = s_k_t + NT;

    const int tid = threadIdx.x;
    const int e = blockIdx.x * NT + tid;
    const bool active = e < A.B;
    int k = 0, tbl = 0;
    if (active) {
        k = A.timestep[e];
        tbl = A.table[e];
    }
    // weather row used by this step; clamped so a terminated env without auto-reset never reads past its table
    const int kw = min(k, A.rows - A.Np - 1);
    int bk, bt;
    const int uniform = glg_stage_weather(A, s_wtile, s_bar, s_misc, active, kw, tbl, bk, bt);

    GlgEnvOut o;
    o.done = 0; o.k_obs = -1; o.tbl_obs = 0; o.k_term = -1; o.tbl_term = 0; o.fin_ret = 0.0; o.fin_len = 0.0;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) o.fin_info[j] = 0.0;
    int bad = 0;
    if (active) {
        const double *wrow = uniform ? s_wtile : (A.weather + ((size_t)tbl * A.rows + (size_t)kw) * GLG_ND);
        GlgCol<NT> Hc{s_cols + (size_t)(2 * GLG_NX) * NT + tid};
        GlgCol<NT> Cc{s_cols + (size_t)(2 * GLG_NX + H_COUNT) * NT + tid};
        GlgSmemStore<NT> st{s_cols + tid};
        double x[GLG_NX], u[GLG_NU], d[GLG_ND];
        const unsigned int ctr = A.step_ctr[e];
        glg_env_prologue<NOISY>(U, A, e, wrow, ctr, Hc, Cc, x, u, d);
        const double fruit_prev = x[25];
        if (NOISY) bad = glg_rk4_step<GENERAL>(GlgConstView{U.K}, Cc, Hc, GlgConstView{U.P}, u, d, x, A.dt, A.n_sub, st, A.integrator);
        else bad = glg_rk4_step<GENERAL>(GlgConstView{U.K}, GlgConstView{U.C}, Hc, GlgConstView{U.P}, u, d, x, A.dt, A.n_sub, st, A.integrator);
        glg_env_epilogue(U, A, e, k, kw, tbl, wrow, x, fruit_prev, bad, ctr, o);
    }
    s_tbl[tid] = o.tbl_obs;
    s_k[tid] = o.k_obs;
    s_tbl_t[tid] = o.tbl_term;
    s_k_t[tid] = o.k_term;
    glg_stats_reduce(A, active, bad, o);
    __syncthreads();
    glg_write_forecast(A, NT, s_tbl, s_k, s_tbl_t, s_k_t, s_wtile, uniform, bk, bt);
}

// ---------------------------------------------------------------------------------------------------------
// reset kernel: tomato_env.py:231-270 for the envs selected by mask (NULL = all)
// ---------------------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(NT) glg_reset_kernel(const __grid_constant__ GlgStepArgs A, const unsigned char *mask,
                                                       const int *table_ids) {
    glg_exp_tbl_fill();
    const int e = blockIdx.x * NT + threadIdx.x;
    if (e >= A.B) return;
    if (mask && !mask[e]) return;
    const int B = A.B;
    const unsigned int ctr = A.step_ctr[e];
    int tbl;
    if (table_ids) tbl = table_ids[e];
    else
        tbl = A.n_reset_tables > 1
                  ? A.reset_tables[glg_rand_below(A.seed, (unsigned long long)(A.env_id_offset + e), ctr, (uint32_t)A.n_reset_tables)]
                  : A.reset_tables[0];
    const double *w0 = A.weather + (size_t)tbl * (size_t)A.rows * GLG_ND;
    double d[GLG_ND], x[GLG_NX], u[GLG_NU], o3[3];
#pragma unroll
    for (int i = 0; i < 7; ++i) d[i] = w0[i];
    glg_init_state(d, x);
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) {
        u[i] = 0.0;
        A.u[(size_t)i * B + e] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) A.x[(size_t)i * B + e] = x[i];
    const double doy = A.start_day[tbl];
    A.timestep[e] = 0;
    A.table[e] = tbl;
    A.time[e] = doy;
    A.time[(size_t)B + e] = 0.0;
    A.step_ctr[e] = ctr + 1u;
    A.ep_return[e] = 0.0;
    A.ep_len[e] = 0;
#pragma unroll
    for (int j = 0; j < GLG_NINFO; ++j) A.ep_info[(size_t)j * B + e] = 0.0;
    A.done[e] = 0;
    A.reward[e] = 0.0;
    double hd[GLG_NOBS_FIXED];
    glg_obs_head(x, u, d, 0, doy, 0.0, hd);
    float *orow = A.obs + (size_t)e * A.obs_dim;
    glg_write_obs_row(A, hd, w0 + GLG_ND, (unsigned long long)(A.env_id_offset + e), ctr + 0x80000000u, orow,
                      A.obs_head + (size_t)e * (A.obs_dim - (A.fc_off >= 0 ? 5 * A.Np : 0)), o3);
    if (A.fc_off >= 0) {
        const int nf = 5 * A.Np;
        for (int j = 0; j < nf; ++j) {
            const int i = j / 5, c = j - 5 * i;
            orow[A.fc_off + j] = (float)w0[(size_t)(1 + i) * GLG_ND + c];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// batched evalF: x_next[b] = RK4^n_sub(x[b]; u[b], d[b], p[b or shared])   (greenlight_model.cpp:96-120)
// Row-major [B][n] inputs (the layout of B stacked evalF argument vectors).
// ---------------------------------------------------------------------------------------------------------
struct GlgLocalView {
    const double *b;
    __device__ __forceinline__ double operator[](int i) const { return b[i]; }
};

template <bool GENERAL, bool PER_ENV_P, int NT>
__global__ void __launch_bounds__(NT) glg_evalf_kernel(const __grid_constant__ GlgUniform U, const double *xin, const double *uin,
                                                       const double *din, const double *pin, double *xout,
                                                       unsigned char *bad_out, int B, double dt, int n_sub, int integrator) {
    glg_exp_tbl_fill();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *s_cols = reinterpret_cast<double *>(smem_raw);  // [2*28 + H_COUNT][NT]
    const int tid = threadIdx.x;
    const int e = blockIdx.x * NT + tid;
    if (e >= B) return;
    double x[GLG_NX], u[GLG_NU], d[GLG_ND];
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) x[i] = xin[(size_t)e * GLG_NX + i];
#pragma unroll
    for (int i = 0; i < GLG_NU; ++i) u[i] = uin[(size_t)e * GLG_NU + i];
#pragma unroll
    for (int i = 0; i < 7; ++i) d[i] = din[(size_t)e * GLG_ND + i];
    GlgCol<NT> Hc{s_cols + (size_t)(2 * GLG_NX) * NT + tid};
    GlgSmemStore<NT> st{s_cols + tid};
    int bad;
    if (PER_ENV_P) {
        const double *pe = pin + (size_t)e * GLG_NP;
        double Kl[K_COUNT], Cl[C_COUNT];
        glg_make_k(GlgLocalView{pe}, Kl);
        glg_make_c(GlgLocalView{pe}, Cl);
        glg_hoist(GlgLocalView{pe}, u, d, Hc);
        bad = glg_rk4_step<GENERAL>(GlgLocalView{Kl}, GlgLocalView{Cl}, Hc, GlgLocalView{pe}, u, d, x, dt, n_sub, st, integrator);
    } else {
        glg_hoist(GlgConstView{U.P}, u, d, Hc);
        bad = glg_rk4_step<GENERAL>(GlgConstView{U.K}, GlgConstView{U.C}, Hc, GlgConstView{U.P}, u, d, x, dt, n_sub, st, integrator);
    }
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) xout[(size_t)e * GLG_NX + i] = x[i];
    if (bad_out) bad_out[e] = (unsigned char)bad;
}

// ---------------------------------------------------------------------------------------------------------
// FMA throughput micro-benchmarks (roofline denominators; MEASURED_PEAKS.json has no FP64/FP32 pipe figure)
// 8 independent accumulators per thread so the pipe, not the dependency chain, is the limit.
// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) glg_fma_peak_kernel(T *out, int iters, T a, T b) {
    T v0 = (T)threadIdx.x, v1 = v0 + (T)1, v2 = v0 + (T)2, v3 = v0 + (T)3, v4 = v0 + (T)4, v5 = v0 + (T)5, v6 = v0 + (T)6,
      v7 = v0 + (T)7;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            v0 = v0 * a + b; v1 = v1 * a + b; v2 = v2 * a + b; v3 = v3 * a + b;
            v4 = v4 * a + b; v5 = v5 * a + b; v6 = v6 * a + b; v7 = v7 * a + b;
        }
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = v0 + v1 + v2 + v3 + v4 + v5 + v6 + v7;
}

// accuracy probe for glg_math.h (tests only; not on the step path)
__global__ void glg_math_kernel(int op, const double *in, double *out, int n) {
    glg_exp_tbl_fill();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = glg_math_eval(op, in[i]);
}
