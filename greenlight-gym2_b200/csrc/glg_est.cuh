// glg_est.cuh -- state estimation (glg_est_* in include/glgym.h): an unscented Kalman filter over the envs' observations.  The
// 2n + 1 = 57 sigma points of env b are envs c = b S .. b S + 56 of a second, internal handle (the shadow handle) that the unchanged
// step kernels advance by one control interval between the two kernels below.
//
//   glg_est_init_kernel  : glg_est_reset: mean <- x0, P <- diag(p0_std^2), the env's step counter recorded, status 0.
//   glg_est_sigma_kernel : one CTA per env.  The step-counter and auto-reset checks (status 8 / 4), the Cholesky factor of P by the
//                          zero-column rule, the sigma points written into the shadow handle's SoA x, the env's controls into the
//                          controls array [B S][6], and the pre-step timestep, table and clock of the env into its shadow envs.
//   glg_est_ut_kernel    : one CTA per env.  Mean and covariance of the propagated points, measurement points h(chi'), S, C, the
//                          m x m Cholesky solve and the posterior.  All sums run in ascending index order; no atomics.
// Each kernel takes a MODE: the GLG_EST_FILTER instantiations are the filter alone; the GLG_EST_RECORD ones also write one slot of
// a smoother's forward record (glg_smooth.cuh) and are launched only for an estimator with a smoother; the GLG_EST_LOG ones also
// write one slot of an EM object's data log (glg_em.cuh): the controls and table the step used, the measurement as given, the
// update flags and the slot's log-likelihood term.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "glg_kernels.cuh"

constexpr int GLG_EST_S = 2 * GLG_NX + 1;  // sigma points per env
constexpr int GLG_EST_NM = 7;              // entries of h(x): glg_obs_state7
constexpr int GLG_EST_NT = 128;            // threads of the sigma and UT CTAs
constexpr int GLG_EST_NX2 = GLG_NX * GLG_NX;

// status bits (per env, rewritten by every glg_est_update)
constexpr unsigned char GLG_EST_NONFINITE = 1, GLG_EST_S_NOT_PD = 2, GLG_EST_REINIT = 4, GLG_EST_OUT_OF_STEP = 8;
// log flags (per env and slot): y_dev was given; the update was applied (y_dev given and status 0)
constexpr unsigned char GLG_EST_LOG_Y = 1, GLG_EST_LOG_APPLIED = 2;
// kernel modes: the filter alone; also the smoother's record; also the record and the EM object's log
constexpr int GLG_EST_FILTER = 0, GLG_EST_RECORD = 1, GLG_EST_LOG = 2;

struct GlgEstArgs {
    int B, N, auto_reset, m;   // m measured entries, midx[0..m) their index in h(x)
    int midx[GLG_EST_NM];
    double gamma, wm0, wc0, wi, dt;
    double p0var[GLG_NX], qvar[GLG_NX], rvar[GLG_EST_NM];
    // env handle, read only, SoA [field][B]
    const double *x, *u, *time;
    const int *timestep, *table;
    const unsigned int *step_ctr;
    const unsigned char *done;
    // shadow handle, SoA [field][B S]; sctrl [B S][6]
    double *sx, *sctrl, *stime;
    int *stimestep, *stable;
    const unsigned char *sdone;
    // estimator
    const double *x0;    // glg_est_reset's source, SoA [28][B]
    const double *y;     // [B][7] or NULL (predict only)
    double *mean;        // [28][B]
    double *cov;         // [B][28][28]
    double *innov;       // [B][7]
    unsigned int *ctr;   // [B] the env's step counter at the last reset / update
    unsigned char *status;
    // RECORD kernels only: the sigma kernel's factor, and the slot of the smoother's record this reset / update writes.  Kept
    // last, so the fields above sit at the same parameter offsets in every instantiation.
    double *lfac;                          // [B][28][28] L of the last sigma kernel, zero above the diagonal
    double *r_mean, *r_xbar;               // [28][B] filtered mean, xbar
    double *r_cov, *r_pm, *r_d;            // [B][28][28] filtered P, P-, D
    unsigned char *r_status;               // [B]
    int *r_timestep;                       // [B]
    // LOG kernels only: the slot of the EM object's log this reset / update writes
    double *l_u;                           // [6][B] the controls the env applied
    int *l_table;                          // [B] its weather table
    double *l_y;                           // [7][B] y as given; 0 where not measured or y is NULL
    unsigned char *l_flags;                // [B] GLG_EST_LOG_Y | GLG_EST_LOG_APPLIED
    double *l_ll;                          // [B] -(v^T S^-1 v + log det S + m log 2 pi) / 2; 0 where no update was applied
};

// The log's measurement and flags for a slot without an applied update; the UT kernel overwrites flags and ll where it applies one
__device__ __forceinline__ void glg_est_log_start(const GlgEstArgs &A, int b) {
    const int B = A.B;
    for (int r = threadIdx.x; r < GLG_EST_NM; r += blockDim.x) {
        bool meas = false;
        for (int q = 0; q < A.m; ++q) meas |= A.midx[q] == r;
        A.l_y[(size_t)r * B + b] = A.y && meas ? A.y[(size_t)b * GLG_EST_NM + r] : 0.0;
    }
    if (threadIdx.x == 0) {
        A.l_flags[b] = A.y ? GLG_EST_LOG_Y : 0;
        A.l_ll[b] = 0.0;
    }
}

// A slot without a one-interval prediction behind it (a reset, status 1, 4 or 8): the filtered mean and covariance as they stand
// after this kernel, xbar = P- = D = 0, and the status and timestep.  Each thread copies entries it alone wrote, if any.
__device__ __forceinline__ void glg_est_record_start(const GlgEstArgs &A, int b, unsigned char status) {
    const int B = A.B;
    const size_t pb = (size_t)b * GLG_EST_NX2;
    for (int o = threadIdx.x; o < GLG_EST_NX2; o += blockDim.x) {
        A.r_cov[pb + o] = A.cov[pb + o];
        A.r_pm[pb + o] = 0.0;
        A.r_d[pb + o] = 0.0;
    }
    for (int i = threadIdx.x; i < GLG_NX; i += blockDim.x) {
        A.r_mean[(size_t)i * B + b] = A.mean[(size_t)i * B + b];
        A.r_xbar[(size_t)i * B + b] = 0.0;
    }
    if (threadIdx.x == 0) {
        A.r_status[b] = status;
        A.r_timestep[b] = A.timestep[b];
    }
}

// A slot whose estimate is the prediction (predict only, or status 2): mean xbar and covariance P-, and the status and timestep
__device__ __forceinline__ void glg_est_record_posterior(const GlgEstArgs &A, int b, const double *xbar,
                                                        const double (*Pm)[GLG_NX + 1]) {
    if (threadIdx.x < GLG_NX) A.r_mean[(size_t)threadIdx.x * A.B + b] = xbar[threadIdx.x];
    for (int o = threadIdx.x; o < GLG_EST_NX2; o += blockDim.x) A.r_cov[(size_t)b * GLG_EST_NX2 + o] = Pm[o / GLG_NX][o % GLG_NX];
    if (threadIdx.x == 0) {
        A.r_status[b] = A.status[b];
        A.r_timestep[b] = A.timestep[b];
    }
}

// mean <- src, P <- diag(p0var), innovation 0, for env b; the block's threads share the 784 entries of P
__device__ __forceinline__ void glg_est_restart(const GlgEstArgs &A, int b, const double *src) {
    const int B = A.B;
    double *P = A.cov + (size_t)b * GLG_EST_NX2;
    for (int o = threadIdx.x; o < GLG_EST_NX2; o += blockDim.x) {
        const int i = o / GLG_NX, j = o - i * GLG_NX;
        P[o] = i == j ? A.p0var[i] : 0.0;
    }
    for (int i = threadIdx.x; i < GLG_NX; i += blockDim.x) A.mean[(size_t)i * B + b] = src[(size_t)i * B + b];
    for (int r = threadIdx.x; r < GLG_EST_NM; r += blockDim.x) A.innov[(size_t)b * GLG_EST_NM + r] = 0.0;
}

template <int MODE>
__global__ void __launch_bounds__(GLG_EST_NT) glg_est_init_kernel(const __grid_constant__ GlgEstArgs A) {
    const int b = blockIdx.x;
    glg_est_restart(A, b, A.x0);
    if (threadIdx.x == 0) {
        A.ctr[b] = A.step_ctr[b];
        A.status[b] = 0;
    }
    if constexpr (MODE >= GLG_EST_RECORD) glg_est_record_start(A, b, 0);
    if constexpr (MODE == GLG_EST_LOG) {  // the reset slot: no controls, no measurement
        glg_est_log_start(A, b);
        if (threadIdx.x < GLG_NU) A.l_u[(size_t)threadIdx.x * A.B + b] = 0.0;
        if (threadIdx.x == 0) A.l_table[b] = A.table[b];
    }
}

template <int MODE>
__global__ void __launch_bounds__(GLG_EST_NT) glg_est_sigma_kernel(const __grid_constant__ GlgEstArgs A) {
    __shared__ double L[GLG_NX][GLG_NX + 1];  // P's lower triangle, factored in place
    __shared__ double xh[GLG_NX];
    __shared__ int s_status;
    const int b = blockIdx.x, t = threadIdx.x, B = A.B;
    const size_t BS = (size_t)B * GLG_EST_S, c0 = (size_t)b * GLG_EST_S;
    if (t == 0) {
        const unsigned int ctr = A.step_ctr[b];
        const int st = ctr != A.ctr[b] + 1u ? GLG_EST_OUT_OF_STEP : (A.auto_reset && A.done[b]) ? GLG_EST_REINIT : 0;
        A.ctr[b] = ctr;
        A.status[b] = (unsigned char)st;
        s_status = st;
    }
    __syncthreads();
    const int st = s_status;
    if (st == GLG_EST_REINIT) glg_est_restart(A, b, A.x);  // the env restarted from init_state(d0) of its new weather table
    if (t < GLG_NX) xh[t] = st == GLG_EST_REINIT ? A.x[(size_t)t * B + b] : A.mean[(size_t)t * B + b];
    if (st == 0) {
        // P = L L^T column by column; column j is zero where d <= 1e-12 P[j][j] (x27, the day counter, has variance exactly 0)
        const double *P = A.cov + (size_t)b * GLG_EST_NX2;
        for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) {
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            if (j <= i) L[i][j] = P[o];
        }
        __syncthreads();
        for (int j = 0; j < GLG_NX; ++j) {
            if (t == j) {
                double s = 0.0;
                for (int k = 0; k < j; ++k) s += L[j][k] * L[j][k];
                const double pjj = L[j][j], d = pjj - s;
                L[j][j] = d <= 1e-12 * pjj ? 0.0 : sqrt(d);
            }
            __syncthreads();
            if (t > j && t < GLG_NX) {
                const double ljj = L[j][j];
                double s = 0.0;
                for (int k = 0; k < j; ++k) s += L[t][k] * L[j][k];
                L[t][j] = ljj == 0.0 ? 0.0 : (L[t][j] - s) / ljj;
            }
            __syncthreads();
        }
    } else {
        for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) L[o / GLG_NX][o % GLG_NX] = 0.0;  // every point at the estimate
        __syncthreads();
    }
    // chi_0 = x, chi_i = x + gamma L[:, i-1], chi_{n+i} = x - gamma L[:, i-1]; explicit rounding, so a host restatement is bit-equal
    if (t < GLG_EST_S) {
        const int col = t == 0 ? 0 : (t - 1) % GLG_NX;
        const double g = t == 0 ? 0.0 : (t <= GLG_NX ? A.gamma : -A.gamma);
#pragma unroll 4
        for (int i = 0; i < GLG_NX; ++i) {
            const double l = i >= col ? L[i][col] : 0.0;
            A.sx[i * BS + c0 + t] = __dadd_rn(xh[i], __dmul_rn(g, l));
        }
        const int k = max(A.timestep[b] - 1, 0);  // the interval the env just took
        A.stimestep[c0 + t] = k;
        A.stable[c0 + t] = A.table[b];
        // the pre-step clock; it feeds only the shadow envs' observation rows, which nothing reads
        A.stime[c0 + t] = A.time[b] - fmod(A.dt / 86400.0, 365.0);
        A.stime[BS + c0 + t] = fmod(A.time[(size_t)B + b] - fmod(A.dt / 3600.0, 24.0) + 24.0, 24.0);
    }
    for (int o = t; o < GLG_EST_S * GLG_NU; o += GLG_EST_NT) A.sctrl[c0 * GLG_NU + o] = A.u[(size_t)(o % GLG_NU) * B + b];
    if constexpr (MODE == GLG_EST_LOG) {
        if (t < GLG_NU) A.l_u[(size_t)t * B + b] = A.u[(size_t)t * B + b];
        if (t == 0) A.l_table[b] = A.table[b];
    }
    if constexpr (MODE >= GLG_EST_RECORD) {  // L for the UT kernel's D; both branches above end in a barrier
        for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) {
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            A.lfac[(size_t)b * GLG_EST_NX2 + o] = j <= i ? L[i][j] : 0.0;
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(GLG_EST_NT) glg_est_ut_kernel(const __grid_constant__ GlgEstArgs A) {
    constexpr bool RECORD = MODE >= GLG_EST_RECORD;
    __shared__ double X[GLG_EST_S][GLG_NX + 1];      // propagated points, then their deviations from the mean
    __shared__ double Y[GLG_EST_S][GLG_EST_NM + 1];  // measurement points, then their deviations
    __shared__ double Pm[GLG_NX][GLG_NX + 1];        // prior covariance P-
    __shared__ double Cm[GLG_NX][GLG_EST_NM + 1];    // cross covariance C, then K S
    __shared__ double Km[GLG_NX][GLG_EST_NM + 1];    // gain K
    __shared__ double Sm[GLG_EST_NM][GLG_EST_NM + 1], Ls[GLG_EST_NM][GLG_EST_NM + 1];
    __shared__ double xbar[GLG_NX], ybar[GLG_EST_NM], v[GLG_EST_NM];
    __shared__ int s_pd;
    const int b = blockIdx.x, t = threadIdx.x, B = A.B, m = A.m;
    const size_t BS = (size_t)B * GLG_EST_S, c0 = (size_t)b * GLG_EST_S;
    if constexpr (MODE == GLG_EST_LOG) glg_est_log_start(A, b);
    if (A.status[b] & (GLG_EST_REINIT | GLG_EST_OUT_OF_STEP)) {  // uniform over the CTA
        if constexpr (RECORD) glg_est_record_start(A, b, A.status[b]);
        return;
    }
    double *innov = A.innov + (size_t)b * GLG_EST_NM;
    // a sigma point's step failed: the shadow env ended before the season did
    const int bad = __syncthreads_or(t < GLG_EST_S && A.sdone[c0 + t] && A.timestep[b] - 1 < A.N);
    if (bad) {
        if (t == 0) A.status[b] |= GLG_EST_NONFINITE;
        if (t < GLG_EST_NM) innov[t] = 0.0;
        if constexpr (RECORD) glg_est_record_start(A, b, A.status[b] | GLG_EST_NONFINITE);
        return;
    }
    for (int o = t; o < GLG_EST_S * GLG_NX; o += GLG_EST_NT) {
        const int i = o / GLG_EST_S, s = o - i * GLG_EST_S;
        X[s][i] = A.sx[i * BS + c0 + s];
    }
    __syncthreads();
    if (t < GLG_EST_S) {
        double h[GLG_EST_NM];
        glg_obs_state7(&X[t][0], h);
        for (int r = 0; r < m; ++r) {
            double yr = 0.0;
#pragma unroll
            for (int q = 0; q < GLG_EST_NM; ++q) yr = q == A.midx[r] ? h[q] : yr;  // a select keeps h in registers
            Y[t][r] = yr;
        }
    }
    __syncthreads();
    if (t < GLG_NX) {
        double s = A.wm0 * X[0][t];
        for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * X[k][t];
        xbar[t] = s;
        if constexpr (RECORD) A.r_xbar[(size_t)t * B + b] = s;
    } else if (t >= 32 && t < 32 + m) {
        const int r = t - 32;
        double s = A.wm0 * Y[0][r];
        for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * Y[k][r];
        ybar[r] = s;
    }
    __syncthreads();
    for (int o = t; o < GLG_EST_S * GLG_NX; o += GLG_EST_NT) {
        const int s = o / GLG_NX, i = o - s * GLG_NX;
        X[s][i] -= xbar[i];
    }
    for (int o = t; o < GLG_EST_S * m; o += GLG_EST_NT) {
        const int s = o / m, r = o - s * m;
        Y[s][r] -= ybar[r];
    }
    __syncthreads();
    // P- (lower triangle, mirrored), S (lower, mirrored) and C; weight times a product, so each covariance is exactly symmetric
    for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) {
        const int i = o / GLG_NX, j = o - i * GLG_NX;
        if (j > i) continue;
        double s = A.wc0 * (X[0][i] * X[0][j]);
        for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * (X[k][i] * X[k][j]);
        if (i == j) s += A.qvar[i];
        Pm[i][j] = s;
        Pm[j][i] = s;
        if constexpr (RECORD) {
            A.r_pm[(size_t)b * GLG_EST_NX2 + o] = s;
            A.r_pm[(size_t)b * GLG_EST_NX2 + j * GLG_NX + i] = s;
        }
    }
    if constexpr (RECORD) {
        // D = sum_{i >= 1} Wc_i (chi_i - x^)(chi'_i - xbar)^T with chi_i - x^ = +-gamma L[:, i-1], the product the sigma kernel
        // added (the i = 0 term is zero); written to the slot as formed
        const double *Lb = A.lfac + (size_t)b * GLG_EST_NX2;
        for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) {
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            double s = 0.0;
            for (int k = 1; k < GLG_EST_S; ++k) {
                const double off = __dmul_rn(k <= GLG_NX ? A.gamma : -A.gamma, Lb[i * GLG_NX + (k - 1) % GLG_NX]);
                s += A.wi * (off * X[k][j]);
            }
            A.r_d[(size_t)b * GLG_EST_NX2 + o] = s;
        }
    }
    for (int o = t; o < m * m + GLG_NX * m; o += GLG_EST_NT) {
        if (o < m * m) {
            const int r = o / m, q = o - r * m;
            if (q > r) continue;
            double s = A.wc0 * (Y[0][r] * Y[0][q]);
            for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * (Y[k][r] * Y[k][q]);
            if (r == q) s += A.rvar[A.midx[r]];
            Sm[r][q] = s;
            Sm[q][r] = s;
        } else {
            const int i = (o - m * m) / m, r = (o - m * m) - i * m;
            double s = A.wc0 * (X[0][i] * Y[0][r]);
            for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * (X[k][i] * Y[k][r]);
            Cm[i][r] = s;
        }
    }
    __syncthreads();
    double *P = A.cov + (size_t)b * GLG_EST_NX2;
    if (!A.y) {  // predict only
        if (t < GLG_NX) A.mean[(size_t)t * B + b] = xbar[t];
        if (t < GLG_EST_NM) innov[t] = 0.0;
        for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) P[o] = Pm[o / GLG_NX][o % GLG_NX];
        if constexpr (RECORD) glg_est_record_posterior(A, b, xbar, Pm);
        return;
    }
    if (t == 0) {  // S = Ls Ls^T (plain Cholesky: d <= 0 or non-finite means S is not positive definite); innovation y - ybar
        int pd = 1;
        for (int j = 0; j < m; ++j) {
            double s = 0.0;
            for (int k = 0; k < j; ++k) s += Ls[j][k] * Ls[j][k];
            const double d = Sm[j][j] - s;
            if (!(d > 0.0) || !isfinite(d)) pd = 0;
            Ls[j][j] = sqrt(d);
            for (int i = j + 1; i < m; ++i) {
                double s2 = 0.0;
                for (int k = 0; k < j; ++k) s2 += Ls[i][k] * Ls[j][k];
                Ls[i][j] = (Sm[i][j] - s2) / Ls[j][j];
            }
        }
        for (int r = 0; r < GLG_EST_NM; ++r) innov[r] = 0.0;
        for (int r = 0; r < m; ++r) {
            v[r] = A.y[(size_t)b * GLG_EST_NM + A.midx[r]] - ybar[r];
            innov[A.midx[r]] = v[r];
        }
        s_pd = pd;
        if (!pd) A.status[b] |= GLG_EST_S_NOT_PD;
        if constexpr (MODE == GLG_EST_LOG) {
            if (pd) {  // l = -(|z|^2 + 2 sum log Ls_rr + m log 2 pi) / 2 with Ls z = v
                double z[GLG_EST_NM], q = 0.0, ld = 0.0;
                for (int r = 0; r < m; ++r) {
                    double s = v[r];
                    for (int k = 0; k < r; ++k) s -= Ls[r][k] * z[k];
                    z[r] = s / Ls[r][r];
                    q += z[r] * z[r];
                    ld += log(Ls[r][r]);
                }
                A.l_flags[b] = GLG_EST_LOG_Y | GLG_EST_LOG_APPLIED;
                A.l_ll[b] = -0.5 * (q + 2.0 * ld + m * 1.8378770664093454836);  // log 2 pi
            }
        }
    }
    __syncthreads();
    if (!s_pd) {  // keep the prediction
        if (t < GLG_NX) A.mean[(size_t)t * B + b] = xbar[t];
        for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) P[o] = Pm[o / GLG_NX][o % GLG_NX];
        if constexpr (RECORD) glg_est_record_posterior(A, b, xbar, Pm);
        return;
    }
    if (t < GLG_NX) {
        // row t of K = C S^-1: solve S k = C[t] by forward and back substitution, then x = xbar + K v and row t of K S
        double *z = &Km[t][0];
        for (int r = 0; r < m; ++r) {
            double s = Cm[t][r];
            for (int k = 0; k < r; ++k) s -= Ls[r][k] * z[k];
            z[r] = s / Ls[r][r];
        }
        for (int r = m - 1; r >= 0; --r) {
            double s = z[r];
            for (int k = r + 1; k < m; ++k) s -= Ls[k][r] * z[k];
            z[r] = s / Ls[r][r];
        }
        double xn = xbar[t];
        for (int r = 0; r < m; ++r) xn += z[r] * v[r];
        A.mean[(size_t)t * B + b] = xn;
        if constexpr (RECORD) A.r_mean[(size_t)t * B + b] = xn;
        for (int a = 0; a < m; ++a) {
            double s = 0.0;
            for (int q = 0; q < m; ++q) s += Sm[a][q] * z[q];
            Cm[t][a] = s;  // (K S)[t][a]; row t of C is no longer needed
        }
    }
    __syncthreads();
    // P = sym(P- - K S K^T)
    for (int o = t; o < GLG_EST_NX2; o += GLG_EST_NT) {
        const int i = o / GLG_NX, j = o - i * GLG_NX;
        double kij = 0.0, kji = 0.0;
        for (int a = 0; a < m; ++a) {
            kij += Km[i][a] * Cm[j][a];
            kji += Km[j][a] * Cm[i][a];
        }
        const double p = 0.5 * ((Pm[i][j] - kij) + (Pm[j][i] - kji));
        P[o] = p;
        if constexpr (RECORD) A.r_cov[(size_t)b * GLG_EST_NX2 + o] = p;
    }
    if constexpr (RECORD) {
        if (t == 0) {
            A.r_status[b] = A.status[b];
            A.r_timestep[b] = A.timestep[b];
        }
    }
}

