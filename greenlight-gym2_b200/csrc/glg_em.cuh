// glg_em.cuh -- noise identification (glg_em_* in include/glgym.h): the E-step of an EM fit of the estimator's diagonal Q and R over
// a smoother's window.  Every (env, slot) pair of the window is independent, so the 57 sigma points of all pairs go to the unchanged
// step kernels of an internal handle (the EM handle) in a few wide launches instead of one launch per slot.  Pair p = b len + k
// (env b, slot k oldest first); the pairs are split into balanced chunks of at most max_points / 57 pairs, and a chunk of np pairs
// is stepped as a batch of np 57 envs of the EM handle, envs c 57 .. c 57 + 56 holding the points of the chunk's pair c.
//
//   glg_em_sigma_kernel  : one CTA per pair of the chunk.  For a linked slot k, the points of (ms_{k-1}, Ps_{k-1}) by the
//                          estimator's factor rule and rounding, with slot k's logged controls and table and pre-step timestep
//                          timestep_k - 1.  A slot without a transition gets 57 points at its smoothed mean ms_k, so the step
//                          only ever sees states the smoother produced.
//   glg_em_expect_kernel : one CTA per pair of the chunk.  The Q term from the stepped points, and the R term from the points of
//                          (ms_k, Ps_k) through glg_obs_state7.  All sums run in ascending index order.
//   glg_em_env_kernel    : one thread per (env, entry): the env's sums over its slots in ascending slot order.
//   glg_em_total_kernel  : one thread per entry: the pooled sums over the envs in ascending env order.  No atomics anywhere.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "glg_smooth.cuh"

constexpr int GLG_EM_NE = GLG_NX + GLG_EST_NM;  // per pair: E (28 Q entries), then the 7 R entries
constexpr int GLG_EM_NS = GLG_EM_NE + 3;        // per env and pooled: the 35 sums, transitions, measured slots, sum of l
constexpr int GLG_EM_NT = 128;
// used flags (per pair): the slot's transition entered the Q sums; its measurement entered the R sums
constexpr unsigned char GLG_EM_USED_Q = 1, GLG_EM_USED_R = 2;

struct GlgEmArgs {
    int B, W, len, first, N;  // the smoother's ring of W slots, len valid ones from ring slot `first`; the env's season length
    int p0, np;               // this chunk: pairs p0 .. p0 + np - 1, stepped as a batch of np 57 envs
    int m, midx[GLG_EST_NM];  // the estimator's measured entries
    double gamma, wm0, wc0, wi;
    // the smoother's output, oldest first, and its record, ring order
    const double *s_mean;                  // [W][28][B]
    const double *s_cov, *gain;            // [W][B][28][28]
    const unsigned char *status;           // [W][B]
    const int *timestep;                   // [W][B]
    // the log, ring order
    const double *l_u, *l_y, *l_ll;        // [W][6][B], [W][7][B], [W][B]
    const int *l_table;                    // [W][B]
    const unsigned char *l_flags;          // [W][B]
    // the EM handle's first np 57 envs, SoA [field][np 57]; hctrl [np 57][6]
    double *hx, *hctrl, *htime;
    int *htimestep, *htable;
    const unsigned char *hdone;
    // output, oldest first
    double *ex;                            // [W][B][35]
    double *fbar;                          // [W][28][B]
    unsigned char *used;                   // [W][B]
    double *env_stats;                     // [B][38]
    double *total;                         // [38]
};

// the pair's env, slot (oldest first), ring slot, and whether the slot is a transition from the slot before it in the window
struct GlgEmPair {
    int b, k, r;
    bool linked;
};
__device__ __forceinline__ GlgEmPair glg_em_pair(const GlgEmArgs &A, int p) {
    GlgEmPair q;
    q.b = p / A.len;
    q.k = p - q.b * A.len;
    q.r = (A.first + q.k) % A.W;
    q.linked = q.k >= 1 && !(A.status[(size_t)q.r * A.B + q.b] & GLG_SMOOTH_SEGMENT);
    return q;
}

// L <- the factor of the covariance at P by the estimator's zero-column rule (P's lower triangle read); ends in a barrier
__device__ __forceinline__ void glg_em_factor(double (*L)[GLG_NX + 1], const double *P) {
    const int t = threadIdx.x;
    for (int o = t; o < GLG_EST_NX2; o += GLG_EM_NT) {
        const int i = o / GLG_NX, j = o - i * GLG_NX;
        L[i][j] = j <= i ? P[o] : 0.0;
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
}

// point s of (x, L): x, x + gamma L[:, s-1], x - gamma L[:, s-1], rounded as the estimator's sigma kernel rounds
__device__ __forceinline__ double glg_em_point(const double (*L)[GLG_NX + 1], const double *x, double gamma, int s, int i) {
    const int col = s == 0 ? 0 : (s - 1) % GLG_NX;
    const double g = s == 0 ? 0.0 : (s <= GLG_NX ? gamma : -gamma);
    const double l = i >= col ? L[i][col] : 0.0;
    return __dadd_rn(x[i], __dmul_rn(g, l));
}

__global__ void __launch_bounds__(GLG_EM_NT) glg_em_sigma_kernel(const __grid_constant__ GlgEmArgs A) {
    __shared__ double L[GLG_NX][GLG_NX + 1];
    __shared__ double xh[GLG_NX];
    const int c = blockIdx.x, t = threadIdx.x, B = A.B;
    const GlgEmPair q = glg_em_pair(A, A.p0 + c);
    const int src = q.linked ? q.k - 1 : q.k;  // the slot whose smoothed moments are propagated
    if (q.linked) {
        glg_em_factor(L, A.s_cov + ((size_t)src * B + q.b) * GLG_EST_NX2);
    } else {
        for (int o = t; o < GLG_EST_NX2; o += GLG_EM_NT) L[o / GLG_NX][o % GLG_NX] = 0.0;
    }
    if (t < GLG_NX) xh[t] = A.s_mean[((size_t)src * GLG_NX + t) * B + q.b];
    __syncthreads();
    const size_t NH = (size_t)A.np * GLG_EST_S, c0 = (size_t)c * GLG_EST_S;
    const size_t rb = (size_t)q.r * B + q.b;
    if (t < GLG_EST_S) {
#pragma unroll 4
        for (int i = 0; i < GLG_NX; ++i) A.hx[i * NH + c0 + t] = glg_em_point(L, xh, A.gamma, t, i);
        A.htimestep[c0 + t] = max(A.timestep[rb] - 1, 0);
        A.htable[c0 + t] = A.l_table[rb];
        A.htime[c0 + t] = 0.0;  // the clock feeds only the EM envs' observation rows, which nothing reads
        A.htime[NH + c0 + t] = 0.0;
    }
    for (int o = t; o < GLG_EST_S * GLG_NU; o += GLG_EM_NT)
        A.hctrl[c0 * GLG_NU + o] = A.l_u[((size_t)q.r * GLG_NU + o % GLG_NU) * B + q.b];
}

__global__ void __launch_bounds__(GLG_EM_NT) glg_em_expect_kernel(const __grid_constant__ GlgEmArgs A) {
    __shared__ double X[GLG_EST_S][GLG_NX + 1];  // stepped points f_i, then f_i - fbar; later the R term's points
    __shared__ double L[GLG_NX][GLG_NX + 1];     // factor of Ps_{k-1}, then M = Ps_k G_{k-1}^T; later the factor of Ps_k
    __shared__ double Ps[GLG_NX][GLG_NX + 1];    // Ps_k
    __shared__ double G[GLG_NX][GLG_NX + 1];     // G_{k-1}
    __shared__ double Z[GLG_NX][GLG_NX + 1];     // Delta (row j: W gamma (f_{j+} - f_{j-})), then Z = L^-T Delta
    __shared__ double fb[GLG_NX], xs[GLG_NX], hb[GLG_EST_NM];
    const int c = blockIdx.x, t = threadIdx.x, B = A.B;
    const GlgEmPair q = glg_em_pair(A, A.p0 + c);
    const size_t rb = (size_t)q.r * B + q.b, kb = (size_t)q.k * B + q.b;
    const bool meas = A.l_flags[rb] & GLG_EST_LOG_APPLIED;
    double *ex = A.ex + kb * GLG_EM_NE;
    const double *Pk = A.s_cov + kb * GLG_EST_NX2;
    for (int o = t; o < GLG_EST_NX2; o += GLG_EM_NT) Ps[o / GLG_NX][o % GLG_NX] = Pk[o];
    if (t < GLG_NX) xs[t] = A.s_mean[((size_t)q.k * GLG_NX + t) * B + q.b];
    const size_t NH = (size_t)A.np * GLG_EST_S, c0 = (size_t)c * GLG_EST_S;
    // a step failed where the season had not ended: the transition is left out
    const int bad = __syncthreads_or(q.linked && t < GLG_EST_S && A.hdone[c0 + t] && A.timestep[rb] - 1 < A.N);
    const bool useq = q.linked && !bad;
    if (useq) {
        const double *Gk = A.gain + ((size_t)(q.k - 1) * B + q.b) * GLG_EST_NX2;
        for (int o = t; o < GLG_EST_S * GLG_NX; o += GLG_EM_NT) {
            const int i = o / GLG_EST_S, s = o - i * GLG_EST_S;
            X[s][i] = A.hx[i * NH + c0 + s];
        }
        for (int o = t; o < GLG_EST_NX2; o += GLG_EM_NT) G[o / GLG_NX][o % GLG_NX] = Gk[o];
        glg_em_factor(L, A.s_cov + ((size_t)(q.k - 1) * B + q.b) * GLG_EST_NX2);  // ends in a barrier
        if (t < GLG_NX) {  // fbar in the UT kernel's order
            double s = A.wm0 * X[0][t];
            for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * X[k][t];
            fb[t] = s;
            A.fbar[((size_t)q.k * GLG_NX + t) * B + q.b] = s;
        }
        for (int o = t; o < GLG_EST_NX2; o += GLG_EM_NT) {
            const int j = o / GLG_NX, i = o - j * GLG_NX;
            Z[j][i] = A.wi * A.gamma * (X[1 + j][i] - X[1 + GLG_NX + j][i]);
        }
        __syncthreads();
        for (int o = t; o < GLG_EST_S * GLG_NX; o += GLG_EM_NT) {
            const int s = o / GLG_NX, i = o - s * GLG_NX;
            X[s][i] -= fb[i];
        }
        if (t < GLG_NX) {  // column t of Z = L^-T Delta by back substitution; a component whose column of L is zero is 0
            for (int j = GLG_NX - 1; j >= 0; --j) {
                double s = Z[j][t];
                for (int a = j + 1; a < GLG_NX; ++a) s -= L[a][j] * Z[a][t];
                Z[j][t] = L[j][j] == 0.0 ? 0.0 : s / L[j][j];
            }
        }
        __syncthreads();
        for (int o = t; o < GLG_EST_NX2; o += GLG_EM_NT) {  // M = Ps_k G_{k-1}^T into L
            const int a = o / GLG_NX, j = o - a * GLG_NX;
            double s = 0.0;
            for (int l = 0; l < GLG_NX; ++l) s += Ps[a][l] * G[j][l];
            L[a][j] = s;
        }
        __syncthreads();
        if (t < GLG_NX) {  // E = diag[Ps_k + (ms_k - fbar)(ms_k - fbar)^T + Phi - C - C^T], C = M Z
            double phi = A.wc0 * (X[0][t] * X[0][t]);
            for (int k = 1; k < GLG_EST_S; ++k) phi += A.wi * (X[k][t] * X[k][t]);
            double cc = 0.0;
            for (int j = 0; j < GLG_NX; ++j) cc += L[t][j] * Z[j][t];
            const double d = xs[t] - fb[t];
            ex[t] = ((Ps[t][t] + d * d) + phi) - cc - cc;
        }
        __syncthreads();
    } else {
        if (t < GLG_NX) {
            ex[t] = 0.0;
            A.fbar[((size_t)q.k * GLG_NX + t) * B + q.b] = 0.0;
        }
    }
    if (t == 0) A.used[kb] = (useq ? GLG_EM_USED_Q : 0) | (meas ? GLG_EM_USED_R : 0);
    if (!meas) {
        if (t < GLG_EST_NM) ex[GLG_NX + t] = 0.0;
        return;
    }
    // R term: the points of (ms_k, Ps_k) through h; E_r = (y_r - hbar_r)^2 + sum Wc_i (h_ir - hbar_r)^2 for measured r
    glg_em_factor(L, Pk);
    for (int o = t; o < GLG_EST_S * GLG_NX; o += GLG_EM_NT) {
        const int s = o / GLG_NX, i = o - s * GLG_NX;
        X[s][i] = glg_em_point(L, xs, A.gamma, s, i);
    }
    __syncthreads();
    if (t < GLG_EST_S) {
        double h[GLG_EST_NM];
        glg_obs_state7(&X[t][0], h);
        for (int r = 0; r < GLG_EST_NM; ++r) X[t][r] = h[r];  // row t is only this thread's
    }
    __syncthreads();
    if (t < GLG_EST_NM) {
        double s = A.wm0 * X[0][t];
        for (int k = 1; k < GLG_EST_S; ++k) s += A.wi * X[k][t];
        hb[t] = s;
        bool measured = false;
        for (int a = 0; a < A.m; ++a) measured |= A.midx[a] == t;
        double v = A.wc0 * ((X[0][t] - s) * (X[0][t] - s));
        for (int k = 1; k < GLG_EST_S; ++k) v += A.wi * ((X[k][t] - s) * (X[k][t] - s));
        const double e = A.l_y[((size_t)q.r * GLG_EST_NM + t) * B + q.b] - s;
        ex[GLG_NX + t] = measured ? e * e + v : 0.0;
    }
}

// env b's sums over its slots, ascending: the 35 entries, transitions, measured slots and the log-likelihood
__global__ void glg_em_env_kernel(const __grid_constant__ GlgEmArgs A) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= A.B * GLG_EM_NS) return;
    const int b = o / GLG_EM_NS, j = o - b * GLG_EM_NS, B = A.B;
    double s = 0.0;
    for (int k = 0; k < A.len; ++k) {
        const size_t kb = (size_t)k * B + b;
        const int r = (A.first + k) % A.W;
        s += j < GLG_EM_NE                ? A.ex[kb * GLG_EM_NE + j]
             : j == GLG_EM_NE             ? (double)(A.used[kb] & GLG_EM_USED_Q)
             : j == GLG_EM_NE + 1         ? (double)((A.used[kb] & GLG_EM_USED_R) >> 1)
                                          : A.l_ll[(size_t)r * B + b];
    }
    A.env_stats[(size_t)b * GLG_EM_NS + j] = s;
}

__global__ void glg_em_total_kernel(const __grid_constant__ GlgEmArgs A) {
    const int j = threadIdx.x;
    if (j >= GLG_EM_NS) return;
    double s = 0.0;
#pragma unroll 8
    for (int b = 0; b < A.B; ++b) s += A.env_stats[(size_t)b * GLG_EM_NS + j];
    A.total[j] = s;
}
