// glg_smooth.cuh -- state smoothing (glg_smooth_* in include/glgym.h): the unscented Rauch-Tung-Striebel smoother over the forward
// record that the estimator's RECORD kernels (glg_est.cuh) write, one slot per glg_est_reset / glg_est_update, into a ring of W
// slots per env.
//
//   glg_smooth_kernel : one CTA per env walks the env's valid slots from the newest to the oldest.  Per linked slot k: the factor
//                       of P-_{k+1} by the estimator's zero-column rule, G_k = D_{k+1} (P-_{k+1})^-1 by 28 row solves, the smoothed
//                       mean and sym(P_k + G_k (Ps_{k+1} - P-_{k+1}) G_k^T) by two 28 x 28 products.  All sums run in ascending
//                       index order; no atomics.  The record is only read, so the smoother can run again as the window moves.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "glg_est.cuh"

constexpr int GLG_SMOOTH_NT = 128;  // threads of the backward CTA
// status bits that start a segment: the slot is not a one-interval prediction and update of the slot before it
constexpr unsigned char GLG_SMOOTH_SEGMENT = GLG_EST_NONFINITE | GLG_EST_REINIT | GLG_EST_OUT_OF_STEP;

struct GlgSmoothArgs {
    int B, W, len, first;        // ring of W slots per env; len valid ones, the oldest at ring slot `first`
    unsigned int active;         // bit j: state j takes part (p0_std[j] or q_std[j] > 0); the others pass through
    // the forward record, ring order
    const double *mean, *xbar;   // [W][28][B]
    const double *cov, *pm, *d;  // [W][B][28][28]
    const unsigned char *status; // [W][B]
    // output, oldest first
    double *s_mean;              // [W][28][B]
    double *s_cov, *gain;        // [W][B][28][28]
};

__global__ void __launch_bounds__(GLG_SMOOTH_NT) glg_smooth_kernel(const __grid_constant__ GlgSmoothArgs A) {
    __shared__ double L[GLG_NX][GLG_NX + 1];   // P-_{k+1}, factored in place
    __shared__ double G[GLG_NX][GLG_NX + 1];   // D_{k+1}, solved in place into G_k
    __shared__ double M[GLG_NX][GLG_NX + 1];   // Ps_{k+1} - P-_{k+1}, then G M G^T
    __shared__ double T[GLG_NX][GLG_NX + 1];   // G M
    __shared__ double Ps[GLG_NX][GLG_NX + 1];  // the smoothed covariance of the slot after the current one
    __shared__ double xs[GLG_NX], dx[GLG_NX];  // its smoothed mean; xs - xbar_{k+1}
    const int b = blockIdx.x, t = threadIdx.x, B = A.B;
    const size_t BX2 = (size_t)B * GLG_EST_NX2, pb = (size_t)b * GLG_EST_NX2;
    for (int k = A.len - 1; k >= 0; --k) {
        const size_t r = (size_t)((A.first + k) % A.W), r1 = (size_t)((A.first + k + 1) % A.W);
        const double *P = A.cov + r * BX2 + pb, *mk = A.mean + r * GLG_NX * B;
        double *so = A.s_cov + (size_t)k * BX2 + pb, *go = A.gain + (size_t)k * BX2 + pb, *mo = A.s_mean + (size_t)k * GLG_NX * B;
        if (k == A.len - 1 || (A.status[r1 * B + b] & GLG_SMOOTH_SEGMENT)) {  // the last slot of a segment: the filtered estimate
            for (int o = t; o < GLG_EST_NX2; o += GLG_SMOOTH_NT) {
                const double p = P[o];
                Ps[o / GLG_NX][o % GLG_NX] = p;
                so[o] = p;
                go[o] = 0.0;
            }
            if (t < GLG_NX) {
                const double x = mk[(size_t)t * B + b];
                xs[t] = x;
                mo[(size_t)t * B + b] = x;
            }
            __syncthreads();
            continue;
        }
        const double *Pm = A.pm + r1 * BX2 + pb, *D = A.d + r1 * BX2 + pb;
        for (int o = t; o < GLG_EST_NX2; o += GLG_SMOOTH_NT) {
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            const bool ai = A.active >> i & 1u, aj = A.active >> j & 1u;
            const double pm = Pm[o];
            if (j <= i) L[i][j] = ai && aj ? pm : 0.0;  // a deterministic state's row and column are left out
            G[i][j] = ai ? D[o] : 0.0;
            M[i][j] = Ps[i][j] - pm;
        }
        if (t < GLG_NX) dx[t] = xs[t] - A.xbar[r1 * GLG_NX * B + (size_t)t * B + b];
        __syncthreads();
        // the estimator's rule: column j is zero where d <= 1e-12 P-[j][j]
        for (int j = 0; j < GLG_NX; ++j) {
            if (t == j) {
                double s = 0.0;
                for (int q = 0; q < j; ++q) s += L[j][q] * L[j][q];
                const double pjj = L[j][j], d = pjj - s;
                L[j][j] = d <= 1e-12 * pjj ? 0.0 : sqrt(d);
            }
            __syncthreads();
            if (t > j && t < GLG_NX) {
                const double ljj = L[j][j];
                double s = 0.0;
                for (int q = 0; q < j; ++q) s += L[t][q] * L[j][q];
                L[t][j] = ljj == 0.0 ? 0.0 : (L[t][j] - s) / ljj;
            }
            __syncthreads();
        }
        if (t < GLG_NX) {
            // row t of G: P- g = d_t by forward substitution through L and back substitution through L^T, in place; a
            // component whose column of L is zero is 0.  Then the smoothed mean x^_k + G (xs_{k+1} - xbar_{k+1}).
            double *g = &G[t][0];
            for (int c = 0; c < GLG_NX; ++c) {
                double s = g[c];
                for (int q = 0; q < c; ++q) s -= L[c][q] * g[q];
                g[c] = L[c][c] == 0.0 ? 0.0 : s / L[c][c];
            }
            for (int c = GLG_NX - 1; c >= 0; --c) {
                double s = g[c];
                for (int q = c + 1; q < GLG_NX; ++q) s -= L[q][c] * g[q];
                g[c] = L[c][c] == 0.0 ? 0.0 : s / L[c][c];
            }
            double s = 0.0;
            for (int c = 0; c < GLG_NX; ++c) s += g[c] * dx[c];
            const double x = mk[(size_t)t * B + b] + s;
            xs[t] = x;
            mo[(size_t)t * B + b] = x;
        }
        __syncthreads();
        for (int o = t; o < GLG_EST_NX2; o += GLG_SMOOTH_NT) {  // T = G M
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            double s = 0.0;
            for (int a = 0; a < GLG_NX; ++a) s += G[i][a] * M[a][j];
            T[i][j] = s;
            go[o] = G[i][j];
        }
        __syncthreads();
        for (int o = t; o < GLG_EST_NX2; o += GLG_SMOOTH_NT) {  // M = T G^T
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            double s = 0.0;
            for (int a = 0; a < GLG_NX; ++a) s += T[i][a] * G[j][a];
            M[i][j] = s;
        }
        __syncthreads();
        for (int o = t; o < GLG_EST_NX2; o += GLG_SMOOTH_NT) {  // Ps_k = sym(P_k + G (Ps_{k+1} - P-_{k+1}) G^T)
            const int i = o / GLG_NX, j = o - i * GLG_NX;
            const double p = 0.5 * ((P[o] + M[i][j]) + (P[j * GLG_NX + i] + M[j][i]));
            Ps[i][j] = p;
            so[o] = p;
        }
        __syncthreads();
    }
}
