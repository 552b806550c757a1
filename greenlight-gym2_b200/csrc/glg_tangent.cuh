// glg_tangent.cuh -- linearisation kernels: exact Jacobians of the right-hand side and of one control interval by forward-mode
// differentiation (GlgDual, glg_math.h) of the flux units (glg_units.h), the hoist (glg_model.h) and the RK4 step (glg_rk4.h).
//
//   RHS Jacobian  (STEP = false): f = RHS(x; u, d, p), df/dx [28][28], df/du [28][6]       -- one evaluation, continuous time
//   step Jacobian (STEP = true) : x_next after one control interval, dx_next/dx, dx_next/du -- glg_rk4_step_tangent
//
// Layout: GLG_TAN_G = 17 consecutive threads per env, thread g of an env carries the GLG_TAN_N = 2 tangent directions 2g and 2g+1
// of the 34 (28 states, then 6 controls).  Every thread recomputes the primal; the threads of one env need nothing from each other,
// so envs are packed densely (no idle lanes) and every step-count decision of a thread is taken on its own, identical, value part.
// The stage state, the stage sum and the hoisted column live in the thread's local memory (GlgDual arrays; see DESIGN.md for the
// measured cost and the ptxas report).  Outputs are row-major float64, J[b][i][j] = d out_i / d in_j.
#pragma once
#include "glg_kernels.cuh"

#define GLG_TAN_N 2
#define GLG_TAN_DIRS (GLG_NX + GLG_NU)
#define GLG_TAN_G ((GLG_TAN_DIRS + GLG_TAN_N - 1) / GLG_TAN_N)
#define GLG_TAN_NT 128

struct GlgTanArgs {
    const double *x, *u;  // element (env e, index i) at x[e * xe + i * xi]: row-major [B][n] or the handle's SoA [n][B]
    long long xe, xi, ue, ui;
    const double *d;                  // row-major [B][10]; NULL: the weather row the handle's step reads
    const double *weather;            // [n_tables][rows][10]
    const int *timestep, *table;
    int rows, Np;
    const double *p;                  // [B][208] (PER_ENV_P)
    double *f, *jx, *ju;              // [B][28] value (f or x_next), [B][28][28], [B][28][6]; f and ju may be NULL
    unsigned char *bad;               // [B] or NULL (STEP)
    int B, n_sub, integrator;
    double dt;
};

template <bool GENERAL, bool PER_ENV_P, bool STEP>
__global__ void __launch_bounds__(GLG_TAN_NT) glg_tangent_kernel(const __grid_constant__ GlgUniform U, const __grid_constant__ GlgTanArgs A) {
    glg_exp_tbl_fill();
    typedef GlgDual<GLG_TAN_N> T;
    const long long t = (long long)blockIdx.x * GLG_TAN_NT + threadIdx.x;
    const int e = (int)(t / GLG_TAN_G), g = (int)(t % GLG_TAN_G);
    if (e >= A.B) return;
    const double *drow = A.d ? A.d + (size_t)e * GLG_ND
                             : A.weather + ((size_t)A.table[e] * A.rows + (size_t)min(A.timestep[e], A.rows - A.Np - 1)) * GLG_ND;
    double d[GLG_ND];
#pragma unroll
    for (int i = 0; i < 7; ++i) d[i] = drow[i];
    T x[GLG_NX], u[GLG_NU], H[H_COUNT];
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) {
        x[i] = T(A.x[e * A.xe + i * A.xi]);
#pragma unroll
        for (int k = 0; k < GLG_TAN_N; ++k) x[i].t[k] = (g * GLG_TAN_N + k == i) ? 1.0 : 0.0;
    }
#pragma unroll
    for (int j = 0; j < GLG_NU; ++j) {
        u[j] = T(A.u[e * A.ue + j * A.ui]);
#pragma unroll
        for (int k = 0; k < GLG_TAN_N; ++k) u[j].t[k] = (g * GLG_TAN_N + k == GLG_NX + j) ? 1.0 : 0.0;
    }
    int bad = 0;
    T S[GLG_NX];
    if (PER_ENV_P) {
        const double *pe = A.p + (size_t)e * GLG_NP;
        double Kl[K_COUNT], Cl[C_COUNT];
        glg_make_k(GlgLocalView{pe}, Kl);
        glg_make_c(GlgLocalView{pe}, Cl);
        glg_hoist(GlgLocalView{pe}, u, d, H);
        if (STEP) bad = glg_rk4_step_tangent<GENERAL>(GlgLocalView{Kl}, GlgLocalView{Cl}, H, GlgLocalView{pe}, u, x, A.dt, A.n_sub, A.integrator);
        else glg_rhs_units<GENERAL>(GlgLocalView{Kl}, GlgLocalView{Cl}, H, GlgLocalView{pe}, u, GlgArrayXT<T>{x}, S);
    } else {
        glg_hoist(GlgConstView{U.P}, u, d, H);
        if (STEP) bad = glg_rk4_step_tangent<GENERAL>(GlgConstView{U.K}, GlgConstView{U.C}, H, GlgConstView{U.P}, u, x, A.dt, A.n_sub, A.integrator);
        else glg_rhs_units<GENERAL>(GlgConstView{U.K}, GlgConstView{U.C}, H, GlgConstView{U.P}, u, GlgArrayXT<T>{x}, S);
    }
    const T *out = STEP ? x : S;
#pragma unroll
    for (int k = 0; k < GLG_TAN_N; ++k) {
        const int j = g * GLG_TAN_N + k;
        if (j < GLG_NX) {
#pragma unroll
            for (int i = 0; i < GLG_NX; ++i) A.jx[((size_t)e * GLG_NX + i) * GLG_NX + j] = out[i].t[k];
        } else if (j < GLG_TAN_DIRS && A.ju) {
#pragma unroll
            for (int i = 0; i < GLG_NX; ++i) A.ju[((size_t)e * GLG_NX + i) * GLG_NU + (j - GLG_NX)] = out[i].t[k];
        }
    }
    if (g == 0) {
        if (A.f)
#pragma unroll
            for (int i = 0; i < GLG_NX; ++i) A.f[(size_t)e * GLG_NX + i] = out[i].v;
        if (STEP && A.bad) A.bad[e] = (unsigned char)bad;
    }
}

template <bool GENERAL, bool PER_ENV_P, bool STEP>
static cudaError_t glg_launch_tangent(const GlgUniform &uni, const GlgTanArgs &a, cudaStream_t s) {
    const long long threads = (long long)a.B * GLG_TAN_G;
    glg_tangent_kernel<GENERAL, PER_ENV_P, STEP><<<(unsigned)((threads + GLG_TAN_NT - 1) / GLG_TAN_NT), GLG_TAN_NT, 0, s>>>(uni, a);
    return cudaGetLastError();
}
// variant selection as glg_evalf_batch_ex: shared p -> GENERAL from the table's structure, per-env p -> GENERAL
template <bool STEP>
static cudaError_t glg_launch_tangent_any(const GlgUniform &uni, bool general, bool per_env_p, const GlgTanArgs &a, cudaStream_t s) {
    if (per_env_p) return glg_launch_tangent<true, true, STEP>(uni, a, s);
    return general ? glg_launch_tangent<true, false, STEP>(uni, a, s) : glg_launch_tangent<false, false, STEP>(uni, a, s);
}
