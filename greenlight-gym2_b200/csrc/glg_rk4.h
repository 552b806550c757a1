// glg_rk4.h -- classical RK4 over one control interval with u, d, p held constant
// (integration contract of greenlight_model.cpp:59-63; fixed-step per BASELINE.json north_star).
//
//   k1=f(x) ; k2=f(x+h/2 k1) ; k3=f(x+h/2 k2) ; k4=f(x+h k3) ; x += h/6 (k1+2k2+2k3+k4)
//
// Storage: the stage state lives in registers (xs); the step state `x` and the weighted stage sum `acc` are
// touched once per stage only, so they are kept behind a STORE policy: on the GPU a shared-memory column per
// thread (bank-conflict free, [i][tid]), on the host a plain array.  The stage loop is deliberately NOT
// unrolled so the kernel holds ONE copy of the ~3k-instruction RHS (I-cache).
#pragma once
#include "glg_model.h"
#include "glg_units.h"

struct GlgLocalStore {  // host / local-memory policy
    double xv[GLG_NX], av[GLG_NX];
    GLG_HD double &x(int i) { return xv[i]; }
    GLG_HD double &acc(int i) { return av[i]; }
};

// Advances xc[28] in place.  Returns 1 if any state became non-finite (mirrors the reference's
// try/except -> terminated, tomato_env.py:119-123), else 0.
template <bool GENERAL, class KV, class CV, class HV, class P, class STORE>
GLG_HD int glg_rk4_step(const KV &K, const CV &C, const HV &H, const P &p, const double *u, const double *d,
                        double *xc, double dt, int n_sub, STORE &st, int integrator = 0) {
    const double h_nom = dt / (double)n_sub;
    double xs[GLG_NX], k[GLG_NX];
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) {
        xs[i] = xc[i];
        st.x(i) = xc[i];
    }
#pragma unroll 1
    for (int s = 0; s < n_sub; ++s) {
        // harvest-stiffness guard (glg_model.h): m equal micro-steps inside this nominal substep, m = 1 normally; the
        // graded integrator (integrator = 1) adds its rules after the first evaluation (k1 does not depend on h)
        int m = glg_micro_steps(C, xs[23], xs[25], h_nom);
        double h = h_nom / (double)m;
#pragma unroll 1
        for (int e = 0; e < 4 * m; ++e) {
            const int stage = e & 3;
            const double lam = glg_rhs<GENERAL>(K, C, H, p, u, d, xs, k);
            if (integrator == 1 && e == 0) {
                int ms = 1 + (int)floor(h_nom * lam * GLG_STIFF_INV_CFL);
                ms = ms > GLG_MAX_MICRO ? GLG_MAX_MICRO : (ms < 1 ? 1 : ms);
                if (ms < glg_graded_m(s)) ms = glg_graded_m(s);
                if (ms > m) {
                    m = ms;
                    h = h_nom / (double)m;
                }
            }
            // stage weights: acc = k1 + 2k2 + 2k3 (+k4 at the end); next stage point x + c*k
            const double w = (stage == 1 || stage == 2) ? 2.0 : 1.0;
            const double c = (stage == 2) ? h : 0.5 * h;
            if (stage == 3) {
#pragma unroll
                for (int i = 0; i < GLG_NX; ++i) {
                    const double xn = st.x(i) + (h / 6.0) * (st.acc(i) + k[i]);
                    st.x(i) = xn;
                    xs[i] = xn;
                }
            } else {
#pragma unroll
                for (int i = 0; i < GLG_NX; ++i) {
                    const double a = (stage == 0) ? k[i] : st.acc(i) + w * k[i];
                    st.acc(i) = a;
                    xs[i] = st.x(i) + c * k[i];
                }
            }
        }
    }
    int bad = 0;
#pragma unroll
    for (int i = 0; i < GLG_NX; ++i) {
        xc[i] = xs[i];
        bad |= !(fabs(xs[i]) <= 1.79769313486231570e308);  // false for NaN and +-inf
    }
    return bad;
}

// Tangent RK4 (glg_tangent.cuh): the same contract as glg_rk4_step -- fixed (integrator = 0) or graded (1) grid, the harvest
// guard, n_sub, dt -- with the state in any scalar type T, typically GlgDual<N> seeded with N tangent directions, and the RHS
// assembled from the flux units (glg_rhs_units).  H is the hoisted per-step column in T (glg_hoist with u in T carries the
// derivative with respect to the controls).  Every step-count decision is taken at the same point as in glg_rk4_step and on
// value parts only, so the tangents are the exact derivative of the discrete map on the grid that was executed.
// Advances xc[28] in place; returns 1 if a value became non-finite.
template <bool GENERAL, class KV, class CV, class HV, class P, class UT, class T>
GLG_HD int glg_rk4_step_tangent(const KV &K, const CV &C, const HV &H, const P &p, const UT *u, T *xc, double dt, int n_sub,
                                int integrator = 0) {
    const double h_nom = dt / (double)n_sub;
    T xs[GLG_NX], k[GLG_NX], x0[GLG_NX], acc[GLG_NX];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < GLG_NX; ++i) {
        xs[i] = xc[i];
        x0[i] = xc[i];
    }
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int s = 0; s < n_sub; ++s) {
        int m = glg_micro_steps(C, glg_value(xs[23]), glg_value(xs[25]), h_nom);
        double h = h_nom / (double)m;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int e = 0; e < 4 * m; ++e) {
            const int stage = e & 3;
            const double lam = glg_rhs_units<GENERAL>(K, C, H, p, u, GlgArrayXT<T>{xs}, k);
            if (integrator == 1 && e == 0) {
                int ms = 1 + (int)floor(h_nom * lam * GLG_STIFF_INV_CFL);
                ms = ms > GLG_MAX_MICRO ? GLG_MAX_MICRO : (ms < 1 ? 1 : ms);
                if (ms < glg_graded_m(s)) ms = glg_graded_m(s);
                if (ms > m) {
                    m = ms;
                    h = h_nom / (double)m;
                }
            }
            const double w = (stage == 1 || stage == 2) ? 2.0 : 1.0;
            const double c = (stage == 2) ? h : 0.5 * h;
            if (stage == 3) {
            #if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < GLG_NX; ++i) {
                    const T xn = x0[i] + (h / 6.0) * (acc[i] + k[i]);
                    x0[i] = xn;
                    xs[i] = xn;
                }
            } else {
            #if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < GLG_NX; ++i) {
                    acc[i] = (stage == 0) ? k[i] : acc[i] + w * k[i];
                    xs[i] = x0[i] + c * k[i];
                }
            }
        }
    }
    int bad = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < GLG_NX; ++i) {
        xc[i] = xs[i];
        bad |= !(fabs(glg_value(xs[i])) <= 1.79769313486231570e308);
    }
    return bad;
}
