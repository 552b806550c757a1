// Test-only host build of the forward-mode linearisation (GlgDual, glg_rhs_units, glg_rk4_step_tangent); never part of the
// product library.  Lets `pytest -m "not gpu"` check the exact Jacobians against the oracle without a GPU.  Built by
// tests/test_gpu_linearize.py with the flags tests/conftest.py uses for hostmath.cpp (-O2 -ffp-contract=off).
#include "../../greenlight-gym2_b200/csrc/glg_model.h"
#include "../../greenlight-gym2_b200/csrc/glg_rk4.h"
#include "../../greenlight-gym2_b200/csrc/glg_units.h"

// all 34 directions (28 states, then 6 controls) in one GlgDual<34>
typedef GlgDual<GLG_NX + GLG_NU> TgDual;
static void tg_seed(const double *x, const double *u, TgDual *xd, TgDual *ud) {
    for (int i = 0; i < GLG_NX; ++i) {
        xd[i] = TgDual(x[i]);
        xd[i].t[i] = 1.0;
    }
    for (int j = 0; j < GLG_NU; ++j) {
        ud[j] = TgDual(u[j]);
        ud[j].t[GLG_NX + j] = 1.0;
    }
}
static void tg_unseed(const TgDual *y, double *f, double *jx, double *ju) {
    for (int i = 0; i < GLG_NX; ++i) {
        if (f) f[i] = y[i].v;
        for (int j = 0; j < GLG_NX; ++j) jx[i * GLG_NX + j] = y[i].t[j];
        if (ju)
            for (int j = 0; j < GLG_NU; ++j) ju[i * GLG_NU + j] = y[i].t[GLG_NX + j];
    }
}

extern "C" {
// f = RHS(x; u, d, p) assembled from the units in the 13-warp order (hostmath's hm_rhs_units with ng = 13), df/dx [28][28],
// df/du [28][6]; returns the transient-stiffness estimate
double tg_rhs_jac(const double *x, const double *u, const double *d, const double *p, int general, double *f, double *jx, double *ju) {
    double K[K_COUNT], C[C_COUNT];
    glg_make_k(p, K);
    glg_make_c(p, C);
    TgDual xd[GLG_NX], ud[GLG_NU], H[H_COUNT], S[GLG_NX];
    tg_seed(x, u, xd, ud);
    glg_hoist(p, ud, d, H);
    const double lam = general ? glg_rhs_units<true>(K, C, H, p, ud, GlgArrayXT<TgDual>{xd}, S)
                               : glg_rhs_units<false>(K, C, H, p, ud, GlgArrayXT<TgDual>{xd}, S);
    tg_unseed(S, f, jx, ju);
    return lam;
}
// x_next after one control interval and its Jacobians dx_next/dx [28][28], dx_next/du [28][6]; returns the non-finite flag
int tg_evalf_jac(const double *x, const double *u, const double *d, const double *p, double dt, int n_sub, int integrator, int general,
                 double *x_next, double *jx, double *ju) {
    double K[K_COUNT], C[C_COUNT];
    glg_make_k(p, K);
    glg_make_c(p, C);
    TgDual xd[GLG_NX], ud[GLG_NU], H[H_COUNT];
    tg_seed(x, u, xd, ud);
    glg_hoist(p, ud, d, H);
    const int bad = general ? glg_rk4_step_tangent<true>(K, C, H, p, ud, xd, dt, n_sub, integrator)
                            : glg_rk4_step_tangent<false>(K, C, H, p, ud, xd, dt, n_sub, integrator);
    tg_unseed(xd, x_next, jx, ju);
    return bad;
}
}
