"""Linearisation by forward-mode differentiation (csrc/glg_tangent.cuh, GlgDual in glg_math.h): the RHS Jacobian and the
control-step Jacobian.  CPU tier: the host build of the same templates (tests/hostmath/tangent.cpp) against the unit-assembled RHS bit for bit,
against central differences of the C oracle, and against the committed forward-difference stiffness trace.  GPU tier: the device
kernels against the host build, against glg_evalf_batch_ex and its central differences, and glg_linearize on a handle.

Scaled comparisons use D^-1 J D with D = diag(max(|x|, 1e-3)) on state columns and 1 on control columns, so entries of very
different units compare on one scale."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, rel_err

DP = C.POINTER(C.c_double)
P = lambda a: a.ctypes.data_as(DP)
GRADED = 3  # oracle_binding.INTEGRATOR_GRADED: glgo_evalf_ex's stiff_guard for the graded grid


HEADERS = [os.path.join(ROOT, "greenlight-gym2_b200", "csrc", h) for h in ("glg_model.h", "glg_math.h", "glg_rk4.h", "glg_units.h")]


def _build_tangent():
    """tests/hostmath/tangent.cpp -> libtangent.so, rebuilt when the source or a device header is newer; next to the source, or
    in the temporary directory when the tree is read-only."""
    src = os.path.join(ROOT, "tests", "hostmath", "tangent.cpp")
    so = os.path.join(ROOT, "tests", "hostmath", "libtangent.so")
    if not os.access(os.path.dirname(so), os.W_OK):
        so = os.path.join(tempfile.gettempdir(), f"glg_libtangent_{os.getuid()}.so")
    if not os.path.exists(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in [src] + HEADERS):
        tmp = so + f".{os.getpid()}"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, src], check=True)
        os.replace(tmp, so)
    return so


class _HostLibs:
    """libhostmath.so (tests/conftest.py: hm_rhs_units, hm_nominal_structure) and libtangent.so (the dual builds)."""

    def __init__(self):
        self.base = C.CDLL(os.path.join(ROOT, "tests", "hostmath", "libhostmath.so"))
        self.base.hm_rhs_units.argtypes = [DP, DP, DP, DP, C.c_int, C.c_int, C.c_int, DP]
        self.base.hm_nominal_structure.argtypes = [DP]
        self.hm_rhs_units = self.base.hm_rhs_units
        self.hm_nominal_structure = self.base.hm_nominal_structure
        self.tg = C.CDLL(_build_tangent())
        self.tg.tg_rhs_jac.argtypes = [DP, DP, DP, DP, C.c_int, DP, DP, DP]
        self.tg.tg_rhs_jac.restype = C.c_double
        self.tg.tg_evalf_jac.argtypes = [DP, DP, DP, DP, C.c_double, C.c_int, C.c_int, C.c_int, DP, DP, DP]
        self.tg.tg_evalf_jac.restype = C.c_int
        self.rhs_jac = self.tg.tg_rhs_jac
        self.evalf_jac = self.tg.tg_evalf_jac


@pytest.fixture(scope="module")
def hm():
    return _HostLibs()


@pytest.fixture(scope="module")
def oracle():
    import oracle_binding as ob
    lib = ob.load()
    lib.glgo_evalf_ex.argtypes = [DP, DP, DP, DP, C.c_double, C.c_int, C.c_int, DP, C.POINTER(C.c_long)]
    return lib


def _scale(x):
    return np.concatenate([np.maximum(np.abs(x), 1e-3), np.ones(6)])


def _scaled(J, D):
    """D^-1 J D for J [..., 28, 34] (state and control columns side by side)."""
    return J * D[..., None, :] / D[..., :28, None]


def host_rhs_jac(hm, x, u, d, p, general):
    f, jx, ju = np.zeros(28), np.zeros((28, 28)), np.zeros((28, 6))
    lam = hm.rhs_jac(P(x), P(u), P(d), P(p), general, P(f), P(jx), P(ju))
    return f, jx, ju, lam


def host_step_jac(hm, x, u, d, p, n_sub, integrator, general):
    xn, jx, ju = np.zeros(28), np.zeros((28, 28)), np.zeros((28, 6))
    bad = hm.evalf_jac(P(x), P(u), P(d), P(p), 900.0, n_sub, integrator, general, P(xn), P(jx), P(ju))
    return xn, jx, ju, bad


def _perturbed(x, u, j, h):
    x, u = x.copy(), u.copy()
    if j < 28:
        x[j] += h
    else:
        u[j - 28] += h
    return x, u


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


# ------------------------------------------------------------------------------------------------ CPU tier
def test_host_dual_rhs_value_is_the_unit_rhs_bit_for_bit(hm, rhs_golden):
    """The value part of the dual RHS is exactly hm_rhs_units' 13-warp assembly (hostmath is built with -ffp-contract=off), for
    the nominal and the general variant, and so is the stiffness estimate the graded grid is chosen from."""
    for i in range(len(rhs_golden["x"])):
        x, u, d, p = (_c(rhs_golden[k][i]) for k in "xudp")
        for general in (0, 1):
            f, _, _, lam = host_rhs_jac(hm, x, u, d, p, general)
            s = np.zeros(30)
            hm.hm_rhs_units(P(x), P(u), P(d), P(p), general, 13, 0, P(s))
            assert np.array_equal(f, s[:28]), (i, general)
            assert lam == s[29], (i, general)


# temperature pairs whose difference enters a fractional power |dT + 1e-10|^e (e = 1/3, 1/4, 0.32, 0.66): screens, cover, floor,
# pipes.  At dT = 0 the exact derivative is of order 1e-10^(e-1) and no difference quotient resolves it.
ROOT_PAIRS = ((2, 3), (2, 7), (7, 3), (2, 20), (20, 3), (3, 5), (2, 8), (9, 2), (19, 2))


# screen controls (thScr, blScr): at u = 1 the screen air flux (1 - u) sqrt(buoy (1 - u) + 1e-10) has the exact slope
# -sqrt(1e-10) rMean, but it bends on a scale of 1e-10 / buoy in u, far below any difference step, and u + h leaves the domain;
# with thScr = blScr the two screens' fluxes tie in fmin(fThScr, fBlScr), and a central difference averages the two one-sided
# slopes where the tangent takes the first argument's; at u = 0 (within a difference step of it) the screens' convection
# coefficients |1.7 u |dT|^(1/3)| have their fabs kink, where the tangent takes fabs'(0) = 0 and a difference straddling 0 cannot
SCREENS = (2, 5)


def _fd_blind_columns(u):
    """Control columns a central difference cannot check at this u (see SCREENS)."""
    if u[2] == u[5]:
        return [28 + c for c in SCREENS]
    return [28 + c for c in SCREENS if u[c] >= 1.0 - 1e-3 or u[c] <= 1e-6]


def _on_root_kink(x, tol=1e-2):
    return min(abs(x[a] - x[b]) for a, b in ROOT_PAIRS) < tol


def _fd_rhs(oracle, x, u, d, p, j, h):
    def F(hh):
        xx, uu = _perturbed(x, u, j, hh)
        o = np.zeros(28)
        oracle.glgo_rhs(P(xx), P(uu), P(d), P(p), P(o))
        return o
    c1 = (F(h) - F(-h)) / (2 * h)
    c2 = (F(h / 2) - F(-h / 2)) / h
    return (4 * c2 - c1) / 3, c1, c2


def test_host_rhs_jacobian_matches_richardson_differences(hm, oracle, rhs_golden):
    """At the golden points: scaled entries within 1e-6 of central differences with Richardson extrapolation of glgo_rhs.  The
    points where two temperatures of a fractional-power flux coincide within 0.01 K (among them the initial states, all at one temperature)
    are left out: the exact derivative there is the root's near-singular slope, which a difference of step 1e-4 |T| averages away.
    Entries whose difference quotient has not converged (h and h/2 disagree by more than 1e-5 scaled) sit on a kink the
    difference straddles -- |tAir - tTop + 1e-10|^0.66 at tAir = tTop, or a screen at u = 1, where sqrt(buoy (1 - u) + 1e-10) bends
    on a scale of 1e-10 / buoy -- and are not compared; they are fewer than 0.5 % of all entries."""
    skipped = total = 0
    worst = 0.0
    pts = [i for i in range(len(rhs_golden["x"])) if not _on_root_kink(rhs_golden["x"][i])]
    assert len(pts) >= 360
    for i in pts:
        x, u, d, p = (_c(rhs_golden[k][i]) for k in "xudp")
        general = 0 if hm.hm_nominal_structure(P(p)) else 1
        _, jx, ju, _ = host_rhs_jac(hm, x, u, d, p, general)
        D = _scale(x)
        J = np.concatenate([jx, ju], 1)
        R = np.zeros_like(J)
        ok = np.ones(J.shape, bool)
        for j in range(34):
            h = 1e-4 * D[j]
            R[:, j], c1, c2 = _fd_rhs(oracle, x, u, d, p, j, h)
            ok[:, j] = np.abs(c1 - c2) * D[j] / D[:28] <= 1e-5
        E = np.abs(_scaled(J, D) - _scaled(R, D))
        worst = max(worst, float(E[ok].max()))
        skipped += int((~ok).sum())
        total += ok.size
    assert worst <= 1e-6, worst
    assert skipped <= 0.005 * total, (skipped, total)


def _pick(n, k=20, skip=()):
    idx = [i for i in np.linspace(0, n - 1, min(n, k + len(skip))).astype(int) if i not in skip]
    return sorted(set(idx))[:k] if n > k else sorted(set(idx))


@pytest.mark.parametrize("truth", ["truth_rule_based", "truth_random_actions", "truth_harvest_window"])
@pytest.mark.parametrize("integrator", [0, 1])
def test_host_step_jacobian_matches_central_differences(hm, oracle, truth, integrator):
    """At least 20 intervals of the rule-based and random-action traces and 12 of the 24 harvest-window points, fixed (n_sub 600) and graded (n_sub 260) grids: scaled
    entries of dx_next/dx and dx_next/du within 1e-6 of central differences of glgo_evalf_ex.  The oracle's executed step count
    is asserted to be the same at x + h and x - h as at x, so no difference straddles a grid switch; intervals that start within
    a difference step of a micro-step boundary (_on_grid_switch) or on a root kink (_on_root_kink) are not used.  The column of a screen
    at u = 0 or closed at u = 1, and both screen columns when the two screens are equal, are not compared (see SCREENS)."""
    z = np.load(os.path.join(GOLDEN, truth + ".npz"))
    p = _c(z["p"])
    n_sub, guard = (600, 0) if integrator == 0 else (260, GRADED)
    pts = [i for i in _pick(len(z["x"]), 24) if not _on_root_kink(z["x"][i], 1e-3)][:20]
    general = 0 if hm.hm_nominal_structure(P(p)) else 1
    worst = 0.0
    used = n_blind = 0
    for i in pts:
        x, u, d = (_c(z[k][i]) for k in "xud")
        if _on_grid_switch(oracle, x, u, d, p, n_sub, guard):
            continue
        used += 1
        _, jx, ju, bad = host_step_jac(hm, x, u, d, p, n_sub, integrator, general)
        assert bad == 0
        n0 = C.c_long(0)
        y = np.zeros(28)
        oracle.glgo_evalf_ex(P(x), P(u), P(d), P(p), 900.0, n_sub, guard, P(y), C.byref(n0))
        D = _scale(x)
        J = np.concatenate([jx, ju], 1)
        R = np.zeros_like(J)
        blind = _fd_blind_columns(u)
        for j in range(34):
            # central differences at h, h/10, ... until two successive ones agree to 1e-7 scaled: a smooth kink (a sigmoid or a
            # root of a tiny argument somewhere on the trajectory) can bend the map on a scale below 1e-5 |x|
            h, prev, conv = 1e-5 * D[j], None, False
            for _ in range(4):
                outs = []
                for s in (1, -1):
                    xx, uu = _perturbed(x, u, j, s * h)
                    o, n = np.zeros(28), C.c_long(0)
                    oracle.glgo_evalf_ex(P(xx), P(uu), P(d), P(p), 900.0, n_sub, guard, P(o), C.byref(n))
                    assert n.value == n0.value, (i, j, h, n.value, n0.value)  # the same grid at x + h, x - h and x
                    outs.append(o)
                c = (outs[0] - outs[1]) / (2 * h)
                if prev is not None and np.max(np.abs(c - prev) * D[j] / D[:28]) <= 1e-7:
                    conv = True
                    break
                prev, h = c, h / 10
            R[:, j] = c
            if not conv:  # no converged reference: the trajectory passes a kink within every step tried
                blind.append(j)
        E = np.abs(_scaled(J, D) - _scaled(R, D))
        E[:, blind] = 0.0
        n_blind += len(blind)
        worst = max(worst, float(E.max()))
    assert worst <= 1e-6, worst
    assert used >= (20 if truth != "truth_harvest_window" else 12), used
    assert n_blind <= 0.1 * 34 * used, n_blind  # the screen columns at their bounds, mostly


def _on_grid_switch(oracle, x, u, d, p, n_sub, guard):
    """True when a difference step of 1e-5 |x| in some direction changes the oracle's executed step count (a harvest micro-step
    boundary): the map jumps there and has no derivative to compare with."""
    D = _scale(x)
    ns = set()
    for j in range(34):
        for s in (1, 0, -1):
            xx, uu = _perturbed(x, u, j, s * 1e-5 * D[j])
            o, n = np.zeros(28), C.c_long(0)
            oracle.glgo_evalf_ex(P(xx), P(uu), P(d), P(p), 900.0, n_sub, guard, P(o), C.byref(n))
            ns.add(n.value)
    return len(ns) > 1


def test_host_rhs_spectra_match_the_forward_difference_trace(hm):
    """The largest |Re lambda| of the exact df/dx at the rule-based truth states matches the committed forward-difference
    trace (make_truth.py) within 1e-4 relative; at the 120 random-action points it spans DESIGN.md's 0.665-0.688 1/s."""
    z = np.load(os.path.join(GOLDEN, "truth_rule_based.npz"))
    p = _c(z["p"])
    lam = np.array([np.abs(np.linalg.eigvals(host_rhs_jac(hm, _c(z["x"][i]), _c(z["u"][i]), _c(z["d"][i]), p, 0)[1]).real).max()
                    for i in range(len(z["x"]))])
    # states on a root kink (among them the season's first, every temperature equal) are left out: a forward difference of step
    # 1e-6 |T| cannot resolve the near-singular slope there (see _on_root_kink); the first state's committed value is 3e-4 off
    ok = np.array([not _on_root_kink(x) for x in z["x"]])
    assert ok.sum() >= len(ok) - 10
    assert np.all(np.abs(lam - z["lam"])[ok] <= 1e-4 * z["lam"][ok]), np.abs(lam / z["lam"] - 1)[ok].max()
    r = np.load(os.path.join(GOLDEN, "truth_random_actions.npz"))
    p = _c(r["p"])
    lr = np.array([np.abs(np.linalg.eigvals(host_rhs_jac(hm, _c(r["x"][i]), _c(r["u"][i]), _c(r["d"][i]), p, 0)[1]).real).max()
                   for i in range(len(r["x"]))])
    assert (round(lr.min(), 3), round(lr.max(), 3)) == (0.665, 0.688), (lr.min(), lr.max())  # 0.66490 .. 0.68815


def test_linearisation_entry_points_exported_and_reject_null():
    from glgym import _lib
    lib = _lib.load()
    for name in ("glg_rhs_jacobian_batch", "glg_evalf_jacobian_batch", "glg_linearize"):
        assert hasattr(lib, name), name
    buf = (C.c_double * (28 * 34))()
    b = C.addressof(buf)
    assert lib.glg_linearize(None, None, None, b, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_linearize(None, None, None, None, None, None) == _lib.GLG_ERR_ARG
    # the pure functions validate before touching a device: NULL inputs, NULL jx, B < 1, bad p_stride / n_sub / integrator
    for args in ((None, b, b, b, 0, b, b, b, 1), (b, b, b, b, 0, b, None, b, 1), (b, b, b, b, 0, b, b, b, 0),
                 (b, b, b, b, 7, b, b, b, 1)):
        assert lib.glg_rhs_jacobian_batch(*args, 0, None) == _lib.GLG_ERR_ARG, args
    good = (b, b, b, b, 0, b, b, b, None, 1, 900.0, 600, 0, 0, None)
    assert lib.glg_evalf_jacobian_batch(*good[:6], None, *good[7:]) == _lib.GLG_ERR_ARG  # NULL jx
    assert lib.glg_evalf_jacobian_batch(None, *good[1:]) == _lib.GLG_ERR_ARG
    assert lib.glg_evalf_jacobian_batch(*good[:11], 0, *good[12:]) == _lib.GLG_ERR_ARG  # n_sub = 0
    assert lib.glg_evalf_jacobian_batch(*good[:12], 2, *good[13:]) == _lib.GLG_ERR_ARG  # integrator = 2
    assert lib.glg_evalf_jacobian_batch(*good[:9], 0, *good[10:]) == _lib.GLG_ERR_ARG  # B = 0


# ------------------------------------------------------------------------------------------------ GPU tier
def _model(integrator):
    from glgym.model import GreenLight
    return GreenLight(integrator=integrator)


def _truth_batch(name, n=16):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    idx = _pick(len(z["x"]), n)
    return _c(z["x"][idx]), _c(z["u"][idx]), _c(z["d"][idx]), _c(z["p"])


def _general_p(p):
    q = p.copy()
    q[70] = 0.05  # sky FIR through the roof: the GENERAL variant
    return q


@pytest.mark.gpu
def test_device_rhs_jacobian_matches_host_dual(hm, rhs_golden):
    m = _model("fixed")
    x, u, d, p = (_c(rhs_golden[k]) for k in "xudp")
    f, jx, ju = (t.cpu().numpy() for t in m.rhs_jacobian_batch(x, u, d, p))
    worst = fworst = 0.0
    for i in range(len(x)):
        general = 0 if hm.hm_nominal_structure(P(p[i])) else 1
        hf, hjx, hju, _ = host_rhs_jac(hm, x[i], u[i], d[i], p[i], general)
        D = _scale(x[i])
        E = np.abs(_scaled(np.concatenate([jx[i], ju[i]], 1), D) - _scaled(np.concatenate([hjx, hju], 1), D))
        worst = max(worst, float(E.max()))
        fworst = max(fworst, rel_err(f[i], hf, 1e-3))
    # the device's contracted FMAs and hardware-seeded roots against the host's separate roundings: single entries of f and of
    # df/dx cancel (the carbohydrate balances to ~1e-8 of their terms, DESIGN.md), which lifts a 1e-16 difference of the terms
    # to ~1e-11 of the result; the step Jacobians, sums over 300 RK4 steps, agree to 1e-12
    assert fworst <= 1e-10, fworst
    assert worst <= 1e-10, worst


@pytest.mark.gpu
@pytest.mark.parametrize("integrator", ["fixed", "graded"])
@pytest.mark.parametrize("general", [False, True])
def test_device_step_jacobian_matches_host_dual_and_evalf(hm, integrator, general):
    m = _model(integrator)
    x, u, d, p = _truth_batch("truth_random_actions")
    if general:
        p = _general_p(p)
    xn, jx, ju, bad = (t.cpu().numpy() for t in m.jacobian_batch(x, u, d, p, return_bad=True))
    ref, rbad = m.evalF_batch(x, u, d, p, return_bad=True)
    assert rel_err(xn, ref.cpu().numpy(), 1e-3) <= 1e-12
    assert np.array_equal(bad, rbad.cpu().numpy())
    worst = 0.0
    for i in range(len(x)):
        _, hjx, hju, hbad = host_step_jac(hm, x[i], u[i], d[i], p, m.n_sub, 0 if integrator == "fixed" else 1, int(general))
        assert hbad == bad[i]
        D = _scale(x[i])
        E = np.abs(_scaled(np.concatenate([jx[i], ju[i]], 1), D) - _scaled(np.concatenate([hjx, hju], 1), D))
        worst = max(worst, float(E.max()))
    assert worst <= 1e-12, worst
    # per-env p with equal rows gives the shared-p result (the GENERAL per-env kernel for both tables)
    pe = np.repeat(p[None], len(x), 0)
    xn2, jx2, ju2 = (t.cpu().numpy() for t in m.jacobian_batch(x, u, d, pe))
    assert rel_err(xn2, xn, 1e-3) <= 1e-12
    D = np.stack([_scale(v) for v in x])
    assert np.abs(_scaled(np.concatenate([jx2, ju2], 2), D) - _scaled(np.concatenate([jx, ju], 2), D)).max() <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("integrator", ["fixed", "graded"])
@pytest.mark.parametrize("general", [False, True])
def test_device_step_jacobian_matches_evalf_differences(integrator, general):
    """Central differences of glg_evalf_batch_ex (steps 1e-5 |x| shrunk by 10 until two agree to 1e-7 scaled) against the
    device Jacobian, at 16 random-action intervals; columns without a converged difference and the screen columns at their
    bounds (SCREENS) are not compared."""
    m = _model(integrator)
    x, u, d, p = _truth_batch("truth_random_actions")
    if general:
        p = _general_p(p)
    _, jx, ju = (t.cpu().numpy() for t in m.jacobian_batch(x, u, d, p))
    B = len(x)
    D = np.stack([_scale(v) for v in x])
    prev, conv, R = None, np.zeros((B, 34), bool), np.zeros((B, 34, 28))
    for level in range(4):
        h = 1e-5 * D / 10 ** level  # [B, 34]
        X = np.repeat(x[:, None], 68, 1)
        U = np.repeat(u[:, None], 68, 1)
        for j in range(34):
            for s, r in ((1, 2 * j), (-1, 2 * j + 1)):
                if j < 28:
                    X[:, r, j] += s * h[:, j]
                else:
                    U[:, r, j - 28] += s * h[:, j]
        out = m.evalF_batch(X.reshape(-1, 28), U.reshape(-1, 6), np.repeat(d, 68, 0), p).cpu().numpy().reshape(B, 34, 2, 28)
        c = np.transpose((out[:, :, 0] - out[:, :, 1]) / (2 * h[:, :, None]), (0, 2, 1))  # [B, 28, 34]
        if prev is not None:
            ok = np.max(np.abs(c - prev) * D[:, None, :] / D[:, :28, None], axis=1) <= 1e-7
            R[ok & ~conv] = np.transpose(c, (0, 2, 1))[ok & ~conv]
            conv |= ok
        prev = c
    R = np.transpose(R, (0, 2, 1))
    E = np.abs(_scaled(np.concatenate([jx, ju], 2), D) - _scaled(R, D))
    for i in range(B):
        E[i][:, _fd_blind_columns(u[i])] = 0.0
        E[i][:, ~conv[i]] = 0.0
    assert conv.sum() >= 0.9 * conv.size, conv.sum()
    assert E.max() <= 1e-6, E.max()


def _venv(B, **kw):
    from glgym.vec_env import GreenLightVecEnv
    return GreenLightVecEnv(B, **kw)


SHORT = dict(season_length=1, start_train_day=0, end_train_day=2)  # 97-step episodes, three weather tables


def _snapshot(env):
    st = env.state_dict()
    views = [env.obs_t, env.reward_t, env.done_t, env.info_t, env.stats_t]
    return st, [v.clone() for v in views]


def _same(a, b):
    sa, va = a
    sb, vb = b
    return all(np.array_equal(sa[k], sb[k]) for k in sa) and all(torch_equal(x, y) for x, y in zip(va, vb))


def torch_equal(a, b):
    import torch
    return torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("integrator", ["fixed", "graded"])
def test_linearize_on_a_handle(integrator):
    """glg_linearize through two auto-resets and each episode's last step (the weather clamp): x_next equals the state the raw
    step then produces, the Jacobians are glg_evalf_jacobian_batch's on the env's state, clamped weather row and parameters bit
    for bit, the env is untouched and the call is one launch."""
    import torch
    from glgym.model import GreenLight
    env = _venv(8, base_env_params=SHORT, integrator=integrator, seed=3)
    env.reset_tensor()
    m = GreenLight(integrator=integrator, n_sub=env.n_sub)
    p64 = np.ascontiguousarray(env.p, dtype=np.float64)
    W = env.weather_tables
    resets = 0
    for t in range(200):
        u = env.rule_controls_tensor().clone()
        before = _snapshot(env)
        n0 = env.launch_count()
        xn, A, Bu = env.linearize_tensor(u)
        assert env.launch_count() == n0 + 1
        assert _same(before, _snapshot(env)), t
        if t % 7 == 0 or t % 97 == 96:
            st = before[0]
            rows = np.stack([W[st["table"][e], min(st["timestep"][e], W.shape[1] - env.Np - 1)] for e in range(8)])
            rx, rA, rB = m.jacobian_batch(st["x"], u, rows, p64)
            assert torch.equal(xn, rx) and torch.equal(A, rA) and torch.equal(Bu, rB), t
        xn_cur = xn.clone()
        env.step_raw_control_tensor(u)
        done = env.done_t.bool()
        x_after = env.state_t.T
        live = ~done
        if live.any():
            assert rel_err(x_after[live].cpu().numpy(), xn_cur[live].cpu().numpy(), 1e-3) <= 1e-12, t
        resets += int(done.any())
    assert resets == 2
    # the env's own u when controls is None
    env.step_raw_control_tensor(env.rule_controls_tensor())
    a = env.linearize_tensor(None)
    b = env.linearize_tensor(env.controls_t.T.contiguous())
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(precision="fp32", role_warps=2), dict(uncertainty_scale=0.3)])
def test_linearize_is_fp64_nominal_on_any_handle(kw):
    import torch
    env = _venv(8, base_env_params=SHORT, seed=5, **kw)
    twin = _venv(8, base_env_params=SHORT, seed=5)
    env.reset_tensor()
    twin.reset_tensor()
    for _ in range(5):
        env.step_rule_based_tensor()
    st = env.state_dict()
    twin.load_state_dict({k: st[k] for k in ("x", "u", "timestep", "table", "time")})
    u = env.rule_controls_tensor().clone()
    a = env.linearize_tensor(u)
    b = twin.linearize_tensor(u)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    env.close()
    twin.close()


@pytest.mark.gpu
def test_linearize_error_paths():
    from glgym import _lib
    env = _venv(4, base_env_params=SHORT)
    with pytest.raises(_lib.GlgError, match=f"status {_lib.GLG_ERR_STATE}"):
        env.linearize_tensor()
    env.reset_tensor()
    assert env._lib.glg_linearize(env._h, None, None, None, None, None) == _lib.GLG_ERR_ARG
    assert env._lib.glg_linearize(None, None, None, None, None, None) == _lib.GLG_ERR_ARG
    import torch
    with pytest.raises(ValueError):
        env.linearize_tensor(torch.zeros((3, 6), dtype=torch.float64, device="cuda"))
    env.close()
