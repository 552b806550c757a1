"""Noise identification (csrc/glg_em.cuh, glgym.estimation.DeviceNoiseEM): the sigma-point E-step against Shumway-Stoffer's
expectations on a linear-Gaussian model, EM's monotone likelihood there, the data log against what the env applied and the caller
passed, the device E-step against a numpy restatement of its contract (include/glgym.h), chunking and replay bit for bit, and the
recovery of a known Q and R."""
import ctypes as C
import types

import numpy as np
import pytest

from test_gpu_estimation import chol_rule, h7, scaled_err, sigma_points, ukf_weights

torch = pytest.importorskip("torch")

N_X = 28
SEGMENT = 1 | 4 | 8
SHORT2 = dict(season_length=7 / 96.0, start_train_day=0, end_train_day=1)  # N = 7, two weather tables
LOG2PI = float(np.log(2 * np.pi))


# ---- numpy restatement of the E-step contract ----------------------------------------------------------------------------------
def estep_q(ms_prev, Ps_prev, ms_k, Ps_k, G_prev, f, wm, wc, g):
    """E_k and fbar of one transition; f [2n+1][n] are the points of (ms_prev, Ps_prev) stepped by the model."""
    n = len(ms_k)
    L = chol_rule(Ps_prev)
    fbar = (wm[:, None] * f).sum(0)
    dF = f - fbar
    Phi = (wc[:, None, None] * (dF[:, :, None] * dF[:, None, :])).sum(0)
    Z = wm[1] * g * (f[1:n + 1] - f[n + 1:])  # row j: W gamma (f_{j+} - f_{j-})
    for j in reversed(range(n)):
        Z[j] = (Z[j] - L[j + 1:, j] @ Z[j + 1:]) / L[j, j] if L[j, j] != 0 else 0.0
    Cm = Ps_k @ G_prev.T @ Z
    d = ms_k - fbar
    return np.diag(Ps_k + np.outer(d, d) + Phi - Cm - Cm.T), fbar


def estep_r(ms, Ps, y, measured, wm, wc, g, h):
    H = h(sigma_points(ms, Ps, g))
    hb = (wm[:, None] * H).sum(0)
    v = (wc[:, None] * (H - hb) ** 2).sum(0)
    return np.where(measured, (y - hb) ** 2 + v, 0.0)


def kalman_rts(A, H, x0, P0, q, r, ys, starts):
    """Textbook Kalman filter and RTS smoother of x' = A x + w, y = H x + v; a slot in `starts` restarts at (x0, P0).  Returns the
    log-likelihood, the smoothed means, covariances and gains (G = 0 across a restart; deterministic rows left out)."""
    n, T = len(x0), len(ys)
    active = (np.diag(P0) > 0) | (q > 0)
    a = np.flatnonzero(active)
    xf, Pf, xp, Pp = [x0], [P0], [None], [None]
    ll = 0.0
    for k in range(1, T):
        if k in starts:
            xf.append(x0); Pf.append(P0); xp.append(None); Pp.append(None)
            continue
        xk, Pk = A @ xf[-1], A @ Pf[-1] @ A.T + np.diag(q ** 2)
        S = H @ Pk @ H.T + np.diag(r ** 2)
        v = ys[k] - H @ xk
        ll += -0.5 * (v @ np.linalg.solve(S, v) + np.linalg.slogdet(S)[1] + len(v) * LOG2PI)
        K = Pk @ H.T @ np.linalg.inv(S)
        Pu = (np.eye(n) - K @ H) @ Pk
        xf.append(xk + K @ v); Pf.append(0.5 * (Pu + Pu.T)); xp.append(xk); Pp.append(Pk)
    xs, Ps, G = list(xf), list(Pf), [np.zeros((n, n)) for _ in range(T)]
    for k in range(T - 2, -1, -1):
        if k + 1 in starts:
            continue
        Gk = np.zeros((n, n))
        Gk[np.ix_(a, a)] = (Pf[k] @ A.T)[np.ix_(a, a)] @ np.linalg.inv(Pp[k + 1][np.ix_(a, a)])
        G[k] = Gk
        xs[k] = xf[k] + Gk @ (xs[k + 1] - xp[k + 1])
        Pk = Pf[k] + Gk @ (Ps[k + 1] - Pp[k + 1]) @ Gk.T
        Ps[k] = 0.5 * (Pk + Pk.T)
    return ll, np.array(xs), np.array(Ps), np.array(G)


def _linear_model(seed):
    rng = np.random.default_rng(seed)
    n = N_X
    A = np.eye(n) + 0.05 * rng.standard_normal((n, n))
    A[27] = 0.0
    A[27, 27] = 1.0
    H = 0.3 * rng.standard_normal((7, n))
    H[:, 27] = 0.0
    Gm = rng.standard_normal((n, n))
    P0 = Gm @ Gm.T / n + 0.1 * np.eye(n)
    P0[27, :] = P0[:, 27] = 0.0
    q = np.abs(rng.standard_normal(n)) * 0.2
    q[27] = 0.0
    r = np.full(7, 0.3)
    return rng, A, H, P0, q, r


def _simulate(rng, A, H, x0, q, r, T, starts):
    xs, ys = [x0], [np.zeros(7)]
    for k in range(1, T):
        x = x0 if k in starts else A @ xs[-1] + q * rng.standard_normal(len(x0))
        xs.append(x)
        ys.append(H @ x + r * rng.standard_normal(7))
    return np.array(xs), np.array(ys)


def _restated_em_sums(A, H, ms, Ps, G, ys, starts, wm, wc, g):
    Eq, Er, ntr = np.zeros(N_X), np.zeros(7), 0
    for k in range(1, len(ms)):
        if k not in starts:
            f = sigma_points(ms[k - 1], Ps[k - 1], g) @ A.T
            Eq += estep_q(ms[k - 1], Ps[k - 1], ms[k], Ps[k], G[k - 1], f, wm, wc, g)[0]
            ntr += 1
            Er += estep_r(ms[k], Ps[k], ys[k], np.ones(7, bool), wm, wc, g, lambda x: x @ H.T)
    return Eq, Er, ntr


# ---- CPU tier ------------------------------------------------------------------------------------------------------------
def test_em_entry_points_exported_and_reject_null():
    from glgym import _lib
    lib = _lib.load()
    out = C.c_void_p()
    assert lib.glg_em_create(None, 0, C.byref(out)) == _lib.GLG_ERR_ARG and not out
    assert lib.glg_em_estep(None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_est_set_noise(None, None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_em_bytes(None) == 0 and lib.glg_em_logged(None) == 0 and lib.glg_em_chunk_pairs(None) == 0
    for view in ("controls", "table", "measurements", "flags", "loglik", "expectation", "prediction", "used", "env_stats",
                 "totals"):
        assert getattr(lib, f"glg_em_{view}_dev")(None) is None
    lib.glg_em_destroy(None)


@pytest.mark.parametrize("kw, exc, match", [
    (dict(max_points=56), ValueError, "max_points"), (dict(max_points=4194305), ValueError, "max_points"),
    (dict(max_points=1e6), ValueError, "max_points"), (dict(fit_q=[True] * 28), ValueError, "fit_q"),
    (dict(fit_q=np.ones(28, bool)), ValueError, "x27"), (dict(fit_r=np.ones(6, bool)), ValueError, "fit_r"),
    (dict(fit_r=np.ones(7, bool)), ValueError, "measured"), (dict(q_floor=[-1.0] * 28), ValueError, "q_floor"),
    (dict(r_floor=[0.1] * 6), ValueError, "r_floor"),
])
def test_em_arguments_are_validated_before_anything_is_created(kw, exc, match):
    from glgym.estimation import DEFAULT_P0_STD, DEFAULT_Q_STD, DeviceNoiseEM, DeviceStateSmoother
    est = types.SimpleNamespace(p0_std=np.array(DEFAULT_P0_STD), q_std=np.array(DEFAULT_Q_STD), measured=["co2_air"],
                                env=types.SimpleNamespace(num_envs=4))
    sm = DeviceStateSmoother.__new__(DeviceStateSmoother)  # never reached: no C object is created
    sm.est, sm.window = est, 8
    with pytest.raises(exc, match=match):
        DeviceNoiseEM(sm, **kw)
    with pytest.raises(TypeError, match="DeviceStateSmoother"):
        DeviceNoiseEM(est)


@pytest.mark.parametrize("kw, match", [(dict(q_std=[np.nan] + [1.0] * 27), "q_std"), (dict(p0_std=[1.0] * 27), "p0_std"),
                                       (dict(r_std=[20.0, 0.0, 2.0, 0.5, 0.5, 500.0, 10.0]), "r_std must be > 0")])
def test_set_noise_is_validated_before_the_library_is_called(kw, match):
    from glgym.estimation import DeviceStateEstimator
    est = DeviceStateEstimator.__new__(DeviceStateEstimator)
    est.measured = ["temp_air"]
    with pytest.raises(ValueError, match=match):
        est.set_noise(**kw)


@pytest.mark.parametrize("alpha, beta, kappa", [(1.0, 2.0, 0.0), (0.5, 2.0, 1.0), (0.8, 1.0, -2.0)])
def test_restated_sigma_point_estep_equals_shumway_stoffer_on_a_linear_gaussian_model(alpha, beta, kappa):
    """For f(x) = A x and h(x) = H x the sigma-point E-step is exact: E_k = diag E[(x_k - A x_{k-1})^2] and the R term is
    (y - H ms)^2 + diag(H Ps H^T).  x27 is deterministic; slot 6 restarts (a segment start: no transition leads to it)."""
    rng, A, H, P0, q, r = _linear_model(11)
    starts = {6}
    T = 11
    x0 = rng.standard_normal(N_X)
    _, ys = _simulate(rng, A, H, x0, q, r, T, starts)
    _, ms, Ps, G = kalman_rts(A, H, x0, P0, q, r, ys, starts)
    wm, wc, g = ukf_weights(alpha, beta, kappa)
    for k in range(1, T):
        if k in starts:
            continue
        f = sigma_points(ms[k - 1], Ps[k - 1], g) @ A.T
        E, fbar = estep_q(ms[k - 1], Ps[k - 1], ms[k], Ps[k], G[k - 1], f, wm, wc, g)
        d = ms[k] - A @ ms[k - 1]
        cross = Ps[k] @ G[k - 1].T @ A.T
        ref = np.diag(Ps[k] + np.outer(d, d) + A @ Ps[k - 1] @ A.T - cross - cross.T)
        assert scaled_err(fbar, A @ ms[k - 1]) <= 1e-12, k
        assert scaled_err(E, ref) <= 1e-12, (k, scaled_err(E, ref))
        Er = estep_r(ms[k], Ps[k], ys[k], np.ones(7, bool), wm, wc, g, lambda x: x @ H.T)
        e = ys[k] - H @ ms[k]
        assert scaled_err(Er, e * e + np.diag(H @ Ps[k] @ H.T)) <= 1e-12, k


def test_restated_em_never_decreases_the_likelihood():
    """20 iterations of the restated E-step and the M-step q_j^2 = sum E_j / transitions, r^2 = sum R / measurements on the
    linear-Gaussian model, from noise 4x too large; p0 is held fixed (a generalised EM step)."""
    rng, A, H, P0, q_true, r_true = _linear_model(3)
    starts = {25}
    T = 60
    x0 = rng.standard_normal(N_X)
    _, ys = _simulate(rng, A, H, x0, q_true, r_true, T, starts)
    wm, wc, g = ukf_weights()
    q, r = 4 * q_true, 4 * r_true
    lls = []
    for _ in range(20):
        ll, ms, Ps, G = kalman_rts(A, H, x0, P0, q, r, ys, starts)
        lls.append(ll)
        Eq, Er, ntr = _restated_em_sums(A, H, ms, Ps, G, ys, starts, wm, wc, g)
        q = np.where(np.arange(N_X) < 27, np.sqrt(Eq / ntr), 0.0)
        r = np.sqrt(Er / ntr)  # every linked slot is measured here
    d = np.diff(lls)
    assert np.all(d >= -1e-9 * np.abs(np.array(lls[1:]))), d
    assert lls[-1] > lls[0]


def noredraw_rts(A, H, x0, P0, q, r, ys, starts):
    """kalman_rts with the estimator's moments on a linear model: its points are not redrawn after adding Q, so Q enters P- but
    not S and C (S = H (P- - Q) H^T + R, C = (P- - Q) H^T)."""
    n, T = len(x0), len(ys)
    a = np.flatnonzero((np.diag(P0) > 0) | (q > 0))
    xf, Pf, xp, Pp = [x0], [P0], [None], [None]
    ll = 0.0
    for k in range(1, T):
        if k in starts:
            xf.append(x0); Pf.append(P0); xp.append(None); Pp.append(None)
            continue
        xk, P0k = A @ xf[-1], A @ Pf[-1] @ A.T
        Pk = P0k + np.diag(q ** 2)
        S = H @ P0k @ H.T + np.diag(r ** 2)
        v = ys[k] - H @ xk
        ll += -0.5 * (v @ np.linalg.solve(S, v) + np.linalg.slogdet(S)[1] + len(v) * LOG2PI)
        K = P0k @ H.T @ np.linalg.inv(S)
        Pu = Pk - K @ S @ K.T
        xf.append(xk + K @ v); Pf.append(0.5 * (Pu + Pu.T)); xp.append(xk); Pp.append(Pk)
    xs, Ps, G = list(xf), list(Pf), [np.zeros((n, n)) for _ in range(T)]
    for k in range(T - 2, -1, -1):
        if k + 1 in starts:
            continue
        Gk = np.zeros((n, n))
        Gk[np.ix_(a, a)] = (Pf[k] @ A.T)[np.ix_(a, a)] @ np.linalg.inv(Pp[k + 1][np.ix_(a, a)])
        G[k] = Gk
        xs[k] = xf[k] + Gk @ (xs[k + 1] - xp[k + 1])
        Pk = Pf[k] + Gk @ (Ps[k + 1] - Pp[k + 1]) @ Gk.T
        Ps[k] = 0.5 * (Pk + Pk.T)
    return ll, np.array(xs), np.array(Ps), np.array(G)


def _em_lls(filt, scale_q, iterations=10):
    rng, A, H, P0, q_true, r_true = _linear_model(3)
    q_true = scale_q * q_true
    T = 80
    x0 = rng.standard_normal(N_X)
    _, ys = _simulate(rng, A, H, x0, q_true, r_true, T, set())
    wm, wc, g = ukf_weights()
    q, r, lls = 4 * q_true, 4 * r_true, []
    for _ in range(iterations):
        ll, ms, Ps, G = filt(A, H, x0, P0, q, r, ys, set())
        lls.append(ll)
        Eq, Er, ntr = _restated_em_sums(A, H, ms, Ps, G, ys, set(), wm, wc, g)
        q, r = np.where(np.arange(N_X) < 27, np.sqrt(Eq / ntr), 0.0), np.sqrt(Er / ntr)
    return np.array(lls), np.median(q[:27] / q_true[:27])


def test_a_filter_that_leaves_q_out_of_s_breaks_ems_monotone_likelihood():
    """The same E-step and M-step on the same data: under the textbook filter the likelihood never decreases; under the
    estimator's moments (Q not in S and C) it does.  And with q far below r, the regime of the greenhouse's climate states, even
    the textbook EM leaves q near its 4x start after 10 iterations: Q is weakly identified there."""
    ll_tb, _ = _em_lls(kalman_rts, 1.0)
    ll_nr, _ = _em_lls(noredraw_rts, 1.0)
    assert np.all(np.diff(ll_tb) >= -1e-9 * np.abs(ll_tb[1:]))
    assert np.any(np.diff(ll_nr) < 0), np.diff(ll_nr)
    _, q_small = _em_lls(kalman_rts, 0.1)
    assert q_small > 3.0, q_small


# ---- GPU tier ------------------------------------------------------------------------------------------------------------
def _env(B, **kw):
    from glgym.vec_env import GreenLightVecEnv
    base = dict(seed=3)
    base.update(kw)
    return GreenLightVecEnv(B, **base)


def _warm(env, steps):
    B = env.num_envs
    env.reset_tensor(table_ids=(torch.arange(B, device="cuda", dtype=torch.int32) * 7) % env.weather_tables.shape[0])
    for _ in range(steps):
        env.step_rule_based_tensor()
    torch.cuda.synchronize()


def _short_env(B, **kw):
    """Envs of a 7-step season on two weather tables; envs 1 and 4 finish four steps after the others."""
    env = _env(B, base_env_params=SHORT2, **kw)
    env.reset_tensor(table_ids=torch.arange(B, device="cuda", dtype=torch.int32) % 2)
    env.step_rule_based_tensor()
    env.step_rule_based_tensor()
    k = env.get_state()[2]
    k[[1, 4]] = 0
    env.set_state(timestep=k)
    return env


def _noisy(est, gen):
    B = est.env.num_envs
    return est.measurements() + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen) * torch.as_tensor(
        est.r_std, device="cuda")


def _p0():
    from glgym.estimation import DEFAULT_P0_STD
    p0 = np.array(DEFAULT_P0_STD)
    p0[11] = 0.0
    return p0


def _trio(env, window, **kw):
    from glgym.estimation import DeviceNoiseEM, DeviceStateEstimator, DeviceStateSmoother
    est = DeviceStateEstimator(env, p0_std=_p0())
    sm = DeviceStateSmoother(est, window)
    em = DeviceNoiseEM(sm, **kw)
    return est, sm, em


def _close(*objs):
    for o in objs:
        o.close()


def _smoother_state(sm):
    s = sm.smooth()
    torch.cuda.synchronize()
    rec = [getattr(sm, k).clone() for k in ("filtered_mean", "filtered_cov", "prior_mean", "prior_cov", "cross_cov", "status",
                                            "timestep")]
    return [v.clone() for v in s] + rec


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_logging_leaves_the_estimator_and_the_smoother_bit_identical(precision):
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B = 6
    env = _short_env(B, precision=precision)
    e1, s1, em = _trio(env, 8)
    e2 = DeviceStateEstimator(env, p0_std=_p0())
    s2 = DeviceStateSmoother(e2, 8)
    e1.reset()
    e2.reset()
    gen = torch.Generator(device="cuda").manual_seed(5)
    reinit = 0
    for t in range(12):
        env.step_rule_based_tensor()
        y = _noisy(e1, gen) if t % 3 else None
        e1.update(y)
        e2.update(y)
        torch.cuda.synchronize()
        for a in ("mean", "cov", "innovation", "status"):
            assert torch.equal(getattr(e1, a), getattr(e2, a)), (t, a)
        reinit += int((e1.status == 4).sum())
    assert reinit >= 4
    for u, v in zip(_smoother_state(s1), _smoother_state(s2)):
        assert torch.equal(u, v)
    _close(em, s1, s2, e1, e2, env)


@pytest.mark.gpu
def test_log_holds_what_the_env_applied_and_the_caller_passed_and_the_loglik_terms():
    from glgym.estimation import DeviceStateEstimator
    B = 5
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 10)
    est, sm, em = _trio(env, 16)
    est.reset()
    wm, wc, _ = ukf_weights()
    gen = torch.Generator(device="cuda").manual_seed(6)
    applied, passed, tables, lls = [np.zeros((B, 6))], [np.zeros((B, 7))], [env.table_t.cpu().numpy().copy()], [np.zeros(B)]
    for t in range(6):
        env.step_rule_based_tensor()
        y = None if t == 2 else _noisy(est, gen)
        m0 = est.mean.clone()
        est.update(y)
        torch.cuda.synchronize()
        applied.append(env.controls_t.T.cpu().numpy().copy())
        tables.append(env.table_t.cpu().numpy().copy())
        passed.append(np.zeros((B, 7)) if y is None else y.cpu().numpy().copy())
        ll = np.zeros(B)
        if y is not None:  # the restated l from the filter's own propagated points
            chi = est.sigma.permute(1, 2, 0).cpu().numpy()
            for b in range(B):
                Y = h7(chi[b])
                yb = (wm[:, None] * Y).sum(0)
                S = (wc[:, None, None] * ((Y - yb)[:, :, None] * (Y - yb)[:, None, :])).sum(0) + np.diag(est.r_std ** 2)
                v = passed[-1][b] - yb
                ll[b] = -0.5 * (v @ np.linalg.solve(S, v) + np.linalg.slogdet(S)[1] + 7 * LOG2PI)
        lls.append(ll)
    assert np.array_equal(em.controls.cpu().numpy(), np.stack(applied))
    assert np.array_equal(em.tables.cpu().numpy(), np.stack(tables))
    assert np.array_equal(em.measurements.cpu().numpy(), np.stack(passed))
    fl = em.flags.cpu().numpy()
    assert fl[0].tolist() == [0] * B and fl[3].tolist() == [0] * B and np.all(fl[[1, 2, 4, 5, 6]] == 3)
    got = em.loglik.cpu().numpy()
    err = np.max(np.abs(got - np.stack(lls)) / np.maximum(np.abs(np.stack(lls)), 1e-300))
    print(f"log-likelihood terms against the restatement: max relative error {err:.2e}")
    assert err <= 1e-12
    _close(em, sm, est, env)


@pytest.mark.gpu
def test_prediction_equals_the_filters_xbar_bit_for_bit_from_the_filtered_moments():
    """With the filtered moments written into the smoother's output (G = 0), the E-step steps the filter's own sigma points: fbar
    is the record's xbar bit for bit.  B = 192 puts the shadow and the EM handles (10 944 and 192 W 57 envs) above the latency
    layout's limit (2 x 148 SMs x 32 = 9472 envs), so both step with the throughput layout."""
    from glgym import _lib
    B, W = 192, 6
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 10)
    est, sm, em = _trio(env, W)
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(7)
    for t in range(W - 1):
        env.step_rule_based_tensor()
        est.update(_noisy(est, gen))
    sm.smooth()
    n = sm.length
    sm._out.mean[:n] = sm.filtered_mean
    sm._out.cov[:n] = sm.filtered_cov
    sm._out.gain.zero_()
    _lib.check(env._lib.glg_em_estep(em._obj, env._stream()), env._h, "glg_em_estep")
    torch.cuda.synchronize()
    assert np.all(em.used.cpu().numpy()[1:] == 3) and np.all(em.used.cpu().numpy()[0] == 2 * 0)
    assert torch.equal(em.prediction[1:], sm.prior_mean[1:])
    _close(em, sm, est, env)


def _restated_estep(env, est, sm, em, s):
    """The device E-step's E and R terms restated in numpy from the smoother's output, with f_i from glg_evalf_batch_ex."""
    from glgym.model import GreenLight
    wm, wc, g = ukf_weights()
    gl = GreenLight(integrator=env.integrator, n_sub=env.n_sub)
    p64 = np.ascontiguousarray(env.p, dtype=np.float64)
    Wt = env.weather_tables
    ms, Ps, G = (v.cpu().numpy() for v in s)
    st, ts = sm.status.cpu().numpy(), sm.timestep.cpu().numpy()
    u, tb, y, fl = (v.cpu().numpy() for v in (em.controls, em.tables, em.measurements, em.flags))
    n, B = ms.shape[:2]
    measured = np.isin(np.arange(7), [["co2_air", "temp_air", "rh_air", "pipe_temp", "24CanTemp", "cFruit", "tSum"].index(m)
                                     for m in est.measured])
    ref = np.zeros((n, B, 35))
    pts, keys = [], []
    for k in range(1, n):
        for b in range(B):
            if not st[k, b] & SEGMENT:
                pts.append(sigma_points(ms[k - 1, b], Ps[k - 1, b], g))
                row = Wt[tb[k, b], min(ts[k, b] - 1, Wt.shape[1] - env.Np - 1)]
                keys.append((k, b, np.repeat(u[k, b][None], 57, 0), np.repeat(row[None], 57, 0)))
    f = gl.evalF_batch(np.concatenate(pts), np.concatenate([q[2] for q in keys]), np.concatenate([q[3] for q in keys]),
                       p64).cpu().numpy().reshape(len(keys), 57, 28)
    for i, (k, b, _, _) in enumerate(keys):
        ref[k, b, :28] = estep_q(ms[k - 1, b], Ps[k - 1, b], ms[k, b], Ps[k, b], G[k - 1, b], f[i], wm, wc, g)[0]
    for k in range(n):
        for b in range(B):
            if fl[k, b] & 2:
                ref[k, b, 28:] = estep_r(ms[k, b], Ps[k, b], y[k, b], measured, wm, wc, g, h7)
    return ref


@pytest.mark.gpu
def test_estep_equals_the_restatement_and_chunking_and_reruns_are_bit_identical():
    """E and the R terms against the restatement; a small max_points (230 pairs: 1536 pairs in 7 balanced chunks, six of 220 and one
    of 216, every one above the latency layout's limit of 9472 points, the first boundary inside env 18's slots) and a second E-step
    give the same bits as one launch.
    glg_evalf_batch_ex agrees with the step kernels to about 1e-9 relative (test_gpu_estimation), and E of a state with a tiny
    q is a difference of such values, so the Q terms are held to that agreement: |dE_j| <= 1e-6 max|E_j| + 2 sqrt(max|E_j|) e_j
    + e_j^2 with e_j = 1e-8 max|f_j|.  x27's E is rounding and is not compared.  The R terms involve no step: 1e-10 scaled."""
    from glgym.estimation import DeviceNoiseEM
    B, W = 128, 12
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 10)
    est, sm, em = _trio(env, W)
    start = env.state_dict()
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(8)
    for t in range(W - 1):
        env.step_rule_based_tensor()
        est.update(None if t == 3 else _noisy(est, gen))
    em.estep()
    torch.cuda.synchronize()
    one = [v.clone() for v in (em.expectation, em.prediction, em.used, em.env_stats, em.totals)]
    em.estep()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(one, (em.expectation, em.prediction, em.used, em.env_stats, em.totals)))
    s = sm.smooth()
    ref = _restated_estep(env, est, sm, em, s)
    got = em.expectation.cpu().numpy()
    errs = {j: scaled_err(got[..., j], ref[..., j]) for j in range(35) if j != 27 and np.any(ref[..., j])}
    print("E-step against the restatement, scaled error per entry:", {j: f"{e:.1e}" for j, e in errs.items()})
    fmax = np.max(np.abs(em.prediction.cpu().numpy()), axis=(0, 1))
    for j in range(27):
        big, e = np.max(np.abs(ref[..., j])), 1e-8 * fmax[j]
        assert np.max(np.abs(got[..., j] - ref[..., j])) <= 1e-6 * big + 2 * np.sqrt(big) * e + e * e, (j, errs.get(j))
    assert max(errs[j] for j in range(28, 35) if j in errs) <= 1e-10
    used = em.used.cpu().numpy()
    tot = em.totals.cpu().numpy()
    assert tot[35] == (used & 1).sum() and tot[36] == (used >> 1 & 1).sum() == B * (W - 2)
    assert np.isclose(tot[37], em.loglik.cpu().numpy().sum(), rtol=1e-12)
    # the same run again (state_dict restores the Philox position), its window in chunks of at most 230 pairs
    em.close()
    em2 = DeviceNoiseEM(sm, max_points=57 * 230)
    assert em2.chunk_pairs == 230
    env.load_state_dict(start)
    gen = torch.Generator(device="cuda").manual_seed(8)
    est.reset()
    for t in range(W - 1):
        env.step_rule_based_tensor()
        est.update(None if t == 3 else _noisy(est, gen))
    em2.estep()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(one, (em2.expectation, em2.prediction, em2.used, em2.env_stats, em2.totals)))
    _close(em2, sm, est, env)


def _drive(env, est, steps, gen, driver):
    B = env.num_envs
    for t in range(steps):
        if driver == "rule":
            env.step_rule_based_tensor()
        else:
            env.step_tensor(torch.rand(B, 6, device="cuda", generator=gen, dtype=torch.float32) * 2 - 1)
        est.update(None if t % 5 == 4 else _noisy(est, gen))


@pytest.mark.gpu
@pytest.mark.parametrize("driver", ["rule", "actions"])
def test_replay_reproduces_the_record_the_log_and_the_estep(driver):
    B, W = 8, 24
    env = _env(B, uncertainty_scale=0.2)
    _warm(env, 5)
    est, sm, em = _trio(env, W)
    start = env.state_dict()
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(9)
    _drive(env, est, W - 1, gen, driver)
    em.estep()
    torch.cuda.synchronize()
    logs = lambda: [v.clone() for v in (em.controls, em.tables, em.measurements, em.flags, em.loglik, em.expectation,
                                        em.prediction, em.used, em.totals)]
    first, rec, mean = logs(), _smoother_state(sm), est.mean.clone()
    em.replay(start)
    em.estep()
    torch.cuda.synchronize()
    assert torch.equal(est.mean, mean)
    assert all(torch.equal(a, b) for a, b in zip(_smoother_state(sm), rec))
    assert all(torch.equal(a, b) for a, b in zip(logs(), first))
    _close(em, sm, est, env)


@pytest.mark.gpu
def test_set_noise_is_staged_until_the_next_reset():
    """The new settings take effect at the next reset, and so does the smoother's deterministic-state mask:
    state 5 gets p0_std = q_std = 0, so after the reset it passes through the
    backward pass, and the smoother equals that of an estimator created with the new values."""
    from glgym.estimation import DEFAULT_Q_STD, DEFAULT_R_STD, DeviceStateEstimator, DeviceStateSmoother
    B = 6
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 5)
    p0, q, r = _p0(), 2 * np.array(DEFAULT_Q_STD), 0.5 * np.array(DEFAULT_R_STD)
    p0[5] = q[5] = 0.0
    est, sm, em = _trio(env, 8)
    ref = DeviceStateEstimator(env, p0_std=p0, q_std=q, r_std=r)
    ref_sm = DeviceStateSmoother(ref, 8)
    est.reset()
    est.set_noise(p0_std=p0, q_std=q, r_std=r)
    assert np.array_equal(est.q_std, DEFAULT_Q_STD)
    env.step_rule_based_tensor()
    est.update(None)
    est.reset()
    ref.reset()
    assert np.array_equal(est.q_std, q) and np.array_equal(est.r_std, r)
    gen = torch.Generator(device="cuda").manual_seed(10)
    for t in range(5):
        env.step_rule_based_tensor()
        y = _noisy(est, gen)
        est.update(y)
        ref.update(y)
        torch.cuda.synchronize()
        for a in ("mean", "cov", "innovation", "status"):
            assert torch.equal(getattr(est, a), getattr(ref, a)), (t, a)
    got, want = _smoother_state(sm), _smoother_state(ref_sm)
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    mean, gain = got[0].cpu().numpy(), got[2].cpu().numpy()
    assert not gain[..., 5, :].any() and not gain[..., :, 5].any() and gain[:-1].any()
    assert np.array_equal(mean[..., 5], sm.filtered_mean.cpu().numpy()[..., 5])
    _close(em, sm, ref_sm, est, ref, env)


@pytest.mark.gpu
def test_estep_refuses_after_the_weather_bank_is_replaced():
    from glgym import _lib
    B = 4
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 5)
    est, sm, em = _trio(env, 6)
    est.reset()
    for _ in range(3):
        env.step_rule_based_tensor()
        est.update(est.measurements())
    em.estep()
    env._lib.glg_set_weather(env._h, env.weather_tables.ctypes.data, env.weather_tables.shape[0], env.weather_tables.shape[1],
                             env.table_start_days.ctypes.data)
    with pytest.raises(_lib.GlgError, match="weather bank was replaced"):
        em.estep()
    _close(em, sm, est, env)


@pytest.mark.gpu
def test_em_recovers_a_known_q_and_r():
    """B = 128, uncertainty_scale 0, rule-based, 192 steps; w ~ N(0, q_true^2) added to the state after each step and
    y = h7(x) + v, v ~ N(0, r_true^2).  EM from 4 q_true and 4 r_true.  Asserted: the first two iterations raise the filter's
    log-likelihood and every measured r_std ends within 20 % of r_true.  The filter's S leaves Q out (the points are not redrawn
    after adding Q), so its log-likelihood is not the one EM's M-step for Q maximises: the later values and the fitted q are
    printed and reported in DESIGN.md, not asserted."""
    from glgym.estimation import DEFAULT_Q_STD, DEFAULT_R_STD, DeviceStateEstimator, DeviceStateSmoother, DeviceNoiseEM
    B, steps = 128, 192
    env = _env(B, uncertainty_scale=0.0, auto_reset=False)
    _warm(env, 0)
    q_true = 0.5 * np.array(DEFAULT_Q_STD)
    q_true[27] = 0.0
    r_true = np.array(DEFAULT_R_STD)
    est = DeviceStateEstimator(env, q_std=4 * q_true, r_std=4 * r_true)
    sm = DeviceStateSmoother(est, steps + 1)
    em = DeviceNoiseEM(sm)
    start = env.state_dict()
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(12)
    qt, rt = torch.as_tensor(q_true, device="cuda"), torch.as_tensor(r_true, device="cuda")
    for _ in range(steps):
        env.step_rule_based_tensor()
        w = torch.randn(28, B, device="cuda", dtype=torch.float64, generator=gen) * qt[:, None]
        x = env.state_t.to(torch.float64) + w
        env.set_state(x=x.T.cpu().numpy())
        y = torch.as_tensor(h7(x.T.cpu().numpy()), device="cuda") + torch.randn(B, 7, device="cuda", dtype=torch.float64,
                                                                                 generator=gen) * rt
        est.update(y)
    hist = em.fit(start, 10)
    last = em.estimate()
    lls = [h.loglik for h in hist]
    print("log-likelihood per iteration:", np.array2string(np.array(lls + [last.loglik]), precision=6))
    print("fitted r_std:", np.array2string(last.r_std, precision=4), "true:", r_true)
    print("fitted q_std / q_true:", np.array2string(last.q_std / np.where(q_true > 0, q_true, 1), precision=3))
    assert lls[1] > lls[0] and lls[2] > lls[1], lls
    assert np.all(np.abs(last.r_std / r_true - 1) <= 0.2), last.r_std / r_true
    _close(em, sm, est, env)
