"""State estimation (csrc/glg_est.cuh, glgym.estimation.DeviceStateEstimator): the unscented Kalman filter against a numpy
restatement of its contract (include/glgym.h), the restatement against a textbook Kalman filter, the propagated sigma points against
glg_evalf_batch_ex, the covariance propagation against glg_linearize, and the output-feedback planner against glg_plan_run."""
import ctypes as C
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

N_X = 28
SHORT2 = dict(season_length=7 / 96.0, start_train_day=0, end_train_day=1)  # N = 7, two weather tables
ROOT_PAIRS = ((2, 3), (2, 7), (7, 3), (2, 20), (20, 3), (3, 5), (2, 8), (9, 2), (19, 2))  # |dT|^0.66 cusps (test_gpu_linearize)


# ---- numpy restatement of the filter contract --------------------------------------------------------------------------------
def ukf_weights(alpha=1.0, beta=2.0, kappa=0.0, n=N_X):
    npl = alpha * alpha * (n + kappa)
    lam = npl - n
    wm = np.full(2 * n + 1, 1.0 / (2.0 * npl))
    wc = wm.copy()
    wm[0] = lam / npl
    wc[0] = wm[0] + 1.0 - alpha * alpha + beta
    return wm, wc, np.sqrt(npl)


def chol_rule(P):
    """P = L L^T column by column; column j is zero where d <= 1e-12 P[j][j]."""
    n = len(P)
    L = np.zeros_like(P)
    for j in range(n):
        s = 0.0
        for k in range(j):
            s += L[j, k] * L[j, k]
        d = P[j, j] - s
        if d <= 1e-12 * P[j, j]:
            continue
        L[j, j] = np.sqrt(d)
        for i in range(j + 1, n):
            s = 0.0
            for k in range(j):
                s += L[i, k] * L[j, k]
            L[i, j] = (P[i, j] - s) / L[j, j]
    return L


def sigma_points(x, P, gamma):
    L = chol_rule(P)
    return np.concatenate([x[None], x[None] + gamma * L.T, x[None] - gamma * L.T])  # [2n+1][n]


def ut_predict(chi, wm, wc, q_std):
    xbar = (wm[:, None] * chi).sum(0)
    D = chi - xbar
    Pm = (wc[:, None, None] * (D[:, :, None] * D[:, None, :])).sum(0) + np.diag(np.asarray(q_std) ** 2)
    return xbar, Pm


def ut_update(chi, xbar, Pm, Y, y, r_std, wm, wc):
    """Y [2n+1][m] measurement points of the measured entries, y [m], r_std [m].  Returns (x, P, innovation)."""
    D = chi - xbar
    ybar = (wm[:, None] * Y).sum(0)
    dY = Y - ybar
    S = (wc[:, None, None] * (dY[:, :, None] * dY[:, None, :])).sum(0) + np.diag(np.asarray(r_std) ** 2)
    Cx = (wc[:, None, None] * (D[:, :, None] * dY[:, None, :])).sum(0)
    K = np.linalg.solve(S, Cx.T).T
    v = y - ybar
    P = Pm - K @ S @ K.T
    return xbar + K @ v, 0.5 * (P + P.T), v


def h7(x):
    """The 7 measurement entries of states x [..., 28] (glg_obs_state7)."""
    x = np.asarray(x)
    t = x[..., 2]
    ppm = 1e6 * 8.3144598 * (t + 273.15) * (x[..., 0] * 1e-6) / (101325 * 44.01e-3)
    rh = np.clip(100 * x[..., 15] / (610.78 * np.exp(17.2694 * t / (t + 238.3))), 0.0, 100.0)
    return np.stack([ppm, t, rh, x[..., 9], x[..., 21], x[..., 25], x[..., 26]], -1)


def scaled_err(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


# ---- CPU tier ------------------------------------------------------------------------------------------------------------
def test_estimation_entry_points_exported_and_reject_null():
    from glgym import _lib
    lib = _lib.load()
    cfg = _lib.GlgEstConfig()
    out = C.c_void_p()
    assert lib.glg_est_create(None, C.byref(cfg), C.byref(out)) == _lib.GLG_ERR_ARG and not out
    assert lib.glg_est_reset(None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_est_update(None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_plan_run_from(None, None, None, None) == _lib.GLG_ERR_ARG
    for view in ("mean", "cov", "innovation", "sigma", "status"):
        assert getattr(lib, f"glg_est_{view}_dev")(None) is None
    lib.glg_est_destroy(None)
    assert C.sizeof(_lib.GlgEstConfig) == 536


@pytest.mark.parametrize("kw, match", [
    (dict(p0_std=[-1.0] + [1.0] * 27), "p0_std"),
    (dict(q_std=[np.nan] + [1.0] * 27), "q_std"),
    (dict(r_std=[np.inf] + [1.0] * 6), "r_std"),
    (dict(p0_std=[1.0] * 27), "p0_std"),
    (dict(r_std=[20.0, 0.0, 2.0, 0.5, 0.5, 500.0, 10.0]), "r_std must be > 0"),
    (dict(alpha=1e-3, kappa=-28.0), "n \\+ lambda"),
    (dict(alpha=0.0), "alpha"),
    (dict(beta=-1.0), "beta"),
    (dict(measured=[]), "at least one"),
    (dict(measured=["temp_air", "temp_air"]), "each once"),
    (dict(measured=["leaf_temp"]), "unknown measurement"),
    (dict(measured=[7]), "indices 0..6"),
])
def test_estimator_arguments_are_validated_before_anything_is_created(kw, match):
    from glgym.estimation import DeviceStateEstimator
    env = types.SimpleNamespace(num_envs=4)  # validation reads num_envs only; a real env is never reached
    with pytest.raises(ValueError, match=match):
        DeviceStateEstimator(env, **kw)


def test_estimator_rejects_more_sigma_points_than_the_step_kernels_were_run_at():
    from glgym.estimation import DeviceStateEstimator
    with pytest.raises(ValueError, match="sigma points"):
        DeviceStateEstimator(types.SimpleNamespace(num_envs=4194304 // 57 + 1))
    r = np.array([20.0, 0.0, 2.0, 0.5, 0.5, 500.0, 10.0])  # r_std 0 on an entry that is not measured is fine
    with pytest.raises(ValueError, match="sigma points"):
        DeviceStateEstimator(types.SimpleNamespace(num_envs=10 ** 6), r_std=r, measured=["co2_air"])


@pytest.mark.parametrize("alpha, beta, kappa", [(1.0, 2.0, 0.0), (0.5, 2.0, 1.0), (0.8, 1.0, -2.0)])
def test_restatement_equals_a_textbook_kalman_filter_on_a_linear_gaussian_model(alpha, beta, kappa):
    """For x' = A x and y = H x the unscented transform is exact, so the restated filter must be the Kalman filter.  State 27 has
    zero variance and a deterministic update, and state 5 starts with p0 = 0: both exercise the zero-column Cholesky rule."""
    rng = np.random.default_rng(7)
    n = N_X
    A = np.eye(n) + 0.05 * rng.standard_normal((n, n))
    A[27] = 0.0
    A[27, 27] = 1.0
    H = 0.3 * rng.standard_normal((7, n))
    G = rng.standard_normal((n, n))
    P = G @ G.T / n + 0.1 * np.eye(n)
    P[5, :] = P[:, 5] = 0.0
    P[27, :] = P[:, 27] = 0.0
    x = rng.standard_normal(n)
    q = np.abs(rng.standard_normal(n)) * 0.1
    q[27] = 0.0
    wm, wc, g = ukf_weights(alpha, beta, kappa)
    chi = sigma_points(x, P, g)
    L = chol_rule(P)
    assert np.all(L[:, 27] == 0) and np.all(L[:, 5] == 0)
    assert np.allclose(L @ L.T, P, rtol=0, atol=1e-14)
    chi_p = chi @ A.T
    xbar, Pm = ut_predict(chi_p, wm, wc, q)
    xkf, Pkf = A @ x, A @ P @ A.T + np.diag(q ** 2)
    assert scaled_err(xbar, xkf) <= 1e-12 and scaled_err(Pm, Pkf) <= 1e-12
    # The measurement points are the propagated points without a redraw after adding Q, so Q enters P- but not S and C: the
    # update is the Kalman filter's when the prediction adds no process noise.
    xbar, Pm = ut_predict(chi_p, wm, wc, np.zeros(n))
    xkf, Pkf = A @ x, A @ P @ A.T
    for idx in ([0, 1, 2, 3, 4, 5, 6], [0, 1, 2], [1]):
        Hm = H[idx]
        r = np.full(len(idx), 0.3)
        y = Hm @ xkf + rng.standard_normal(len(idx))
        xu, Pu, v = ut_update(chi_p, xbar, Pm, chi_p @ Hm.T, y, r, wm, wc)
        S = Hm @ Pkf @ Hm.T + np.diag(r ** 2)
        K = Pkf @ Hm.T @ np.linalg.inv(S)
        Pt = (np.eye(n) - K @ Hm) @ Pkf
        assert scaled_err(xu, xkf + K @ (y - Hm @ xkf)) <= 1e-12
        assert scaled_err(Pu, 0.5 * (Pt + Pt.T)) <= 1e-12
        assert scaled_err(v, y - Hm @ xkf) <= 1e-12


# ---- GPU tier ------------------------------------------------------------------------------------------------------------
def _env(B, **kw):
    from glgym.vec_env import GreenLightVecEnv
    base = dict(seed=3)
    base.update(kw)
    return GreenLightVecEnv(B, **base)


def _warm(env, steps, seed=0):
    """Reset onto distinct weather tables and run the rule-based controller for a while, so the envs hold distinct states."""
    B = env.num_envs
    n_tab = env.weather_tables.shape[0]
    env.reset_tensor(table_ids=(torch.arange(B, device="cuda", dtype=torch.int32) * 7) % n_tab)
    for _ in range(steps):
        env.step_rule_based_tensor()
    torch.cuda.synchronize()


def _p0(scale=1.0):
    from glgym.estimation import DEFAULT_P0_STD
    p0 = np.array(DEFAULT_P0_STD) * scale
    p0[11] = 0.0  # a second zero column besides x27's
    return p0


def _step_and_update(env, est, y=None):
    """One rule-based step of the env and the estimator's update; returns the pre-update mean and covariance (numpy) and the
    controls and weather rows of the step."""
    m0, P0 = est.mean.cpu().numpy().copy(), est.cov.cpu().numpy().copy()
    k0 = env.timestep_t.cpu().numpy().copy()
    tb = env.table_t.cpu().numpy().copy()
    env.step_rule_based_tensor()
    est.update(y)
    torch.cuda.synchronize()
    W = env.weather_tables
    rows = np.stack([W[tb[b], min(k0[b], W.shape[1] - env.Np - 1)] for b in range(env.num_envs)])
    u = env.controls_t.T.cpu().numpy().copy()
    return m0, P0, u, rows


@pytest.mark.gpu
@pytest.mark.parametrize("integrator", ["fixed", "graded"])
def test_sigma_points_are_one_nominal_step_of_the_numpy_sigma_points(integrator):
    from glgym.estimation import DeviceStateEstimator
    from glgym.model import GreenLight
    B = 4
    env = _env(B, integrator=integrator, uncertainty_scale=0.1)
    _warm(env, 20)
    est = DeviceStateEstimator(env, p0_std=_p0())
    est.reset()
    wm, wc, g = ukf_weights()
    m = GreenLight(integrator=integrator, n_sub=env.n_sub)
    p64 = np.ascontiguousarray(env.p, dtype=np.float64)
    for step in range(3):
        m0, P0, u, rows = _step_and_update(env, est, est.measurements())
        assert np.all(est.status.cpu().numpy() == 0)
        chi = np.stack([sigma_points(m0[b], P0[b], g) for b in range(B)])  # [B][57][28]
        xs = np.ascontiguousarray(chi.reshape(-1, 28))
        ref = m.evalF_batch(xs, np.repeat(u, 57, 0), np.repeat(rows, 57, 0), p64).cpu().numpy().reshape(B, 57, 28)
        got = est.sigma.permute(1, 2, 0).cpu().numpy()
        err = np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-3))
        assert err <= 1e-9, (step, err)
    est.close()
    env.close()


def _restated_update(est, m0, P0, y, idx, r_std):
    """numpy x, P and innovation of one update from the device's propagated sigma points."""
    wm, wc, _ = ukf_weights()
    chi = est.sigma.permute(1, 2, 0).cpu().numpy()
    out = []
    for b in range(chi.shape[0]):
        xbar, Pm = ut_predict(chi[b], wm, wc, est.q_std)
        if y is None:
            out.append((xbar, Pm, np.zeros(7)))
            continue
        x, P, v = ut_update(chi[b], xbar, Pm, h7(chi[b])[:, idx], y[b, idx], r_std[idx], wm, wc)
        vv = np.zeros(7)
        vv[idx] = v
        out.append((x, P, vv))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("measured", [None, ["co2_air", "temp_air", "rh_air"], ["cFruit"], "predict"])
def test_predict_and_update_equal_the_restatement(measured):
    from glgym.estimation import DeviceStateEstimator, MEASUREMENT_NAMES
    B = 6
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 30)
    meas = None if measured == "predict" else measured
    est = DeviceStateEstimator(env, p0_std=_p0(), measured=meas)
    est.reset()
    idx = np.array([MEASUREMENT_NAMES.index(n) for n in est.measured])
    gen = torch.Generator(device="cuda").manual_seed(1)
    for step in range(4):
        y = None
        if measured != "predict":
            y = est.measurements() + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen) * torch.as_tensor(
                est.r_std, device="cuda")
        m0, P0, _, _ = _step_and_update(env, est, y)
        assert np.all(est.status.cpu().numpy() == 0)
        ref = _restated_update(est, m0, P0, None if y is None else y.cpu().numpy(), idx, est.r_std)
        mean, cov, inn = est.mean.cpu().numpy(), est.cov.cpu().numpy(), est.innovation.cpu().numpy()
        for b in range(B):
            x, P, v = ref[b]
            assert scaled_err(mean[b], x) <= 1e-12, (step, b)
            assert scaled_err(cov[b], P) <= 1e-12, (step, b)
            assert np.array_equal(cov[b], cov[b].T)
            assert np.max(np.abs(inn[b] - v)) <= 1e-12 * max(np.max(np.abs(v)), 1.0), (step, b)
            assert abs(cov[b][27, 27]) <= 1e-24  # the day counter: deterministic up to the rounding of the weighted mean
    est.close()
    env.close()


@pytest.mark.gpu
def test_small_spread_covariance_propagation_matches_the_linearisation():
    """With p0 ~ 1e-6 |x| and q = 0 the predicted covariance is A P0 A^T to first order, A = glg_linearize's step Jacobian.
    Measured 1.07e-10 relative (Frobenius) on its first run; the tolerance is 1e-8."""
    from glgym.estimation import DeviceStateEstimator
    B = 8
    env = _env(B)
    _warm(env, 40)
    u = env.rule_controls_tensor().clone()
    x = env.state_t.T.cpu().numpy()
    ok = [b for b in range(B) if min(abs(x[b, a] - x[b, c]) for a, c in ROOT_PAIRS) > 0.05]
    assert len(ok) >= 4
    _, A, _ = env.linearize_tensor(u)
    A = A.cpu().numpy()
    p0 = 1e-6 * np.maximum(np.abs(x), 1e-3)
    p0[:, 27] = 0.0
    est = DeviceStateEstimator(env, p0_std=np.ones(28), q_std=np.zeros(28))
    est.reset()
    # the covariance is per env: write diag(p0_b^2) directly into the estimator's buffer
    est.cov.zero_()
    est.cov[:, range(28), range(28)] = torch.as_tensor(p0 ** 2, device="cuda")
    env.step_raw_control_tensor(u)
    est.update(None)
    Pm = est.cov.cpu().numpy()
    errs = []
    for b in ok:
        ref = A[b] @ np.diag(p0[b] ** 2) @ A[b].T
        errs.append(np.linalg.norm(Pm[b] - ref) / np.linalg.norm(ref))
    print("small-spread relative Frobenius error:", max(errs))
    assert max(errs) <= 1e-8, errs  # 1.07e-10 on the first run (one B200)
    est.close()
    env.close()


@pytest.mark.gpu
def test_auto_reset_restarts_the_filter():
    from glgym.estimation import DeviceStateEstimator
    B = 6
    env = _env(B, base_env_params=SHORT2)
    env.reset_tensor(table_ids=torch.arange(B, device="cuda", dtype=torch.int32) % 2)
    env.step_rule_based_tensor()
    env.step_rule_based_tensor()
    k = env.get_state()[2]
    k[[1, 4]] = 0  # these envs finish four steps after the others
    env.set_state(timestep=k)
    est = DeviceStateEstimator(env, p0_std=_p0())
    est.reset()
    p0sq = np.diag(est.p0_std ** 2)
    seen = 0
    for _ in range(12):
        m0, P0 = est.mean.cpu().numpy().copy(), est.cov.cpu().numpy().copy()
        env.step_rule_based_tensor()
        est.update(est.measurements())
        torch.cuda.synchronize()
        done, st = env.done_t.cpu().numpy().astype(bool), est.status.cpu().numpy()
        x = env.state_t.T.cpu().numpy()
        mean, cov = est.mean.cpu().numpy(), est.cov.cpu().numpy()
        for b in range(B):
            if done[b]:
                seen += 1
                assert st[b] == 4 and np.array_equal(mean[b], x[b]) and np.array_equal(cov[b], p0sq)
            else:
                assert st[b] == 0 and not np.array_equal(mean[b], m0[b])
    assert seen >= 4
    est.close()
    env.close()


@pytest.mark.gpu
def test_non_finite_sigma_point_and_out_of_step_env_are_flagged():
    from glgym.estimation import DeviceStateEstimator
    B = 4
    env = _env(B)
    _warm(env, 10)
    est = DeviceStateEstimator(env, p0_std=_p0())
    x0 = env.state_t.T.clone()
    x0[2, 5] = float("nan")
    est.reset(x0)
    m0, P0 = est.mean.cpu().numpy().copy(), est.cov.cpu().numpy().copy()
    env.step_rule_based_tensor()
    est.update(est.measurements())
    torch.cuda.synchronize()
    st = est.status.cpu().numpy()
    assert st.tolist() == [0, 0, 1, 0]
    mean, cov = est.mean.cpu().numpy(), est.cov.cpu().numpy()
    assert np.array_equal(mean[2], m0[2], equal_nan=True) and np.array_equal(cov[2], P0[2])
    assert np.all(np.isfinite(mean[[0, 1, 3]]))
    # an extra env step between two updates
    m1, P1 = mean.copy(), cov.copy()
    env.step_rule_based_tensor()
    env.step_rule_based_tensor()
    est.update(est.measurements())
    torch.cuda.synchronize()
    assert np.all(est.status.cpu().numpy() == 8)
    assert np.array_equal(est.mean.cpu().numpy(), m1, equal_nan=True) and np.array_equal(est.cov.cpu().numpy(), P1)
    # back in step: the step counter was recorded
    env.step_rule_based_tensor()
    est.update(est.measurements())
    torch.cuda.synchronize()
    assert est.status.cpu().numpy().tolist() == [0, 0, 1, 0]
    est.close()
    env.close()


@pytest.mark.gpu
def test_determinism_fences_and_fp32():
    from glgym import _lib
    from glgym.estimation import DeviceStateEstimator
    B = 8
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 5)
    e1, e2 = DeviceStateEstimator(env), DeviceStateEstimator(env)
    with pytest.raises(_lib.GlgError, match="not been reset"):
        e1.update(None)
    e1.reset()
    e2.reset()
    gen = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(5):
        env.step_rule_based_tensor()
        y = e1.measurements() + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen)
        e1.update(y)
        e2.update(y)
        torch.cuda.synchronize()
        for a in ("mean", "cov", "innovation", "status"):
            assert torch.equal(getattr(e1, a), getattr(e2, a)), a
    env._lib.glg_set_weather(env._h, env.weather_tables.ctypes.data, env.weather_tables.shape[0], env.weather_tables.shape[1],
                             env.table_start_days.ctypes.data)
    with pytest.raises(_lib.GlgError, match="weather bank was replaced"):
        e1.update(None)
    with pytest.raises(_lib.GlgError, match="weather bank was replaced"):
        e1.reset()
    e1.close()  # before its env
    env.close()
    e2.close()  # after its env
    env32 = _env(B, precision="fp32", uncertainty_scale=0.1)
    _warm(env32, 5)
    e3 = DeviceStateEstimator(env32)
    e3.reset()
    for _ in range(4):
        env32.step_rule_based_tensor()
        e3.update(e3.measurements())
    torch.cuda.synchronize()
    assert np.all(e3.status.cpu().numpy() == 0)
    assert bool(torch.isfinite(e3.mean).all()) and bool(torch.isfinite(e3.cov).all())
    e3.close()
    env32.close()


def _sigma_ybar(est):
    wm, _, _ = ukf_weights()
    chi = est.sigma.permute(1, 2, 0).cpu().numpy()
    return np.einsum("s,bsm->bm", wm, h7(chi))


@pytest.mark.gpu
def test_filter_tracks_the_observed_quantities_better_than_open_loop():
    """A true env at uncertainty_scale 0.2 under the rule-based controller for two days from a wrong prior.  Over the second day the
    RMS of ybar - y for tAir, RH and CO2 is lower with updates than with predict-only."""
    from glgym.estimation import DeviceStateEstimator
    B, steps = 16, 192
    env = _env(B, uncertainty_scale=0.2)
    _warm(env, 0)
    x0 = env.state_t.T.clone()
    x0[:, 2:15] += 1.5                       # temperatures 1.5 K off
    x0[:, 22:26] *= 1.1                      # crop pools 10 % off
    filt, olp = DeviceStateEstimator(env), DeviceStateEstimator(env)
    filt.reset(x0)
    olp.reset(x0)
    gen = torch.Generator(device="cuda").manual_seed(4)
    rstd = torch.as_tensor(filt.r_std, device="cuda")
    res = {"filt": [], "olp": []}
    truth_err = {"filt": [], "olp": []}
    for t in range(steps):
        env.step_rule_based_tensor()
        y_true = filt.measurements()
        y = y_true + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen) * rstd
        filt.update(y)
        olp.update(None)
        if t >= steps // 2:
            for name, e in (("filt", filt), ("olp", olp)):
                res[name].append(_sigma_ybar(e)[:, :3] - y_true.cpu().numpy()[:, :3])
                truth_err[name].append(e.mean.cpu().numpy() - env.state_t.T.cpu().numpy())
    assert np.all(filt.status.cpu().numpy() == 0)
    rms = {k: np.sqrt(np.mean(np.square(np.stack(v)), axis=(0, 1))) for k, v in res.items()}
    print("RMS of ybar - y (co2, tAir, RH), filter:", rms["filt"], "open loop:", rms["olp"])
    st = {k: np.sqrt(np.mean(np.square(np.stack(v)), axis=(0, 1))) for k, v in truth_err.items()}
    print("per-state RMS of x^ - x, filter:", np.array2string(st["filt"], precision=4), "open loop:",
          np.array2string(st["olp"], precision=4))
    assert np.all(rms["filt"] < rms["olp"]), rms
    assert float(filt.cov[:, 2, 2].max()) <= filt.r_std[1] ** 2
    filt.close()
    olp.close()
    env.close()


@pytest.mark.gpu
def test_plan_from_given_states_is_bit_identical_to_planning_from_the_env():
    from glgym.estimation import DeviceStateEstimator
    from glgym.planning import DevicePlanner
    B, K, H = 4, 16, 4
    env = _env(B, uncertainty_scale=0.2)
    _warm(env, 6)
    p1, p2 = DevicePlanner(env, H, K, 4, 2, seed=5), DevicePlanner(env, H, K, 4, 2, seed=5)
    a1 = p1.plan().clone()
    a2 = p2.plan(env.state_t.T).clone()
    torch.cuda.synchronize()
    assert torch.equal(a1, a2)
    for v in ("mean", "std", "candidates", "returns"):
        assert torch.equal(getattr(p1, v), getattr(p2, v)), v
    # from the estimate: a twin env holding that state plans the same
    est = DeviceStateEstimator(env)
    est.reset()
    for _ in range(3):
        env.step_rule_based_tensor()
        est.update(est.measurements())
    torch.cuda.synchronize()
    twin = _env(B, uncertainty_scale=0.2)
    twin.load_state_dict(env.state_dict())
    twin.set_state(x=est.mean.cpu().numpy())
    p3, p4 = DevicePlanner(env, H, K, 4, 2, seed=9), DevicePlanner(twin, H, K, 4, 2, seed=9)
    a3 = p3.plan(est.mean).clone()
    a4 = p4.plan().clone()
    torch.cuda.synchronize()
    assert torch.equal(a3, a4)
    for v in ("mean", "std", "candidates", "returns"):
        assert torch.equal(getattr(p3, v), getattr(p4, v)), v
    with pytest.raises(ValueError):
        p3.plan(est.mean.float())
    for o in (p1, p2, p3, p4, est):
        o.close()
    env.close()
    twin.close()
