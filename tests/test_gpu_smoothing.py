"""State smoothing (csrc/glg_smooth.cuh, glgym.estimation.DeviceStateSmoother): the unscented RTS smoother against a numpy
restatement of its contract (include/glgym.h), the restatement against a textbook Kalman filter and RTS smoother, the forward record
against the estimator's own outputs, and the estimator's outputs with a smoother against those without one."""
import ctypes as C
import types

import numpy as np
import pytest

from test_gpu_estimation import chol_rule, scaled_err, sigma_points, ukf_weights, ut_predict, ut_update

torch = pytest.importorskip("torch")

N_X = 28
SEGMENT = 1 | 4 | 8  # status bits that start a segment
SHORT2 = dict(season_length=7 / 96.0, start_train_day=0, end_train_day=1)  # N = 7, two weather tables


# ---- numpy restatement of the smoother contract ------------------------------------------------------------------------------
def offsets(P, gamma):
    """chi_i - x^ = +-gamma L[:, i-1] ([2n+1][n]; row 0 is 0), L by the filter's Cholesky rule."""
    L = chol_rule(P)
    return np.concatenate([np.zeros((1, len(P))), gamma * L.T, -gamma * L.T])


def cross_cov(off, chi_p, xbar, wc):
    return (wc[:, None, None] * (off[:, :, None] * (chi_p - xbar)[:, None, :])).sum(0)


def gain_rule(D, Pm, active):
    """G = D P-^-1 by row solves through the zero-column factor of P- with the deterministic rows and columns left out."""
    n = len(Pm)
    Pz = np.where(active[:, None] & active[None, :], Pm, 0.0)
    L = chol_rule(Pz)
    nz = np.diag(L) != 0
    G = np.zeros_like(D)
    for i in np.flatnonzero(active):
        g = D[i].copy()
        for c in range(n):
            g[c] = (g[c] - L[c, :c] @ g[:c]) / L[c, c] if nz[c] else 0.0
        for c in reversed(range(n)):
            g[c] = (g[c] - L[c + 1:, c] @ g[c + 1:]) / L[c, c] if nz[c] else 0.0
        G[i] = g
    return G


def urts(mean, cov, xbar, pm, D, status, active):
    """Smoothed means, covariances and gains of one env's slots [L][...], oldest first."""
    xs, Ps, G = mean.copy(), cov.copy(), np.zeros_like(cov)
    for k in range(len(mean) - 2, -1, -1):
        if status[k + 1] & SEGMENT:
            continue
        G[k] = gain_rule(D[k + 1], pm[k + 1], active)
        xs[k] = mean[k] + G[k] @ (xs[k + 1] - xbar[k + 1])
        P = cov[k] + G[k] @ (Ps[k + 1] - pm[k + 1]) @ G[k].T
        Ps[k] = 0.5 * (P + P.T)
    return xs, Ps, G


# ---- CPU tier ------------------------------------------------------------------------------------------------------------
def test_smoothing_entry_points_exported_and_reject_null():
    from glgym import _lib
    lib = _lib.load()
    out = C.c_void_p()
    assert lib.glg_smooth_create(None, 4, C.byref(out)) == _lib.GLG_ERR_ARG and not out
    assert lib.glg_smooth_run(None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_smooth_length(None) == 0 and lib.glg_smooth_first(None) == 0 and lib.glg_smooth_bytes(None) == 0
    for view in ("mean", "cov", "gain", "filtered_mean", "filtered_cov", "prior_mean", "prior_cov", "cross", "status",
                 "timestep"):
        assert getattr(lib, f"glg_smooth_{view}_dev")(None) is None
    lib.glg_smooth_destroy(None)


@pytest.mark.parametrize("window, exc, match", [(1, ValueError, "window"), (0, ValueError, "window"), (2.5, ValueError, "window"),
                                                (True, ValueError, "window"), ("8", ValueError, "window"),
                                                (8, TypeError, "DeviceStateEstimator")])
def test_smoother_arguments_are_validated_before_anything_is_created(window, exc, match):
    from glgym.estimation import DeviceStateSmoother
    est = types.SimpleNamespace(env=types.SimpleNamespace(num_envs=4))  # never reached: no C object is created
    with pytest.raises(exc, match=match):
        DeviceStateSmoother(est, window)


@pytest.mark.parametrize("alpha, beta, kappa", [(1.0, 2.0, 0.0), (0.5, 2.0, 1.0), (0.8, 1.0, -2.0)])
def test_restated_ukf_and_urts_equal_a_textbook_kalman_filter_and_rts_smoother(alpha, beta, kappa):
    """For x' = A x and y = H x the unscented transform is exact, so the restated filter plus smoother must be the Kalman filter
    plus the RTS smoother.  x27 is deterministic (p0 = q = 0); the filter restarts at step 6 (a segment start).  The UKF's
    measurement points are not redrawn after adding Q, so Q enters P- but not S and C: process noise is added on the
    predict-only steps, and the measured steps add none, where both filters are the textbook one."""
    rng = np.random.default_rng(11)
    n, steps, restart = N_X, 11, 6
    A = np.eye(n) + 0.05 * rng.standard_normal((n, n))
    A[27] = 0.0
    A[27, 27] = 1.0
    H = 0.3 * rng.standard_normal((7, n))
    Gm = rng.standard_normal((n, n))
    P0 = Gm @ Gm.T / n + 0.1 * np.eye(n)
    P0[27, :] = P0[:, 27] = 0.0
    q = np.abs(rng.standard_normal(n)) * 0.1
    q[27] = 0.0
    r = np.full(7, 0.3)
    active = (np.diag(P0) > 0) | (q > 0)
    assert not active[27] and active[:27].all()
    wm, wc, g = ukf_weights(alpha, beta, kappa)
    x = rng.standard_normal(n)
    rec = {k: [] for k in ("mean", "cov", "xbar", "pm", "D", "status")}
    tb = {k: [] for k in ("mean", "cov", "xp", "Pp", "C")}

    def push(d, **kw):
        for k, v in kw.items():
            d[k].append(v)

    push(rec, mean=x, cov=P0, xbar=np.zeros(n), pm=np.zeros((n, n)), D=np.zeros((n, n)), status=0)
    push(tb, mean=x, cov=P0, xp=np.zeros(n), Pp=np.zeros((n, n)), C=np.zeros((n, n)))
    xu, Pu, xk, Pk = x, P0, x, P0
    for k in range(1, steps):
        if k == restart:
            xu = xk = rng.standard_normal(n)
            Pu = Pk = P0
            push(rec, mean=xu, cov=Pu, xbar=np.zeros(n), pm=np.zeros((n, n)), D=np.zeros((n, n)), status=4)
            push(tb, mean=xk, cov=Pk, xp=np.zeros(n), Pp=np.zeros((n, n)), C=np.zeros((n, n)))
            continue
        measured = k % 2 == 1
        qk = np.zeros(n) if measured else q
        # restated UKF with the forward record
        chi = sigma_points(xu, Pu, g)
        chi_p = chi @ A.T
        xbar, Pm = ut_predict(chi_p, wm, wc, qk)
        D = cross_cov(offsets(Pu, g), chi_p, xbar, wc)
        # textbook Kalman filter
        xp, Pp = A @ xk, A @ Pk @ A.T + np.diag(qk ** 2)
        Ck = Pk @ A.T
        if measured:
            y = H @ xp + rng.standard_normal(7)
            xu, Pu, _ = ut_update(chi_p, xbar, Pm, chi_p @ H.T, y, r, wm, wc)
            S = H @ Pp @ H.T + np.diag(r ** 2)
            K = Pp @ H.T @ np.linalg.inv(S)
            xk = xp + K @ (y - H @ xp)
            Pt = (np.eye(n) - K @ H) @ Pp
            Pk = 0.5 * (Pt + Pt.T)
        else:
            xu, Pu, xk, Pk = xbar, Pm, xp, Pp
        push(rec, mean=xu, cov=Pu, xbar=xbar, pm=Pm, D=D, status=0)
        push(tb, mean=xk, cov=Pk, xp=xp, Pp=Pp, C=Ck)
        assert scaled_err(xbar, xp) <= 1e-12 and scaled_err(Pm, Pp) <= 1e-12 and scaled_err(D, Ck) <= 1e-12
        assert scaled_err(xu, xk) <= 1e-12 and scaled_err(Pu, Pk) <= 1e-12
    rec = {k: np.array(v) for k, v in rec.items()}
    xs, Ps, G = urts(rec["mean"], rec["cov"], rec["xbar"], rec["pm"], rec["D"], rec["status"], active)
    # textbook RTS on each segment, over the non-deterministic states
    a = np.flatnonzero(active)
    for lo, hi in ((0, restart), (restart, steps)):
        xt, Pt = tb["mean"][hi - 1], tb["cov"][hi - 1]
        assert np.array_equal(xs[hi - 1], rec["mean"][hi - 1]) and np.array_equal(Ps[hi - 1], rec["cov"][hi - 1])
        assert not G[hi - 1].any()
        for k in range(hi - 2, lo - 1, -1):
            Gt = np.zeros((n, n))
            Gt[np.ix_(a, a)] = tb["C"][k + 1][np.ix_(a, a)] @ np.linalg.inv(tb["Pp"][k + 1][np.ix_(a, a)])
            xt = tb["mean"][k] + Gt @ (xt - tb["xp"][k + 1])
            Pt = tb["cov"][k] + Gt @ (Pt - tb["Pp"][k + 1]) @ Gt.T
            assert scaled_err(G[k], Gt) <= 1e-12, k
            assert scaled_err(xs[k], xt) <= 1e-12, k
            assert scaled_err(Ps[k], Pt) <= 1e-12, k
    assert np.array_equal(xs[:, 27], rec["mean"][:, 27]) and np.array_equal(Ps[:, 27], rec["cov"][:, 27])
    assert not G[:, 27].any() and not G[:, :, 27].any()


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


def _p0():
    from glgym.estimation import DEFAULT_P0_STD
    p0 = np.array(DEFAULT_P0_STD)
    p0[11] = 0.0  # a zero column besides x27's in the first factor; q_std[11] > 0 makes it active
    return p0


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


def _record(sm):
    return {k: getattr(sm, k).cpu().numpy() for k in ("filtered_mean", "filtered_cov", "prior_mean", "prior_cov", "cross_cov",
                                                      "status", "timestep")}


def _active(est):
    return (est.p0_std > 0) | (est.q_std > 0)


def _restate(rec, b, active, lo=0, hi=None):
    sl = slice(lo, hi)
    return urts(rec["filtered_mean"][sl, b], rec["filtered_cov"][sl, b], rec["prior_mean"][sl, b], rec["prior_cov"][sl, b],
                rec["cross_cov"][sl, b], rec["status"][sl, b], active)


def _check_against_restatement(sm, s, segments_on_their_own=False):
    """The smoothed output of every env against the restatement fed with the recorded forward quantities; the last slot of
    each segment is the filtered estimate bit for bit, with gain 0."""
    rec = _record(sm)
    mean, cov, gain = (v.cpu().numpy() for v in s)
    active = _active(sm.est)
    n = len(mean)
    for b in range(mean.shape[1]):
        starts = [k for k in range(1, n) if rec["status"][k, b] & SEGMENT] if segments_on_their_own else []
        for lo, hi in zip([0] + starts, starts + [n]):
            xs, Ps, G = _restate(rec, b, active, lo, hi)
            for k in range(lo, hi):
                assert scaled_err(mean[k, b], xs[k - lo]) <= 1e-12, (b, k)
                assert scaled_err(cov[k, b], Ps[k - lo]) <= 1e-12, (b, k)
                if not G[k - lo].any():
                    assert not gain[k, b].any(), (b, k)
                    continue
                # G = D P-^-1 carries P-'s condition number: its rounding differs from the restatement's by up to 3.1e-11
                # scaled (first run, one B200), while G P- = D holds to 3.4e-15 in units of the states' standard deviations
                assert scaled_err(gain[k, b], G[k - lo]) <= 1e-9, (b, k)
                Pm, D, P = rec["prior_cov"][k + 1, b], rec["cross_cov"][k + 1, b], rec["filtered_cov"][k, b]
                a, r = np.flatnonzero(active), np.flatnonzero(active & (np.diag(P) > 0))  # a row of P may be 0 (p0_std 0)
                sd = np.sqrt(np.diag(Pm)[a])[None, :] * np.sqrt(np.diag(P)[r])[:, None]
                assert np.max(np.abs((gain[k, b] @ Pm - D)[np.ix_(r, a)]) / sd) <= 1e-12, (b, k)
            assert np.array_equal(mean[hi - 1, b], rec["filtered_mean"][hi - 1, b])
            assert np.array_equal(cov[hi - 1, b], rec["filtered_cov"][hi - 1, b])
            assert not gain[hi - 1, b].any()
        assert np.array_equal(cov[:, b], np.swapaxes(cov[:, b], -1, -2))
    return rec


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_recording_leaves_the_estimator_bit_identical(precision):
    """Two estimators on one env, one with a smoother, over a trajectory where envs finish under auto-reset."""
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B = 6
    env = _short_env(B, precision=precision)
    e1, e2 = DeviceStateEstimator(env, p0_std=_p0()), DeviceStateEstimator(env, p0_std=_p0())
    sm = DeviceStateSmoother(e1, 8)
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
        assert torch.equal(sm.filtered_mean[-1], e1.mean) and torch.equal(sm.filtered_cov[-1], e1.cov)
        assert torch.equal(sm.status[-1], e1.status) and torch.equal(sm.timestep[-1], env.timestep_t.to(torch.int32))
    assert reinit >= 4
    assert sm.length == 8
    sm.close()
    e1.close()
    e2.close()
    env.close()


@pytest.mark.gpu
def test_record_after_a_predict_only_update():
    """P- and xbar are the estimator's output of a predict-only update, bit for bit; D matches the restatement from the shadow
    handle's propagated points and the factor of the recorded previous P."""
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B = 4
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 20)
    est = DeviceStateEstimator(env, p0_std=_p0())
    sm = DeviceStateSmoother(est, 4)
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(6)
    env.step_rule_based_tensor()
    est.update(_noisy(est, gen))
    env.step_rule_based_tensor()
    est.update(None)
    torch.cuda.synchronize()
    rec = _record(sm)
    assert sm.length == 3 and rec["status"].tolist() == [[0] * B] * 3
    assert np.array_equal(rec["prior_cov"][-1], est.cov.cpu().numpy())
    assert np.array_equal(rec["prior_mean"][-1], est.mean.cpu().numpy())
    assert not rec["prior_cov"][0].any() and not rec["cross_cov"][0].any() and not rec["prior_mean"][0].any()
    wm, wc, g = ukf_weights()
    chi_p = est.sigma.permute(1, 2, 0).cpu().numpy()
    for b in range(B):
        D = cross_cov(offsets(rec["filtered_cov"][-2, b], g), chi_p[b], rec["prior_mean"][-1, b], wc)
        assert scaled_err(rec["cross_cov"][-1, b], D) <= 1e-12, b
        xbar, Pm = ut_predict(chi_p[b], wm, wc, est.q_std)
        assert scaled_err(rec["prior_mean"][-1, b], xbar) <= 1e-12 and scaled_err(rec["prior_cov"][-1, b], Pm) <= 1e-12
    sm.close()
    est.close()
    env.close()


@pytest.mark.gpu
def test_smoothed_estimates_equal_the_restatement_and_x27_passes_through():
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B = 6
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 30)
    est = DeviceStateEstimator(env, p0_std=_p0())
    sm = DeviceStateSmoother(est, 16)
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(7)
    for t in range(10):
        env.step_rule_based_tensor()
        est.update(None if t == 4 else _noisy(est, gen))
    s = sm.smooth()
    torch.cuda.synchronize()
    assert s.mean.shape == (11, B, 28) and s.cov.shape == (11, B, 28, 28) and s.gain.shape == (11, B, 28, 28)
    rec = _check_against_restatement(sm, s)
    assert np.all(rec["status"] == 0)
    mean, cov, gain = (v.cpu().numpy() for v in s)
    assert np.any(gain[:-1] != 0)
    assert np.array_equal(mean[..., 27], rec["filtered_mean"][..., 27])
    assert np.array_equal(cov[..., 27, :], rec["filtered_cov"][..., 27, :])
    assert np.array_equal(cov[..., :, 27], rec["filtered_cov"][..., :, 27])
    assert not gain[..., 27, :].any() and not gain[..., :, 27].any()
    # the history is left intact: a second run over a cleared output gives the same output
    first = [v.clone() for v in s]
    for v in s:
        v.fill_(float("nan"))
    again = sm.smooth()
    assert all(torch.equal(a, b) for a, b in zip(again, first))
    sm.close()
    est.close()
    env.close()


@pytest.mark.gpu
def test_auto_reset_and_out_of_step_split_segments():
    """Envs finish under auto-reset inside the window (status 4), then every env is stepped twice between two updates
    (status 8): the smoothed values equal smoothing each segment on its own."""
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B = 6
    env = _short_env(B)
    est = DeviceStateEstimator(env, p0_std=_p0())
    sm = DeviceStateSmoother(est, 16)
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(8)
    for t in range(12):
        env.step_rule_based_tensor()
        if t == 8:
            env.step_rule_based_tensor()
        est.update(_noisy(est, gen))
    s = sm.smooth()
    torch.cuda.synchronize()
    rec = _check_against_restatement(sm, s, segments_on_their_own=True)
    st = rec["status"]
    assert np.all(st[9] == 8) and (st == 4).sum() >= 4
    gain = s.gain.cpu().numpy()
    for b in range(B):
        for k in range(1, len(st)):
            if st[k, b] & SEGMENT:
                assert not gain[k - 1, b].any(), (b, k)
    sm.close()
    est.close()
    env.close()


@pytest.mark.gpu
def test_ring_wrap_keeps_the_last_window_estimates_oldest_first():
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B, W = 4, 5
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 10)
    est = DeviceStateEstimator(env, p0_std=_p0())
    sm = DeviceStateSmoother(est, W)
    est.reset()
    hist = [(est.mean.cpu().numpy().copy(), est.cov.cpu().numpy().copy(), env.timestep_t.cpu().numpy().copy())]
    gen = torch.Generator(device="cuda").manual_seed(9)
    for t in range(12):
        env.step_rule_based_tensor()
        est.update(_noisy(est, gen))
        torch.cuda.synchronize()
        hist.append((est.mean.cpu().numpy().copy(), est.cov.cpu().numpy().copy(), env.timestep_t.cpu().numpy().copy()))
        assert sm.length == min(t + 2, W)
    s = sm.smooth()
    torch.cuda.synchronize()
    rec = _check_against_restatement(sm, s)
    assert np.array_equal(rec["filtered_mean"], np.stack([h[0] for h in hist[-W:]]))
    assert np.array_equal(rec["filtered_cov"], np.stack([h[1] for h in hist[-W:]]))
    assert np.array_equal(rec["timestep"], np.stack([h[2] for h in hist[-W:]]))
    # per env-slot: x^, xbar, xs (28 doubles each), P, P-, D, Ps, G (784 each), status and timestep; per env: the factor
    assert sm.bytes == W * B * ((3 * 28 + 5 * 28 * 28) * 8 + 1 + 4) + B * 28 * 28 * 8
    sm.close()
    est.close()
    env.close()


@pytest.mark.gpu
def test_determinism_and_fences():
    from glgym import _lib
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B = 6
    env = _env(B, uncertainty_scale=0.1)
    _warm(env, 5)
    e1, e2 = DeviceStateEstimator(env), DeviceStateEstimator(env)
    out = C.c_void_p()
    assert env._lib.glg_smooth_create(e1._e, 1, C.byref(out)) == _lib.GLG_ERR_ARG and not out
    e1.reset()  # before the smoother: not recorded
    s1, s2 = DeviceStateSmoother(e1, 6), DeviceStateSmoother(e2, 6)
    with pytest.raises(_lib.GlgError, match="already has a smoother"):
        DeviceStateSmoother(e1, 6)
    env.step_rule_based_tensor()
    e1.update(None)
    assert s1.length == 0
    with pytest.raises(_lib.GlgError, match="nothing recorded"):
        s1.smooth()
    e1.reset()
    e2.reset()
    gen = torch.Generator(device="cuda").manual_seed(10)
    for _ in range(8):
        env.step_rule_based_tensor()
        y = _noisy(e1, gen)
        e1.update(y)
        e2.update(y)
    a, b = s1.smooth(), s2.smooth()
    torch.cuda.synchronize()
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    for name in ("prior_mean", "prior_cov", "cross_cov", "status", "timestep"):
        assert torch.equal(getattr(s1, name), getattr(s2, name)), name
    s1.close()
    s3 = DeviceStateSmoother(e1, 3)  # the estimator's smoother slot is free again
    e2.close()  # the estimator before its smoother: the smoother can only be closed
    with pytest.raises(RuntimeError, match="closed"):
        s2.smooth()
    s2.close()
    s3.close()
    e1.close()
    env.close()


@pytest.mark.gpu
def test_smoothed_track_is_not_worse_than_the_filtered_one():
    """The estimator test's setting: 16 envs at uncertainty_scale 0.2, rule-based, two days from a wrong prior.  Over the window
    the smoothed RMS error of CO2, air temperature and vapour pressure (RH) against the true state is not above the filtered one."""
    from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
    B, steps = 16, 192
    env = _env(B, uncertainty_scale=0.2)
    _warm(env, 0)
    x0 = env.state_t.T.clone()
    x0[:, 2:15] += 1.5
    x0[:, 22:26] *= 1.1
    est = DeviceStateEstimator(env)
    sm = DeviceStateSmoother(est, steps + 1)
    est.reset(x0)
    truth = [env.state_t.T.cpu().numpy().copy()]
    gen = torch.Generator(device="cuda").manual_seed(4)
    for _ in range(steps):
        env.step_rule_based_tensor()
        est.update(_noisy(est, gen))
        truth.append(env.state_t.T.cpu().numpy().copy())
    s = sm.smooth()
    torch.cuda.synchronize()
    truth = np.stack(truth)
    assert np.all(sm.status.cpu().numpy() == 0)
    rms = lambda m: np.sqrt(np.mean(np.square(m - truth), axis=(0, 1)))
    sm_rms, f_rms = rms(s.mean.cpu().numpy()), rms(sm.filtered_mean.cpu().numpy())
    print("per-state RMS of x - x_true, smoothed:", np.array2string(sm_rms, precision=4), "filtered:",
          np.array2string(f_rms, precision=4))
    for j in (0, 2, 15):
        assert sm_rms[j] <= f_rms[j], (j, sm_rms[j], f_rms[j])
    sm.close()
    est.close()
    env.close()
