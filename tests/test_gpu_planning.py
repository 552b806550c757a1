"""Receding-horizon planner (csrc/glg_plan.cuh, glgym.planning.DevicePlanner) against restatements: the returns against a second
env stepped with the same sequences, the samples against numpy + philox_ref, the CEM update against a numpy lexsort of the device's
own candidates and returns."""
import ctypes as C

import numpy as np
import pytest

import philox_ref

torch = pytest.importorskip("torch")

SHORT2 = dict(season_length=7 / 96.0, start_train_day=0, end_train_day=1)  # N = 7, two weather tables


def test_plan_entry_points_reject_null_arguments():
    """CPU tier: the C entry points fail loudly on NULL objects instead of touching memory."""
    from glgym import _lib
    lib = _lib.load()
    cfg = _lib.GlgPlanConfig(4, 8, 2, 1, 1.0, 0.5, 0)
    out = C.c_void_p()
    assert lib.glg_plan_create(None, C.byref(cfg), C.byref(out)) == _lib.GLG_ERR_ARG and not out
    assert lib.glg_plan_run(None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_plan_evaluate(None, None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_plan_shift(None, None) == _lib.GLG_ERR_ARG
    for view in ("mean", "std", "candidates", "returns"):
        assert getattr(lib, f"glg_plan_{view}_dev")(None) is None
    lib.glg_plan_destroy(None)
    assert C.sizeof(_lib.GlgPlanConfig) == 40


def _env(B, **kw):
    from glgym.vec_env import GreenLightVecEnv
    base = dict(seed=3, base_env_params=SHORT2)  # the default integrator: random actions keep the state finite
    base.update(kw)
    return GreenLightVecEnv(B, **base)


def _warm_start(env, steps=2, seed=0):
    """Reset onto alternating tables and take a few random steps, so the envs hold distinct states."""
    B = env.num_envs
    env.reset_tensor(table_ids=torch.arange(B, device="cuda", dtype=torch.int32) % 2)
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    for _ in range(steps):
        env.step_tensor(torch.rand(B, 6, device="cuda", generator=g) * 2 - 1)
    torch.cuda.synchronize()


def masked_returns(rewards, dones, gamma):
    """R = sum_t d_t alive_t r_t, d_0 = 1, d_{t+1} = d_t gamma, alive_{t+1} = alive_t (1 - done_t)."""
    R = np.zeros(rewards.shape[1])
    alive = np.ones(rewards.shape[1], bool)
    d = 1.0
    for r, dn in zip(rewards, dones):
        R[alive] = R[alive] + d * r[alive]
        alive &= ~dn
        d *= gamma
    return R


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_plan_scores_equal_stepping_a_clone(precision):
    """evaluate(seq) is bit-equal to a second env of B K envs loaded with the replicated states and stepped with the same
    sequences; some envs start two steps before the episode end, so the horizon crosses it and the masking is exercised."""
    from glgym.planning import DevicePlanner
    B, K, H, gamma = 6, 8, 5, 0.9
    env = _env(B, precision=precision)
    _warm_start(env)
    x, u, k = env.get_state()
    k[[1, 4]] = env.N - 2
    env.set_state(timestep=k)
    planner = DevicePlanner(env, H, K, 2, 1, gamma=gamma)
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    seq = torch.rand(H, B * K, 6, device="cuda", generator=g) * 2 - 1
    got = planner.evaluate(seq).cpu().numpy().reshape(-1)

    ref = _env(B * K, precision=precision, auto_reset=False)
    st = env.state_dict()
    rep = {n: np.repeat(a, K, axis=0) for n, a in st.items()}
    rep["ep_return"][:] = 0; rep["ep_len"][:] = 0; rep["ep_info"][:] = 0
    ref.load_state_dict(rep)
    rew, dn = [], []
    for t in range(H):
        ref.step_tensor(seq[t])
        rew.append(ref.reward_t.cpu().numpy().copy())
        dn.append(ref.done_t.cpu().numpy().astype(bool))
    rew, dn = np.array(rew), np.array(dn)
    want = masked_returns(rew, dn, gamma)
    assert np.isfinite(rew).all() and ref.episode_stats()["nonfinite"] == 0  # no step failed: every done is an episode end
    # the horizon crosses the episode end where it should: envs 1 and 4 (timestep N - 2) end with their third step, the others
    # (timestep 2) not at all
    assert dn[2, 1 * K:2 * K].all() and dn[2, 4 * K:5 * K].all() and dn[:2].sum() == 0
    assert dn.sum() == dn[:, K:2 * K].sum() + dn[:, 4 * K:5 * K].sum()
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), np.abs(got - want).max()
    assert np.all(np.isfinite(got))
    planner.close(); ref.close(); env.close()


def _snapshot(env):
    out = {f"state.{n}": a for n, a in env.state_dict().items()}
    for n in ("obs_t", "terminal_obs_t", "reward_t", "done_t", "info_t", "stats_t"):
        out[n] = getattr(env, n).cpu().numpy().copy()
    return out


@pytest.mark.gpu
def test_plan_leaves_the_env_untouched():
    from glgym.planning import DevicePlanner
    env = _env(8, observation_modules=["StateObservations", "IndoorClimateObservations", "WeatherForecastObservations"])
    _warm_start(env, steps=8)  # past the episode end of N = 7: terminal rows and statistics are non-trivial
    before = _snapshot(env)
    planner = DevicePlanner(env, 4, 16, 4, 2, gamma=0.95, seed=1)
    a = planner.plan()
    planner.evaluate(torch.zeros(4, 8 * 16, 6, device="cuda"))
    torch.cuda.synchronize()
    after = _snapshot(env)
    for n in before:
        assert before[n].tobytes() == after[n].tobytes(), n
    assert a.shape == (8, 6) and bool(torch.isfinite(a).all())
    planner.close(); env.close()


def expected_candidates(mean, std, seed, call, it, K):
    """[H][B K][6] samples of glg_plan_sample_kernel from float32 mean / std [H][B][6]."""
    H, B, _ = mean.shape
    out = np.empty((H, B * K, 6), np.float32)
    lo, hi = seed & philox_ref.MASK, (seed >> 32) & philox_ref.MASK
    for c in range(B * K):
        b, k = divmod(c, K)
        for t in range(H):
            z = np.zeros(6)
            if k:
                for p in range(3):
                    r = philox_ref.philox4x32_10(66, call, (it * H + t) * 3 + p, c, lo, hi)
                    u1, u2 = 1.0 - philox_ref.u01(r[0], r[1]), philox_ref.u01(r[2], r[3])
                    rad, ang = np.sqrt(-2.0 * np.log(u1)), 6.283185307179586 * u2
                    z[2 * p], z[2 * p + 1] = rad * np.cos(ang), rad * np.sin(ang)
            m, s = mean[t, b].astype(np.float64), std[t, b].astype(np.float64)
            out[t, c] = np.clip(m + s * z, -1.0, 1.0).astype(np.float32)
    return out


def _within_one_ulp(got, want):
    return np.all(np.abs(got.astype(np.float64) - want) <= np.spacing(np.abs(want)).astype(np.float64))


@pytest.mark.gpu
def test_plan_samples_match_restatement():
    from glgym.planning import DevicePlanner
    B, K, H, seed = 4, 16, 4, 0x1234_5678_9ABC
    env = _env(B)
    _warm_start(env)
    planner = DevicePlanner(env, H, K, 4, 1, seed=seed)
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    planner.mean.copy_(torch.rand(H, B, 6, device="cuda", generator=g) * 2.4 - 1.2)  # beyond [-1, 1]: candidate 0 is clipped
    planner.std.copy_(torch.rand(H, B, 6, device="cuda", generator=g) * 0.9 + 0.1)
    for call in range(2):
        mean, std = planner.mean.cpu().numpy().copy(), planner.std.cpu().numpy().copy()
        planner.plan()
        got = planner.candidates.cpu().numpy().reshape(H, B * K, 6)
        want = expected_candidates(mean, std, seed, call, 0, K)
        assert _within_one_ulp(got, want), call
        assert np.array_equal(got[:, ::K], np.clip(mean, -1, 1)), call  # candidate 0 = the clipped mean
        assert (np.abs(got) == 1.0).any()  # the clamp was exercised
    planner.close(); env.close()


def expected_update(cand, ret, E):
    """New mean / std [H][B][6] from candidates [H][B][K][6] and returns [B][K]: elites by a lexsort (descending return, ties to
    the lower k, non-finite last), then their fp64 mean and population standard deviation."""
    H, B, K, _ = cand.shape
    mean, std = np.empty((H, B, 6)), np.empty((H, B, 6))
    for b in range(B):
        key = np.where(np.isfinite(ret[b]), ret[b], -np.inf)
        el = np.sort(np.lexsort((np.arange(K), -key))[:E])
        a = cand[:, b, el].astype(np.float64)
        m = a.sum(axis=1) / E
        mean[:, b], std[:, b] = m, np.sqrt(((a - m[:, None]) ** 2).sum(axis=1) / E)
    return mean, std


@pytest.mark.gpu
@pytest.mark.parametrize("E", [1, 5, 32])
def test_plan_update_matches_restatement(E):
    from glgym.planning import DevicePlanner
    B, K, H = 4, 32, 3
    env = _env(B)
    _warm_start(env)
    planner = DevicePlanner(env, H, K, E, 2, gamma=0.97, seed=9)
    for call in range(2):
        a = planner.plan().cpu().numpy().copy()
        cand = planner.candidates.cpu().numpy().copy()
        ret = planner.returns.cpu().numpy().copy()
        mean, std = expected_update(cand, ret, E)
        assert np.allclose(planner.mean.cpu().numpy(), mean, rtol=0, atol=1e-6), call
        assert np.allclose(planner.std.cpu().numpy(), std, rtol=0, atol=1e-6), call
        assert np.array_equal(a, planner.mean[0].cpu().numpy()), call
        if E == K:
            assert np.allclose(mean, cand.astype(np.float64).mean(axis=2), rtol=0, atol=1e-6)
        env.step_tensor(torch.as_tensor(a, device="cuda"))
        planner.shift()
    planner.close(); env.close()


@pytest.mark.gpu
def test_plan_shift():
    from glgym.planning import DevicePlanner
    B, H, init_std = 5, 4, 0.3
    env = _env(B)
    planner = DevicePlanner(env, H, 4, 2, 1, init_std=init_std)
    assert torch.equal(planner.mean, torch.zeros(H, B, 6, device="cuda"))
    assert torch.equal(planner.std, torch.full((H, B, 6), init_std, device="cuda"))
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    planner.mean.copy_(torch.rand(H, B, 6, device="cuda", generator=g))
    planner.std.copy_(torch.rand(H, B, 6, device="cuda", generator=g))
    m = planner.mean.clone()
    planner.shift()
    assert torch.equal(planner.mean[:-1], m[1:]) and torch.equal(planner.mean[-1], torch.zeros(B, 6, device="cuda"))
    assert torch.equal(planner.std, torch.full((H, B, 6), init_std, device="cuda"))
    planner.close(); env.close()


@pytest.mark.gpu
def test_plan_is_deterministic_and_seeded():
    from glgym.planning import DevicePlanner
    B, K, H = 6, 64, 4
    env = _env(B)
    _warm_start(env)
    p1, p2, p3 = (DevicePlanner(env, H, K, 8, 3, seed=s) for s in (21, 21, 22))
    a1 = p1.plan().clone()
    a2 = p2.plan().clone()
    assert torch.equal(a1, a2) and torch.equal(p1.candidates, p2.candidates) and torch.equal(p1.returns, p2.returns)
    assert torch.equal(p1.mean, p2.mean) and torch.equal(p1.std, p2.std)
    p3.plan()
    assert not torch.equal(p1.candidates, p3.candidates)
    for p in (p1, p2, p3):
        p.close()
    env.close()


@pytest.mark.gpu
def test_plan_fences():
    from glgym import _lib
    from glgym.planning import DevicePlanner
    B = 4
    env = _env(B)
    for bad in (dict(horizon=0), dict(n_candidates=0), dict(n_elites=0), dict(n_elites=9), dict(n_candidates=4097, n_elites=1),
                dict(n_iterations=0), dict(gamma=0.0), dict(gamma=1.5), dict(gamma=float("nan")), dict(init_std=0.0),
                dict(init_std=-1.0), dict(init_std=float("inf"))):
        cfg = dict(horizon=2, n_candidates=8, n_elites=2, n_iterations=1)
        cfg.update(bad)
        with pytest.raises(_lib.GlgError, match="status -1"):
            DevicePlanner(env, **cfg)
    big = _env(1025, n_sub=1)
    with pytest.raises(_lib.GlgError, match="4194304"):
        DevicePlanner(big, 1, 4096, 1, 1)
    big.close()
    # un-reset env
    planner = DevicePlanner(env, 2, 8, 2, 1)
    a = torch.empty(B, 6, device="cuda")
    assert env._lib.glg_plan_run(planner._p, a.data_ptr(), None) == _lib.GLG_ERR_STATE
    with pytest.raises(_lib.GlgError, match="not been reset"):
        planner.plan()
    with pytest.raises(_lib.GlgError, match="not been reset"):
        planner.evaluate(torch.zeros(2, B * 8, 6, device="cuda"))
    _warm_start(env, steps=1)
    planner.plan()
    assert env._lib.glg_plan_run(planner._p, None, None) == _lib.GLG_ERR_ARG
    assert env._lib.glg_plan_evaluate(planner._p, None, planner.returns.data_ptr(), None) == _lib.GLG_ERR_ARG
    assert env._lib.glg_plan_evaluate(planner._p, a.data_ptr(), None, None) == _lib.GLG_ERR_ARG
    with pytest.raises(ValueError):
        planner.evaluate(torch.zeros(3, B * 8, 6, device="cuda"))
    # a new weather bank invalidates the planner, which shares the env's bank
    W = env.weather_tables
    _lib.check(env._lib.glg_set_weather(env._h, W.ctypes.data, W.shape[0], W.shape[1], env.table_start_days.ctypes.data), env._h,
               "glg_set_weather")
    assert env._lib.glg_plan_run(planner._p, a.data_ptr(), None) == _lib.GLG_ERR_STATE
    with pytest.raises(_lib.GlgError, match="weather bank"):
        planner.plan()
    with pytest.raises(_lib.GlgError, match="weather bank"):
        planner.evaluate(torch.zeros(2, B * 8, 6, device="cuda"))
    p2 = DevicePlanner(env, 2, 8, 2, 1)  # a planner created under the new bank works
    assert p2.plan().shape == (B, 6)
    planner.close()
    with pytest.raises(RuntimeError, match="closed"):
        planner.plan()
    env.close()
    with pytest.raises(RuntimeError, match="env"):
        p2.plan()
    with pytest.raises(RuntimeError, match="env"):
        p2.shift()
    p2.close()  # after its env: frees only the planner's own memory


@pytest.mark.gpu
def test_closed_loop_planner_beats_holding():
    """16 envs, one day (96 steps) from the January start states: MPC (H = 8, K = 128, E = 16, I = 3) against the hold policy
    a = 0, which keeps the reset controls (heating off)."""
    from glgym.planning import DevicePlanner
    from glgym.vec_env import GreenLightVecEnv
    B, steps = 16, 96
    env = GreenLightVecEnv(B, seed=0)
    env.reset_tensor()
    start = env.state_dict()
    planner = DevicePlanner(env, 8, 128, 16, 3, seed=0)
    r_plan = []
    for _ in range(steps):
        a = planner.plan()
        _, r, _ = env.step_tensor(a)
        r_plan.append(r.cpu().numpy().copy())
        planner.shift()
    env.load_state_dict(start)
    zero = torch.zeros(B, 6, device="cuda")
    r_hold = []
    for _ in range(steps):
        _, r, _ = env.step_tensor(zero)
        r_hold.append(r.cpu().numpy().copy())
    m_plan, m_hold = float(np.mean(r_plan)), float(np.mean(r_hold))
    print(f"mean reward per step: planner {m_plan:+.5f}, hold {m_hold:+.5f}")
    assert m_plan >= m_hold, (m_plan, m_hold)
    planner.close(); env.close()
