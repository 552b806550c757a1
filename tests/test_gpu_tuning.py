"""Per-env rule-based controls (csrc glg_rule_controls, GreenLightVecEnv.rule_controls_tensor) and the CEM tuner over the
controller's settings (glgym.tuning.RuleControllerTuner): the controls-then-raw-step path against the fused rule-based step, per-env
settings against the host controller and against one handle per settings vector, and the tuner's fitness and update against numpy
restatements."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

SHORT = dict(season_length=1, start_train_day=0, end_train_day=2)  # N = 96 (97 steps per episode), three weather tables
THREE = dict(start_train_day=0, end_train_day=2)                    # full season, three weather tables
CUSTOM = dict(lamps_on=2, lamps_off=20, heat_correction=1.5, temp_setpoint_day=21.0, co2_day=1000, useBlScr=0)
OTHER = dict(temp_setpoint_day=22.0, temp_setpoint_night=14.0, heat_deadzone=3.0, co2_day=600, vent_heat_Pband=7.0, rh_max=80.0,
             thScrSpNight=3.0, lamps_off_sun=250.0, lamp_rad_sum_limit=15.0)


# ------------------------------------------------------------------------------------------------ CPU tier
def test_rule_controls_exported_and_rejects_null():
    from glgym import _lib
    lib = _lib.load()
    assert hasattr(lib, "glg_rule_controls")
    buf = (C.c_double * 6)()
    assert lib.glg_rule_controls(None, None, C.addressof(buf), None) == _lib.GLG_ERR_ARG
    assert lib.glg_rule_controls(None, None, None, None) == _lib.GLG_ERR_ARG


def test_controller_setting_names_and_from_vector():
    from glgym.controller import DEFAULT_SETTINGS, SETTING_NAMES, RuleBasedController
    assert SETTING_NAMES == tuple(DEFAULT_SETTINGS) and len(SETTING_NAMES) == 29
    v = np.arange(29, dtype=np.float64) + 0.25
    c = RuleBasedController.from_vector(v)
    assert np.array_equal(c.settings_vector(), v)
    with pytest.raises(ValueError):
        RuleBasedController.from_vector(v[:28])


@pytest.mark.parametrize("kw", [
    dict(bounds={"no_such_setting": (0.0, 1.0)}),
    dict(base={"no_such_setting": 1.0}),
    dict(bounds={"temp_setpoint_day": (20.0, 20.0)}),
    dict(bounds={"temp_setpoint_day": (21.0, 20.0)}),
    dict(bounds={"temp_setpoint_day": (20.0, 24.0)}),                      # shipped 19.5 lies outside
    dict(bounds={"co2_day": (400.0, 1200.0)}, base={"co2_day": 1300.0}),
    dict(bounds={"vent_heat_Pband": (-1.0, 10.0)}),                         # a proportional band through 0
    dict(bounds={"tHeatBand": (-2.0, 0.0)}, base={"tHeatBand": -1.0}),
    dict(bounds={"co2Band": (-200.0, 50.0)}),
    dict(n_candidates=8, n_elites=0),
    dict(n_candidates=8, n_elites=9),
    dict(horizon=0),
    dict(horizon=5762),                                                     # N + 2 for the default 60-day season
    dict(horizon=98, base_env_params=dict(season_length=1)),
])
def test_tuner_rejects_bad_arguments(kw):
    """Every check runs before an env is built, so these need no GPU."""
    from glgym.tuning import RuleControllerTuner
    with pytest.raises(ValueError):
        RuleControllerTuner(**kw)


def _np_fitness(rewards, dones, K, S):
    """Restatement: per env, the sum of the rewards up to and including its first done; bad if that done comes before the
    last step or a counted reward is not finite; per candidate the mean over its S envs, -inf if any of them is bad."""
    H, B = rewards.shape
    ret, bad = np.zeros(B), np.zeros(B, bool)
    for c in range(B):
        hit = np.nonzero(dones[:, c])[0]
        end = hit[0] if hit.size else H - 1
        bad[c] = (hit.size and hit[0] < H - 1) or not np.all(np.isfinite(rewards[:end + 1, c]))
        ret[c] = sum(float(r) for r in rewards[:end + 1, c])
    fit = ret.reshape(K, S).mean(axis=1)
    fit[bad.reshape(K, S).any(axis=1)] = -np.inf
    return fit


def test_fitness_accumulation_against_numpy():
    from glgym.tuning import SeasonFitness
    K, S, H = 8, 3, 6
    rng = np.random.default_rng(0)
    rewards = rng.normal(size=(H, K * S))
    dones = np.zeros((H, K * S), bool)
    dones[2, 2 * S + 1] = True                              # candidate 2: an env done mid-horizon -> -inf
    rewards[3, 5 * S + 0] = np.nan                          # candidate 5: a non-finite reward -> -inf
    dones[H - 1, 6 * S + 2] = True                          # candidate 6: done on the last step -> finite
    dones[H - 1, 7 * S:] = True                             # candidate 7: every env done on the last step -> finite
    rewards[1, 4 * S + 2] = np.inf                          # candidate 4: +inf reward -> -inf
    rewards[:, 3 * S:4 * S] = rewards[:, 1 * S:2 * S]       # candidates 1 and 3 tie
    acc = SeasonFitness(K, S, "cpu")
    for t in range(H):
        acc.add(torch.from_numpy(rewards[t]), torch.from_numpy(dones[t].astype(np.uint8)), last=t == H - 1)
    got = acc.result().numpy()
    ref = _np_fitness(rewards, dones, K, S)
    assert np.array_equal(np.isinf(got), np.isinf(ref)) and set(np.nonzero(np.isinf(ref))[0]) == {2, 4, 5}
    assert np.allclose(got[np.isfinite(ref)], ref[np.isfinite(ref)], rtol=1e-15, atol=0)
    assert got[1] == got[3]


def _np_update(cand, fit, E, tuned):
    order = np.lexsort((np.arange(len(fit)), -fit))   # largest first, ties to the lower index, -inf last
    el = order[:E]
    x = cand[el][:, tuned]
    return el, x.mean(axis=0), x.std(axis=0)


@pytest.mark.parametrize("E", [1, 4, 5, 8])
def test_elite_update_against_numpy(E):
    from glgym.tuning import elite_update
    rng = np.random.default_rng(E)
    K = 8
    cand = rng.normal(size=(K, 29))
    fit = np.array([1.0, 3.0, 2.0, 3.0, -np.inf, 2.0, 0.5, 2.0])  # ties at the top and across the E = 4 / 5 boundary
    tuned = np.array([0, 6, 7, 10, 28])
    el, m, s = elite_update(torch.from_numpy(cand), torch.from_numpy(fit), E, torch.from_numpy(tuned))
    el_r, m_r, s_r = _np_update(cand, fit, E, tuned)
    assert el.tolist() == el_r.tolist()
    assert np.allclose(m.numpy(), m_r, rtol=1e-14, atol=1e-15) and np.allclose(s.numpy(), s_r, rtol=1e-13, atol=1e-15)
    if E == 1:
        assert el.tolist() == [1] and np.all(s.numpy() == 0)


# ------------------------------------------------------------------------------------------------ GPU tier
def _env(B, **kw):
    from glgym.vec_env import GreenLightVecEnv
    return GreenLightVecEnv(B, **kw)


def _views(env):
    return dict(x=env.state_t, u=env.controls_t, obs=env.obs_t, term=env.terminal_obs_t, reward=env.reward_t, done=env.done_t,
                info=env.info_t, stats=env.stats_t)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,role_warps,integrator,scale", [  # fp32 runs on kernel C only (role_warps 2, 3)
    (p, r, i, 0.0) for p in ("fp64", "fp32") for r in (1, 2, 3) for i in ("fixed", "graded") if (p, r) != ("fp32", 1)]
    + [("fp64", 2, "graded", 0.2)])
def test_rule_controls_then_raw_step_equals_fused_step(precision, role_warps, integrator, scale):
    """rule_controls_tensor(None) + step_raw_control_tensor is bit-identical to step_rule_based_tensor over 200 steps of 97-step
    episodes (two auto-resets), in every output; with uncertainty both paths key the Philox noise by env id."""
    kw = dict(precision=precision, role_warps=role_warps, integrator=integrator, uncertainty_scale=scale, seed=11,
              base_env_params=SHORT, info_mode="minimal")
    a, b = _env(8, **kw), _env(8, **kw)
    for env in (a, b):
        env.set_rule_controller(CUSTOM)
        env.reset_tensor()
    va, vb = _views(a), _views(b)
    resets = 0
    for t in range(200):
        a.step_raw_control_tensor(a.rule_controls_tensor())
        b.step_rule_based_tensor()
        for n in va:
            assert torch.equal(va[n], vb[n]), (t, n)
        resets += int(vb["done"].any())
    assert resets == 2
    assert torch.isfinite(va["x"]).all()
    a.close()
    b.close()


def _per_env_setup(env, k0):
    B = env.num_envs
    env.reset_tensor(table_ids=torch.arange(B, device=env.device, dtype=torch.int32) % 2)
    env.set_state(timestep=np.asarray(k0, dtype=np.int32))


@pytest.mark.gpu
def test_per_env_settings_match_host_controller_and_one_handle_per_setting():
    from glgym.controller import RuleBasedController
    sets = [dict(), CUSTOM, OTHER]
    B = 6
    k0 = [8, 40, 70, 24, 56, 88]          # two tables (e % 2), different timesteps and hours of day
    which = [e % 3 for e in range(B)]
    vecs = np.stack([RuleBasedController(**s).settings_vector() for s in sets])
    settings = torch.as_tensor(vecs[which], device="cuda")
    env = _env(B, base_env_params=THREE)
    _per_env_setup(env, k0)
    refs = []
    for s in sets:
        r = _env(B, base_env_params=THREE)
        r.set_rule_controller(s)
        _per_env_setup(r, k0)
        refs.append(r)
    W = env.weather_tables
    worst = 0.0
    for t in range(100):
        u = env.rule_controls_tensor(settings)
        if t % 20 == 0:  # the controls against the host controller on each env's state, weather row and clock
            x, k, tb, tm = (v.cpu().numpy() for v in (env.state_t, env.timestep_t, env.table_t, env.time_t))
            for e in range(B):
                d = W[tb[e], min(k[e], W.shape[1] - env.Np - 1)]
                ref = RuleBasedController(**sets[which[e]]).predict(x[:, e], d, tm[1, e], tm[0, e])[0]
                worst = max(worst, float(np.abs(u[e].cpu().numpy() - ref).max()))
        env.step_raw_control_tensor(u)
        for r in refs:
            r.step_rule_based_tensor()
        for j, r in enumerate(refs):
            cols = [e for e in range(B) if which[e] == j]
            for n, (va, vb) in enumerate(zip((env.state_t, env.controls_t), (r.state_t, r.controls_t))):
                assert torch.equal(va[:, cols], vb[:, cols]), (t, j, n)
            for va, vb in ((env.obs_t, r.obs_t), (env.reward_t, r.reward_t), (env.done_t, r.done_t)):
                assert torch.equal(va[cols], vb[cols]), (t, j)
    assert worst <= 1e-14, worst
    for r in refs:
        r.close()
    env.close()


@pytest.mark.gpu
def test_rule_controls_fences():
    from glgym import _lib
    env = _env(4, base_env_params=SHORT)
    with pytest.raises(_lib.GlgError, match=f"status {_lib.GLG_ERR_STATE}"):
        env.rule_controls_tensor()
    env.reset_tensor()
    for shape in ((4, 28), (3, 29), (4 * 29,)):
        with pytest.raises(ValueError):
            env.rule_controls_tensor(torch.zeros(shape, dtype=torch.float64, device="cuda"))
    assert env._lib.glg_rule_controls(env._h, None, None, None) == _lib.GLG_ERR_ARG
    n0 = env.launch_count()
    u = env.rule_controls_tensor(torch.zeros((4, 29), dtype=torch.float32, device="cuda") + 5)  # dtype converted
    assert env.launch_count() == n0 + 1 and u.shape == (4, 6) and u.dtype == torch.float64
    env.close()


def _run_tuner(**kw):
    from glgym.tuning import RuleControllerTuner
    tuner = RuleControllerTuner(n_candidates=32, n_elites=6, horizon=96, seed=4, base_env_params=THREE, **kw)
    gens = []
    for _ in range(2):
        mean0 = tuner.mean.clone()
        tuner.generation()
        gens.append((mean0, tuner.candidates.clone(), tuner.fitness.clone(), tuner.mean.clone(), tuner.std.clone()))
    return tuner, gens


@pytest.mark.gpu
def test_tuner_generations():
    from glgym.controller import SETTING_NAMES
    from glgym.tuning import DEFAULT_BOUNDS
    t1, gens = _run_tuner()
    t2, _ = _run_tuner()
    assert t1.n_scenarios == 3 and t1.env.num_envs == 96
    assert t1.history == t2.history and t1.best_settings == t2.best_settings and len(t1.history) == 2
    lo, hi = t1.lo.cpu().numpy(), t1.hi.cpu().numpy()
    tuned = np.array([SETTING_NAMES.index(k) for k in DEFAULT_BOUNDS])
    fixed = np.setdiff1d(np.arange(29), tuned)
    base = np.array([t1.base[k] for k in SETTING_NAMES])
    best_seen = -np.inf
    for mean0, cand, fit, mean1, std1 in gens:
        c, f = cand.cpu().numpy(), fit.cpu().numpy()
        assert np.all(c >= lo) and np.all(c <= hi)
        assert np.array_equal(c[:, fixed], np.broadcast_to(base[fixed], (32, len(fixed))))
        assert np.array_equal(c[0], np.clip(mean0.cpu().numpy(), lo, hi))     # candidate 0 is the clamped mean
        assert np.isfinite(f).all() and len(np.unique(f)) > 1
        _, m_r, s_r = _np_update(c, f, 6, tuned)
        assert np.allclose(mean1.cpu().numpy()[tuned], m_r, rtol=1e-14, atol=0)
        assert np.allclose(std1.cpu().numpy()[tuned], s_r, rtol=1e-12, atol=1e-15)
        assert np.array_equal(mean1.cpu().numpy()[fixed], base[fixed]) and np.all(std1.cpu().numpy()[fixed] == 0)
        best_seen = max(best_seen, f.max())
    assert t1.best_fitness == best_seen
    got = t1.evaluate([t1.best_settings])
    assert got[0] == t1.best_fitness                                          # bit for bit
    t1.close()
    t2.close()


@pytest.mark.gpu
def test_tuner_common_random_numbers():
    """Under uncertainty two identical candidates see the same noise sample: identical fitness.  The noise is applied."""
    from glgym.tuning import RuleControllerTuner
    kw = dict(n_candidates=4, n_elites=2, horizon=96, base_env_params=THREE)
    noisy = RuleControllerTuner(uncertainty_scale=0.2, seed=1, **kw)
    f = noisy.evaluate([OTHER, OTHER, {}, OTHER])
    assert f[0] == f[1] == f[3] and np.isfinite(f).all()
    assert noisy.evaluate([OTHER])[0] == f[0]                                 # same sample in every rollout
    noisy.close()
    plain = RuleControllerTuner(seed=1, **kw)
    assert plain.evaluate([OTHER])[0] != f[0]
    plain.close()
