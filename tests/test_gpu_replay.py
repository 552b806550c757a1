"""Device replay buffer (csrc/glg_replay.cuh, glgym.replay.DeviceReplayBuffer) against a numpy restatement of SB3 2.6.0's
ReplayBuffer (optimize_memory_usage=False, handle_timeout_termination=True: add / sample / _get_samples) filled the way
OffPolicyAlgorithm._store_transition fills it behind VecNormalize.  SB3 is pinned by the reference and not installed here, so the
restatement below is the oracle, fed with the raw outputs of an identical second env as in test_normalize.py."""
import ctypes as C

import numpy as np
import pytest

import philox_ref
from test_normalize import NpVecNormalize

torch = pytest.importorskip("torch")


class NpReplayBuffer:
    """SB3 ReplayBuffer with _store_transition's next-observation rule (terminal row of a done env)."""

    def __init__(self, buffer_size, n_envs, obs_dim):
        self.buffer_size, self.n_envs = max(buffer_size // n_envs, 1), n_envs
        shape = (self.buffer_size, n_envs)
        self.observations = np.zeros(shape + (obs_dim,), np.float32)
        self.next_observations = np.zeros(shape + (obs_dim,), np.float32)
        self.actions = np.zeros(shape + (6,), np.float32)
        self.rewards, self.dones, self.timeouts = (np.zeros(shape, np.float32) for _ in range(3))
        self.pos, self.full = 0, False

    def add(self, obs, next_obs, action, reward, done, infos):
        self.observations[self.pos] = np.array(obs)
        self.next_observations[self.pos] = np.array(next_obs)
        self.actions[self.pos] = np.array(action)
        self.rewards[self.pos] = np.array(reward)
        self.dones[self.pos] = np.array(done)
        self.timeouts[self.pos] = np.array([info.get("TimeLimit.truncated", False) for info in infos])
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full, self.pos = True, 0

    def size(self):
        return self.buffer_size if self.full else self.pos

    def get_samples(self, batch_inds, env_indices, vn=None):
        o, no = self.observations[batch_inds, env_indices], self.next_observations[batch_inds, env_indices]
        r = self.rewards[batch_inds, env_indices].reshape(-1, 1)
        if vn is not None:
            o, no = vn.norm_obs(o.astype(np.float64)), vn.norm_obs(no.astype(np.float64))
            r = np.clip(r / np.sqrt(vn.ret_rms.var + vn.eps), -vn.cr, vn.cr).astype(np.float32)
        dones = (self.dones[batch_inds, env_indices] * (1 - self.timeouts[batch_inds, env_indices])).reshape(-1, 1)
        return o, self.actions[batch_inds, env_indices], no, dones, r


def store_transition(ref, last_obs, env, actions, auto_reset=True):
    """_store_transition on the env's raw outputs of the step that just ran; returns the new _last_original_obs."""
    obs = env.obs_t.cpu().numpy().copy()
    done = env.done_t.cpu().numpy().astype(bool)
    nxt = obs.copy()
    if auto_reset:
        nxt[done] = env.terminal_obs_t.cpu().numpy()[done]
    infos = [{"TimeLimit.truncated": False} for _ in range(len(done))]
    ref.add(last_obs, nxt, actions.cpu().numpy(), env.reward_t.cpu().numpy().astype(np.float32), done, infos)
    return obs


def replay_draws(seed, call, n, upper, B):
    """glg_replay_draw (csrc/glg_philox.h): counter (65, call, i, 0), key = seed."""
    out = np.zeros((n, 2), np.int64)
    for i in range(n):
        r = philox_ref.philox4x32_10(65, call, i, 0, seed & philox_ref.MASK, (seed >> 32) & philox_ref.MASK)
        out[i] = (r[0] * upper) >> 32, (r[1] * B) >> 32
    return out


SHORT = dict(season_length=7 / 96.0)


def test_replay_entry_points_reject_null_arguments():
    """CPU tier: the C entry points fail loudly on NULL objects instead of touching memory."""
    from glgym import _lib
    lib = _lib.load()
    cfg = _lib.GlgReplayConfig(1000, 1, 1, 1, 0, 0.99, 10.0, 10.0, 1e-8, 0)
    out = C.c_void_p()
    assert lib.glg_replay_create(None, C.byref(cfg), C.byref(out)) == _lib.GLG_ERR_ARG and not out
    assert lib.glg_replay_reset(None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_replay_store(None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_replay_sample(None, 1, None, None, None, None, None, None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_replay_size(None) == 0 and lib.glg_replay_bytes(None) == 0
    lib.glg_replay_destroy(None)
    assert C.sizeof(_lib.GlgReplayConfig) == 64


@pytest.mark.gpu
def test_replay_matches_sb3_restatement():
    """Statistics, normalised current observation and samples (indices, normalised observations, actions, rewards, dones) after
    every store, 5 slots per env and 15 steps so the ring wraps and episodes end inside the run."""
    from glgym.replay import DeviceReplayBuffer
    from glgym.vec_env import GreenLightVecEnv
    B, gamma, seed, n = 200, 0.9631, 11, 1000
    kw = dict(n_sub=300, integrator="fixed", seed=5, base_env_params=SHORT)
    env, raw = GreenLightVecEnv(B, **kw), GreenLightVecEnv(B, **kw)
    rb = DeviceReplayBuffer(env, 5 * B + 3, gamma=gamma, seed=seed)
    assert rb.capacity == 5
    vn, ref = NpVecNormalize(B, env.obs_dim, gamma), NpReplayBuffer(5 * B + 3, B, env.obs_dim)
    o = rb.reset()
    last = raw.reset_tensor().cpu().numpy().copy()
    assert np.allclose(o.cpu().numpy(), vn.reset(last.astype(np.float64)), atol=2e-6)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    idx = torch.empty((n, 2), dtype=torch.int32, device="cuda")
    calls, n_done, sampled_done = 0, 0, 0
    for t in range(15):
        a = torch.rand(B, 6, device="cuda", generator=g) * 2 - 1
        no, r, d = rb.step(a)
        raw.step_tensor(a)
        obs, rew, done = raw.obs_t.cpu().numpy(), raw.reward_t.cpu().numpy(), raw.done_t.cpu().numpy().astype(bool)
        eo, _ = vn.step(obs.astype(np.float64), rew, done)
        assert np.allclose(no.cpu().numpy(), eo, atol=2e-6), t
        assert np.array_equal(r.cpu().numpy(), rew) and np.array_equal(d.cpu().numpy().astype(bool), done)
        st = rb.stats.cpu().numpy()
        assert np.allclose(st[:-1, 0], vn.obs_rms.mean, rtol=1e-9, atol=1e-9) and np.allclose(st[:-1, 1], vn.obs_rms.var, rtol=1e-7, atol=1e-12)
        assert abs(st[-1, 0] - vn.ret_rms.mean) <= 1e-10 and abs(st[-1, 1] - vn.ret_rms.var) <= 1e-9 * vn.ret_rms.var
        assert st[0, 2] == vn.obs_rms.count
        last = store_transition(ref, last, raw, a)
        n_done += int(done.sum())
        assert rb.size == ref.size() and rb.full == ref.full
        if t in (0, 2, 4, 5, 9, 14):
            s = rb.sample(n, indices_out=idx)
            got = idx.cpu().numpy()
            assert np.array_equal(got, replay_draws(seed, calls, n, ref.size(), B)), t
            calls += 1
            eo_, ea, eno, ed, er = ref.get_samples(got[:, 0], got[:, 1], vn)
            assert np.allclose(s.observations.cpu().numpy(), eo_, atol=2e-6, rtol=0), t
            assert np.allclose(s.next_observations.cpu().numpy(), eno, atol=2e-6, rtol=0), t
            assert np.array_equal(s.actions.cpu().numpy(), ea) and np.array_equal(s.dones.cpu().numpy(), ed), t
            assert np.allclose(s.rewards.cpu().numpy(), er, rtol=1e-6, atol=1e-7), t
            assert s.observations.shape == (n, env.obs_dim) and s.rewards.shape == (n, 1) and s.dones.shape == (n, 1)
            sampled_done += int(ed.sum())
    assert ref.full and n_done >= B and sampled_done > 0  # the ring wrapped; terminal transitions were stored and sampled
    rb.close(); env.close(); raw.close()


RAW_CASES = {
    "default": dict(),
    "forecast_in_the_middle": dict(observation_modules=["IndoorClimateObservations", "WeatherForecastObservations", "TimeObservations",
                                                        "ControlObservations"]),
    "no_forecast": dict(observation_modules=["IndoorClimateObservations", "BasicCropObservations", "ControlObservations",
                                             "WeatherObservations"]),
    "state_observations": dict(observation_modules=["StateObservations", "IndoorClimateObservations", "WeatherForecastObservations"]),
    "two_tables": dict(base_env_params=dict(SHORT, start_train_day=0, end_train_day=1)),
    "no_auto_reset": dict(auto_reset=False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(RAW_CASES))
def test_replay_raw_rows_are_bit_exact(case):
    """Without normalisation every sampled observation / next observation is, bit for bit, the row the env produced -- terminal
    rows included -- although the buffer stored it without its forecast block."""
    from glgym.replay import DeviceReplayBuffer
    from glgym.vec_env import GreenLightVecEnv
    B, cap, steps = 64, 8, 20
    kw = dict(n_sub=60, integrator="fixed", seed=3, base_env_params=SHORT)
    kw.update(RAW_CASES[case])
    auto_reset = kw.get("auto_reset", True)
    if not auto_reset:
        # a table of exactly N + Np + 1 rows, so stepping past N = 7 reaches the clamp kw = rows - Np - 1
        from glgym.weather import load_weather_data
        kw["weather_tables"] = load_weather_data(None, "Bleiswijk", "GL", 2009, 0, SHORT["season_length"], 49, 900, 10)[:7 + 48 + 1]
    env = GreenLightVecEnv(B, **kw)
    rb = DeviceReplayBuffer(env, cap * B, norm_obs=False, norm_reward=False, seed=4)
    ref = NpReplayBuffer(cap * B, B, env.obs_dim)
    last = rb.reset().cpu().numpy().copy()
    assert np.array_equal(last, env.obs_t.cpu().numpy())  # norm_obs off: the current observation is the raw row
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    n_done, switched = 0, False
    n = 4096
    idx = torch.empty((n, 2), dtype=torch.int32, device="cuda")
    for t in range(steps):
        a = torch.rand(B, 6, device="cuda", generator=g) * 2 - 1
        tb = env.table_t.cpu().numpy().copy()
        rb.step(a)
        last = store_transition(ref, last, env, a, auto_reset)
        done = env.done_t.cpu().numpy().astype(bool)
        n_done += int(done.sum())
        switched |= bool((done & (env.table_t.cpu().numpy() != tb)).any())
        if t in (5, 12, steps - 1):
            s = rb.sample(n, indices_out=idx)
            got = idx.cpu().numpy()
            eo, ea, eno, ed, er = ref.get_samples(got[:, 0], got[:, 1])
            assert np.array_equal(s.observations.cpu().numpy().view(np.uint32), eo.view(np.uint32)), (case, t)
            assert np.array_equal(s.next_observations.cpu().numpy().view(np.uint32), eno.view(np.uint32)), (case, t)
            assert np.array_equal(s.actions.cpu().numpy(), ea) and np.array_equal(s.dones.cpu().numpy(), ed)
            assert np.array_equal(s.rewards.cpu().numpy().view(np.uint32), er.view(np.uint32))
    assert n_done > 0
    if case == "two_tables":
        assert env.weather_tables.shape[0] == 2 and switched  # some env was reset in place into the other table
    if case == "no_auto_reset":
        # stepped past N: the forecast rows of the last observations are clamped to the end of the table
        rows = env.weather_tables.shape[1]
        assert int(env.timestep_t.max().item()) - 1 > rows - env.Np - 1
    rb.close(); env.close()


@pytest.mark.gpu
def test_replay_fences():
    from glgym import _lib
    from glgym.replay import DeviceReplayBuffer
    from glgym.vec_env import GreenLightVecEnv
    B = 32
    env = GreenLightVecEnv(B, n_sub=60, integrator="fixed", base_env_params=SHORT)
    a = torch.zeros(B, 6, device="cuda")
    with pytest.raises(_lib.GlgError):
        DeviceReplayBuffer(env, 0)
    with pytest.raises(_lib.GlgError):
        DeviceReplayBuffer(env, 100, gamma=1.5)
    rb = DeviceReplayBuffer(env, 4 * B)
    with pytest.raises(_lib.GlgError, match="empty"):
        rb.sample(8)  # before reset
    with pytest.raises(_lib.GlgError, match="before glg_replay_reset"):
        rb.store(a)
    rb.reset()
    with pytest.raises(_lib.GlgError, match="empty"):
        rb.sample(8)  # reset, nothing stored
    rb.step(a)
    with pytest.raises(ValueError):
        rb.sample(0)
    f = torch.empty(8 * env.obs_dim, device="cuda")
    assert env._lib.glg_replay_sample(rb._r, 0, *([f.data_ptr()] * 5), None, None) == _lib.GLG_ERR_ARG
    assert rb.sample(8).observations.shape == (8, env.obs_dim) and rb.size == 1
    # a new weather bank invalidates the stored forecast keys
    W = env.weather_tables
    _lib.check(env._lib.glg_set_weather(env._h, W.ctypes.data, W.shape[0], W.shape[1], env.table_start_days.ctypes.data), env._h, "glg_set_weather")
    with pytest.raises(_lib.GlgError, match="weather bank"):
        rb.store(a)
    with pytest.raises(_lib.GlgError, match="weather bank"):
        rb.sample(8)
    rb2 = DeviceReplayBuffer(env, 4 * B)  # a buffer created under the new bank works
    rb2.reset()
    rb2.step(a)
    assert rb2.sample(8).dones.shape == (8, 1)
    rb.close()
    with pytest.raises(RuntimeError):
        rb.sample(8)
    env.close()
    with pytest.raises(RuntimeError, match="env"):
        rb2.sample(8)
    rb2.close()  # after its env: frees only the buffer's own memory


@pytest.mark.gpu
def test_replay_buffers_are_independent_and_seeded():
    from glgym.replay import DeviceReplayBuffer
    from glgym.vec_env import GreenLightVecEnv
    B = 64
    env = GreenLightVecEnv(B, n_sub=60, integrator="fixed", base_env_params=SHORT)
    r1, r2, r3 = (DeviceReplayBuffer(env, 6 * B, seed=s) for s in (7, 7, 8))
    env.reset_tensor()
    for r in (r1, r2, r3):
        r.reset(reset_env=False)
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    for t in range(9):
        a = torch.rand(B, 6, device="cuda", generator=g) * 2 - 1
        env.step_tensor(a)
        for r in (r1, r2, r3):
            r.store(a)
    i1, i2, i3 = (torch.empty((500, 2), dtype=torch.int32, device="cuda") for _ in range(3))
    s1 = [x.clone() for x in r1.sample(500, indices_out=i1)]
    s2 = r2.sample(500, indices_out=i2)
    assert all(torch.equal(x, y) for x, y in zip(s1, s2)) and torch.equal(i1, i2)  # same seed, same stores: same samples
    s3 = r3.sample(500, indices_out=i3)
    assert not torch.equal(i1, i3) and not torch.equal(s1[1], s3.actions)  # another seed draws other transitions
    assert torch.equal(r1.stats, r2.stats) and torch.equal(r1.obs, r3.obs)
    r1.close()
    for t in range(3):  # the others keep working after one is closed
        a = torch.rand(B, 6, device="cuda", generator=g) * 2 - 1
        env.step_tensor(a)
        r2.store(a)
        r3.store(a)
    assert r2.size == r3.size == 6 and r2.full
    assert bool(torch.isfinite(r2.sample(256).observations).all()) and bool(torch.isfinite(r3.sample(256).next_observations).all())
    with pytest.raises(RuntimeError):
        r1.store(a)
    r2.close(); r3.close(); env.close()


@pytest.mark.gpu
def test_replay_bytes_against_raw_rows():
    """At the default stack the compressed buffer holds at most 1/8 of SB3's raw-row layout (observations and next_observations
    float32 [cap][B][obs_dim], actions [cap][B][6], rewards / dones / timeouts float32 [cap][B])."""
    from glgym.replay import DeviceReplayBuffer
    from glgym.vec_env import GreenLightVecEnv
    B = 256
    env = GreenLightVecEnv(B, n_sub=60, integrator="fixed")
    rb = DeviceReplayBuffer(env, 100 * B)
    raw = rb.capacity * B * (2 * env.obs_dim * 4 + 6 * 4 + 3 * 4)
    assert env.obs_dim == 263 and rb.nbytes <= raw / 8, (rb.nbytes, raw)
    rb.close(); env.close()
