"""Device rollout as its own object (glg_rollout_* in include/glgym.h, glgym.rollout.DeviceRollout): several rollouts on one env, each
with its own buffers and statistics; the fences of a closed rollout or env.  The kernels themselves are checked against the numpy
restatement of SB3 in test_normalize.py."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

SHORT = dict(season_length=7 / 96.0)


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()


def test_rollout_entry_points_reject_null_arguments():
    """CPU tier: the C entry points fail loudly on NULL objects instead of touching memory."""
    from glgym import _lib
    lib = _lib.load()
    cfg = _lib.GlgRolloutConfig(4, 1, 1, 1, 0.99, 0.95, 10.0, 10.0, 1e-8)
    out = C.c_void_p()
    assert lib.glg_rollout_create(None, C.byref(cfg), C.byref(out)) == _lib.GLG_ERR_ARG and not out
    values = np.zeros(8, np.float32)
    assert lib.glg_rollout_store(None, 0, None) == _lib.GLG_ERR_ARG
    assert lib.glg_rollout_carry(None, None) == _lib.GLG_ERR_ARG
    assert lib.glg_rollout_gae(None, values.ctypes.data, None) == _lib.GLG_ERR_ARG
    for view in ("obs", "rewards", "starts", "advantages", "returns", "stats"):
        assert getattr(lib, f"glg_rollout_{view}_dev")(None) is None
    lib.glg_rollout_destroy(None)
    assert C.sizeof(_lib.GlgRolloutConfig) == 56


@pytest.mark.gpu
def test_rollout_buffers_are_independent():
    """Two rollouts with different n_steps and gamma on one env, both fed after every step, hold bit for bit what a single rollout
    with the same settings holds on an identical env stepped with the same actions: each has its own buffers and statistics.
    Episodes end inside the run.  After one is closed the other keeps working."""
    from glgym.rollout import DeviceRollout
    from glgym.vec_env import GreenLightVecEnv
    B = 96
    kw = dict(n_sub=60, integrator="fixed", seed=5, base_env_params=SHORT)
    settings = [dict(n_steps=4, gamma=0.9631, gae_lambda=0.947), dict(n_steps=6, gamma=0.99, gae_lambda=0.9)]
    env = GreenLightVecEnv(B, **kw)
    rolls = [DeviceRollout(env, **s) for s in settings]
    refs = [DeviceRollout(GreenLightVecEnv(B, **kw), **s) for s in settings]
    env.reset_tensor()
    for roll, ref in zip(rolls, refs):
        roll._store(-1)
        ref.reset()
        assert same_bits(roll.obs[0], ref.obs[0]) and same_bits(roll.stats, ref.stats)
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    n_done = 0

    def step(pairs):
        nonlocal n_done
        a = torch.rand(B, 6, device="cuda", generator=g) * 2 - 1
        env.step_tensor(a)
        n_done += int(env.done_t.sum().item())
        for roll, ref in pairs:
            roll._store(roll.t)  # the store half of roll.step(): the env was stepped once for both rollouts
            roll.t += 1
            ref.step(a)
            assert same_bits(roll.stats, ref.stats)
            if roll.t == roll.n_steps:
                for name in ("obs", "rewards", "episode_starts", "stats"):
                    assert same_bits(getattr(roll, name), getattr(ref, name)), name
                values = torch.randn(roll.n_steps + 1, B, device="cuda", generator=g)
                for x, y in zip(roll.finish(values), ref.finish(values)):
                    assert same_bits(x, y)
                roll.begin()
                ref.begin()

    for _ in range(12):  # three rollouts of the first, two of the second
        step(list(zip(rolls, refs)))
    assert n_done >= B
    rolls[0].close()
    refs[0].close()
    refs[0].env.close()
    for _ in range(6):
        step([(rolls[1], refs[1])])
    with pytest.raises(RuntimeError, match="closed"):
        rolls[0].step(torch.zeros(B, 6, device="cuda"))
    rolls[1].close(); refs[1].close(); refs[1].env.close(); env.close()


@pytest.mark.gpu
def test_rollout_fences():
    from glgym import _lib
    from glgym.rollout import DeviceRollout
    from glgym.vec_env import GreenLightVecEnv
    B = 32
    env = GreenLightVecEnv(B, n_sub=60, integrator="fixed", base_env_params=SHORT)
    a, values = torch.zeros(B, 6, device="cuda"), torch.zeros(5, B, device="cuda")
    for bad in (dict(n_steps=0), dict(gamma=1.5), dict(gae_lambda=-0.1), dict(clip_obs=0.0), dict(clip_reward=0.0), dict(epsilon=0.0)):
        with pytest.raises(_lib.GlgError, match="invalid n_steps"):
            DeviceRollout(env, **dict(dict(n_steps=4), **bad))
    roll, other = DeviceRollout(env, 4), DeviceRollout(env, 4)
    roll.reset()
    with pytest.raises(_lib.GlgError, match="t outside"):
        roll._store(4)
    n0 = env.launch_count()
    roll.step(a)
    roll.finish(values)
    assert env.launch_count() - n0 == 1 + 3 + 1  # step, store, GAE: all counted by the env's handle
    roll.close()
    roll.close()  # idempotent
    for call in (lambda: roll.step(a), lambda: roll.finish(values), lambda: roll.begin()):
        with pytest.raises(RuntimeError, match="closed"):
            call()
    other.reset()
    other.step(a)
    env.close()
    for call in (lambda: other.step(a), lambda: other.finish(values), lambda: other.begin()):
        with pytest.raises(RuntimeError, match="env"):
            call()
    other.close()  # after its env: frees only the rollout's own memory
