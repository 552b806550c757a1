"""Lifetime of the C objects (csrc/glg_capi.cu): an env and its companions free every device allocation when destroyed, in
either order, and a setter that rejects its input leaves the env exactly as it was."""
import gc

import numpy as np
import pytest

torch = pytest.importorskip("torch")

SHORT2 = dict(season_length=7 / 96.0, start_train_day=0, end_train_day=1)  # N = 7, two weather tables


def _env(B, **kw):
    from glgym.vec_env import GreenLightVecEnv
    base = dict(seed=3, n_sub=30, base_env_params=SHORT2)
    base.update(kw)
    return GreenLightVecEnv(B, **base)


def _free_bytes():
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def _round(companions_first):
    """One env of 4096 with a rollout, a 2^20-transition replay buffer and a small planner, each used once, then destroyed."""
    from glgym.planning import DevicePlanner
    from glgym.replay import DeviceReplayBuffer
    from glgym.rollout import DeviceRollout
    B = 4096
    env = _env(B)
    roll = DeviceRollout(env, n_steps=2)
    rb = DeviceReplayBuffer(env, 2**20)
    planner = DevicePlanner(env, horizon=2, n_candidates=8, n_elites=2, n_iterations=1)
    assert rb.nbytes > 200 << 20
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    roll.reset()
    roll.step(torch.rand(B, 6, device="cuda", generator=g) * 2 - 1)
    roll.step(torch.rand(B, 6, device="cuda", generator=g) * 2 - 1)
    roll.finish(torch.zeros(3, B, device="cuda"))
    rb.reset()
    rb.step(torch.rand(B, 6, device="cuda", generator=g) * 2 - 1)
    rb.sample(256)
    a = planner.plan()
    assert bool(torch.isfinite(a).all())
    torch.cuda.synchronize()
    objs = [roll, rb, planner]
    if companions_first:
        for o in objs:
            o.close()
        env.close()
    else:
        env.close()
        for o in objs:
            o.close()


@pytest.mark.gpu
def test_create_destroy_rounds_return_all_device_memory():
    _round(True)  # warm-up: module loads, the step kernels' local memory, torch's own buffers
    base = _free_bytes()
    for i in range(20):
        _round(i % 2 == 0)
        free = _free_bytes()
        assert abs(free - base) <= 8 << 20, (i, (base - free) / 2**20)


@pytest.mark.gpu
def test_rejected_bank_setters_leave_the_env_unchanged():
    from glgym import _lib
    B = 64
    env, twin = _env(B, seed=5), _env(B, seed=5)
    L = env._lib
    short = np.zeros((1, 3, 10))
    assert L.glg_set_weather(env._h, short.ctypes.data, 1, 3, None) == _lib.GLG_ERR_ARG
    assert b"rows < N + Np + 1" in L.glg_last_error(env._h)
    n_tables = env.weather_tables.shape[0]
    ids = np.array([0, n_tables], dtype=np.int32)
    assert L.glg_set_reset_tables(env._h, ids.ctypes.data, 2) == _lib.GLG_ERR_ARG
    assert b"id out of range" in L.glg_last_error(env._h)
    env.reset_tensor()
    twin.reset_tensor()
    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    for _ in range(20):  # N = 7: every env auto-resets twice, drawing from the reset-table list
        a = torch.rand(B, 6, device="cuda", generator=g) * 2 - 1
        o1, r1, d1 = env.step_tensor(a)
        o2, r2, d2 = twin.step_tensor(a)
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2)
        assert torch.equal(env.state_t, twin.state_t) and torch.equal(env.table_t, twin.table_t)
    env.close()
    twin.close()
