"""DeviceRollout -- the reference's `VecNormalize(VecMonitor(SubprocVecEnv))` + SB3 `RolloutBuffer` (gl_gym/RL/utils.py:60-67,
RL/experiment_manager.py:142-147, configs/agents/ppo.yml) as CUDA kernels on the env handle's own outputs
(csrc/glg_rollout.cuh behind glg_rollout_* in include/glgym.h): running observation / return statistics, normalisation and
clipping straight into the [T+1][B][obs_dim] rollout buffer, and generalised advantage estimation.  Nothing leaves the device.

    roll = DeviceRollout(env, n_steps=32, gamma=0.9631, gae_lambda=0.9470)
    obs = roll.reset()                               # normalised, slot 0
    for t in range(roll.n_steps):
        actions, values[t] = policy(obs)
        obs, reward, done = roll.step(actions)       # raw env step + statistics + normalisation; obs = slot t + 1
    values[T] = policy.value(obs)
    adv, ret = roll.finish(values)                   # GAE
    roll.begin()                                     # next rollout continues from slot T
    roll.close()                                     # frees the buffers; several rollouts may share one env

`glgym.normalize` keeps the same arithmetic as eager torch ops (the round-1 implementation, 4.5 ms per step at 65 536 envs);
the tests check both against a numpy restatement of SB3 2.6.0, which is pinned by the reference but not installed here
("unpinned against real SB3").
"""
import torch

from . import _lib
from .vec_env import _EnvCompanion


class DeviceRollout(_EnvCompanion):
    _kind, _destroy = "rollout buffer", "glg_rollout_destroy"

    def __init__(self, env, n_steps, gamma=0.99, gae_lambda=0.95, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 epsilon=1e-8, training=True):
        self.n_steps = int(n_steps)
        cfg = _lib.GlgRolloutConfig(self.n_steps, int(training), int(norm_obs), int(norm_reward), float(gamma), float(gae_lambda),
                                    float(clip_obs), float(clip_reward), float(epsilon))
        super().__init__(env, "glg_rollout_create", cfg)
        T, B, D, r, L = self.n_steps, env.num_envs, env.obs_dim, self._obj, self._lib
        self.obs = self._view(L.glg_rollout_obs_dev(r), (T + 1, B, D), "<f4")
        self.rewards = self._view(L.glg_rollout_rewards_dev(r), (T, B), "<f4")
        self.episode_starts = self._view(L.glg_rollout_starts_dev(r), (T + 1, B), "<f4")
        self.advantages = self._view(L.glg_rollout_advantages_dev(r), (T, B), "<f4")
        self.returns = self._view(L.glg_rollout_returns_dev(r), (T, B), "<f4")
        self.stats = self._view(L.glg_rollout_stats_dev(r), (D + 1, 3), "<f8")  # running (mean, var, count); last row: returns
        self.t = 0

    def _store(self, t):
        _lib.check(self._lib.glg_rollout_store(self._live(), t, self.env._stream()), self.env._h, "glg_rollout_store")

    def reset(self):
        self._live()
        self.env.reset_tensor()
        self._store(-1)
        self.t = 0
        return self.obs[0]

    def step(self, actions, noise=None):
        self._live()
        if self.t >= self.n_steps:
            raise RuntimeError("rollout buffer is full: call finish() / begin()")
        _, _, done = self.env.step_tensor(actions, noise)
        self._store(self.t)
        self.t += 1
        return self.obs[self.t], self.rewards[self.t - 1], done

    def step_rule_based(self, noise=None):
        self._live()
        _, _, done = self.env.step_rule_based_tensor(noise)
        self._store(self.t)
        self.t += 1
        return self.obs[self.t], self.rewards[self.t - 1], done

    def finish(self, values):
        """values: CUDA float32 [T+1, B] (row T = value of obs[T]).  Returns (advantages, returns) [T, B]."""
        r = self._live()
        v = values.to(device=self.env.device, dtype=torch.float32).contiguous()
        assert v.shape == (self.n_steps + 1, self.env.num_envs)
        _lib.check(self._lib.glg_rollout_gae(r, v.data_ptr(), self.env._stream()), self.env._h, "glg_rollout_gae")
        return self.advantages, self.returns

    def begin(self):
        """Continue with the next rollout: slot T becomes slot 0 (SB3 keeps `_last_obs` / `_last_episode_starts`)."""
        _lib.check(self._lib.glg_rollout_carry(self._live(), self.env._stream()), self.env._h, "glg_rollout_carry")
        self.t = 0
        return self.obs[0]

    @property
    def obs_mean(self):
        return self.stats[:-1, 0]

    @property
    def obs_var(self):
        return self.stats[:-1, 1]
