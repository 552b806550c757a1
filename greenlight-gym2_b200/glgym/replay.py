"""DeviceReplayBuffer -- the off-policy half of the reference's training pipeline, `VecNormalize(VecMonitor(SubprocVecEnv))` + SB3's
`ReplayBuffer` as SAC fills it (gl_gym/RL/utils.py:60-67, RL/experiment_manager.py:174-194; SB3 2.6.0
OffPolicyAlgorithm._store_transition, common/buffers.py ReplayBuffer with optimize_memory_usage=False), as CUDA kernels on the env
handle's outputs (csrc/glg_replay.cuh behind glg_replay_* in include/glgym.h).  Nothing leaves the device.

    rb = DeviceReplayBuffer(env, buffer_size=1_000_000)
    obs = rb.reset()                               # normalised current observation [B, obs_dim]
    for step in range(...):
        actions = policy(obs)                      # in [-1, 1]
        obs, reward, done = rb.step(actions)       # env step + VecNormalize statistics + the transition into the ring
        batch = rb.sample(256)                     # ReplayBufferSamples of torch tensors on the env's device

Transitions are stored without their WeatherForecastObservations block (240 of the default row's 263 floats), which the sample
kernel rebuilds from the env's weather bank: 221 B per transition at the default stack instead of 2140 B.  Differences from SB3:
the next observation of an env that finished is the raw terminal row (SB3 stores unnormalize(normalize(row)), equal up to float32
rounding except in columns clipped at +-clip_obs), and the sample indices come from device Philox keyed by `seed` instead of numpy's
global generator.  Replacing the env's weather bank (glg_set_weather) invalidates the buffer.
"""
import collections

import torch

from . import _lib
from .vec_env import _EnvCompanion

# SB3 common/type_aliases.py ReplayBufferSamples: field names and order
ReplayBufferSamples = collections.namedtuple("ReplayBufferSamples", ["observations", "actions", "next_observations", "dones", "rewards"])


class DeviceReplayBuffer(_EnvCompanion):
    _kind, _destroy = "replay buffer", "glg_replay_destroy"
    _r = property(lambda self: self._obj)  # the glg_replay object, for calling the C entry points directly

    def __init__(self, env, buffer_size, gamma=0.99, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, epsilon=1e-8,
                 training=True, seed=0):
        cfg = _lib.GlgReplayConfig(int(buffer_size), int(training), int(norm_obs), int(norm_reward), 0, float(gamma), float(clip_obs),
                                   float(clip_reward), float(epsilon), int(seed) & (2**64 - 1))
        super().__init__(env, "glg_replay_create", cfg)
        B, D, r, L = env.num_envs, env.obs_dim, self._obj, self._lib
        self.capacity = max(int(buffer_size) // B, 1)
        self.obs = self._view(L.glg_replay_obs_dev(r), (B, D), "<f4")          # normalised current observation
        self.stats = self._view(L.glg_replay_stats_dev(r), (D + 1, 3), "<f8")  # running (mean, var, count); last row: returns
        self._out = {}  # n -> output tensors of sample(n), reused by the next sample(n)

    def reset(self, reset_env=True):
        """Resets every env and starts each env's next transition from its new observation; stored transitions are kept.
        reset_env=False: the caller has just reset the env itself (e.g. for another buffer on the same env)."""
        r = self._live()
        if reset_env:
            self.env.reset_tensor()
        _lib.check(self._lib.glg_replay_reset(r, self.env._stream()), self.env._h, "glg_replay_reset")
        return self.obs

    def store(self, actions):
        """Adds the transition of the env step that just ran (any step_*_tensor of the env); actions: float32 [B, 6] to store."""
        r = self._live()
        a = actions.to(device=self.env.device, dtype=torch.float32).contiguous()
        _lib.check(self._lib.glg_replay_store(r, a.data_ptr(), self.env._stream()), self.env._h, "glg_replay_store")

    def step(self, actions, noise=None):
        """env.step_tensor(actions) + store(actions).  Returns (normalised obs, raw reward [B] f64, done [B] u8), device views."""
        self._live()
        a = actions.to(device=self.env.device, dtype=torch.float32).contiguous()
        _, reward, done = self.env.step_tensor(a, noise)
        self.store(a)
        return self.obs, reward, done

    def sample(self, n, indices_out=None):
        """ReplayBuffer.sample(n) behind VecNormalize: observations / next_observations [n, obs_dim] normalised and clipped,
        actions [n, 6], rewards [n, 1] normalised and clipped, dones [n, 1].  The tensors are reused by the next sample of the same
        n.  indices_out: optional int32 [n, 2] device tensor that receives the drawn (slot, env) pairs."""
        r = self._live()
        n = int(n)
        if n < 1:
            raise ValueError("sample(n) needs n >= 1")
        out = self._out.get(n)
        if out is None:
            dev, D = self.env.device, self.env.obs_dim
            f = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
            out = self._out[n] = ReplayBufferSamples(f(n, D), f(n, 6), f(n, D), f(n, 1), f(n, 1))
        idx = 0
        if indices_out is not None:
            if indices_out.dtype != torch.int32 or indices_out.device != self.env.device or not indices_out.is_contiguous() or \
                    tuple(indices_out.shape) != (n, 2):
                raise ValueError("indices_out must be a contiguous int32 [n, 2] tensor on the env's device")
            idx = indices_out.data_ptr()
        _lib.check(self._lib.glg_replay_sample(r, n, out.observations.data_ptr(), out.next_observations.data_ptr(), out.actions.data_ptr(),
                                               out.rewards.data_ptr(), out.dones.data_ptr(), idx, self.env._stream()),
                   self.env._h, "glg_replay_sample")
        return out

    @property
    def size(self):
        """Valid slots per env (SB3 ReplayBuffer.size())."""
        return int(self._lib.glg_replay_size(self._live()))

    @property
    def full(self):
        return self.size == self.capacity

    @property
    def nbytes(self):
        """Device bytes the buffer holds."""
        return int(self._lib.glg_replay_bytes(self._live()))

    def close(self):
        super().close()
        self._out = {}
