"""DevicePlanner -- a model-predictive controller for the batched env: receding-horizon planning by the cross-entropy method (CEM),
with every candidate action sequence scored by the env's own step kernels and reward (csrc/glg_plan.cuh behind glg_plan_* in
include/glgym.h).  Each decision simulates n_candidates sequences of `horizon` steps from every env's current state, n_iterations
times, on a second handle of B * n_candidates planning envs; the env itself is only read.

    planner = DevicePlanner(env, horizon=12, n_candidates=256, n_elites=32, n_iterations=3)
    env.reset_tensor()
    for step in range(...):
        a = planner.plan()          # float32 [B, 6] in [-1, 1]
        env.step_tensor(a)
        planner.shift()             # warm start of the next decision

The planner uses the nominal model (no parametric uncertainty) and the weather bank as perfect weather over the horizon, which is
the forecast the env observes as long as horizon <= Np.  `evaluate(seq)` scores caller-supplied sequences the same way.
`plan(x)` plans from given states instead of the env's, e.g. a DeviceStateEstimator's estimate (output-feedback MPC).
"""
import torch

from . import _lib
from .vec_env import _EnvCompanion


class DevicePlanner(_EnvCompanion):
    _kind, _destroy = "planner", "glg_plan_destroy"
    _p = property(lambda self: self._obj)  # the glg_plan object, for calling the C entry points directly

    def __init__(self, env, horizon, n_candidates, n_elites, n_iterations, gamma=1.0, init_std=0.5, seed=0):
        cfg = _lib.GlgPlanConfig(int(horizon), int(n_candidates), int(n_elites), int(n_iterations), float(gamma), float(init_std),
                                 int(seed) & (2**64 - 1))
        super().__init__(env, "glg_plan_create", cfg)
        self.horizon, self.n_candidates, self.n_elites, self.n_iterations = int(horizon), int(n_candidates), int(n_elites), int(n_iterations)
        H, B, K, p, L = self.horizon, env.num_envs, self.n_candidates, self._obj, self._lib
        self.mean = self._view(L.glg_plan_mean_dev(p), (H, B, 6), "<f4")               # writeable: re-initialise the distribution
        self.std = self._view(L.glg_plan_std_dev(p), (H, B, 6), "<f4")
        self.candidates = self._view(L.glg_plan_candidates_dev(p), (H, B, K, 6), "<f4")  # last iteration's samples
        self.returns = self._view(L.glg_plan_returns_dev(p), (B, K), "<f8")              # last roll-out's discounted returns
        self._actions = torch.empty((B, 6), dtype=torch.float32, device=env.device)

    def plan(self, x=None):
        """One decision: n_iterations CEM iterations from the env's current states, or from the states x (a float64 CUDA [B, 28]
        tensor, e.g. a DeviceStateEstimator's `mean`, which is used without a copy; the env's controls, clock and timestep still
        apply).  Returns the new mean[0] as a float32 [B, 6] tensor (overwritten by the next plan())."""
        p = self._live()
        if x is None:
            _lib.check(self._lib.glg_plan_run(p, self._actions.data_ptr(), self.env._stream()), self.env._h, "glg_plan_run")
            return self._actions
        B = self.env.num_envs
        if not (isinstance(x, torch.Tensor) and x.dtype == torch.float64 and x.device == self.env.device and tuple(x.shape) == (B, 28)):
            raise ValueError(f"x must be a float64 tensor of shape [{B}, 28] on {self.env.device}")
        xs = x.t()  # the C side reads [28][B]
        if not xs.is_contiguous():
            xs = xs.contiguous()
        _lib.check(self._lib.glg_plan_run_from(p, xs.data_ptr(), self._actions.data_ptr(), self.env._stream()), self.env._h,
                   "glg_plan_run_from")
        return self._actions

    def shift(self):
        """Moves the horizon one step on: mean[t] <- mean[t + 1], mean[H - 1] <- 0 (hold the controls), std <- init_std."""
        _lib.check(self._lib.glg_plan_shift(self._live(), self.env._stream()), self.env._h, "glg_plan_shift")

    def evaluate(self, seq):
        """Discounted returns of caller-supplied sequences from the env's current states: seq float32 [H, B * K, 6] (or
        [H, B, K, 6]), candidate c = b * K + k starting from env b.  Returns the `returns` view, float64 [B, K]."""
        p = self._live()
        H, BK = self.horizon, self.env.num_envs * self.n_candidates
        s = seq.to(device=self.env.device, dtype=torch.float32).contiguous()
        if s.numel() != H * BK * 6:
            raise ValueError(f"seq must hold [{H}, {BK}, 6] actions")
        _lib.check(self._lib.glg_plan_evaluate(p, s.data_ptr(), self.returns.data_ptr(), self.env._stream()), self.env._h,
                   "glg_plan_evaluate")
        return self.returns
