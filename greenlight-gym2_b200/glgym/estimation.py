"""DeviceStateEstimator -- an unscented Kalman filter (UKF) that estimates every env's 28-state from its observations, on the device
(csrc/glg_est.cuh behind glg_est_* in include/glgym.h).  A greenhouse controller measures air temperature, CO2, humidity and pipe
temperature and tracks the crop through proxies; the cover, screen, floor, soil and top-compartment temperatures and the crop's
carbohydrate pools are never observed.  The filter turns the observations into a state estimate and its covariance, so a
model-based controller can run on what a real one would know:

    env = GreenLightVecEnv(B, uncertainty_scale=0.2)
    est = DeviceStateEstimator(env)
    planner = DevicePlanner(env, horizon=12, n_candidates=256, n_elites=32, n_iterations=3)
    env.reset_tensor(); est.reset()
    for step in range(...):
        env.step_tensor(planner.plan(est.mean))          # MPC on the estimate (output feedback)
        est.update(est.measurements() + sensor_noise)    # predict over the step just taken, then update
        planner.shift()

Each update propagates the 57 sigma points of every env through one control interval of the nominal model with the step kernels
(one glg_step_raw_control of an internal handle of 57 B envs), with the controls the env just applied and the weather row it read.
An env that finished under auto-reset restarts the filter from its new state, init_state(d0), a known function of the weather
table rather than privileged information.

Defaults (per state, in the model's units; x27 is the deterministic day counter and gets 0 everywhere):
- p0_std: 1 K for every temperature, 50 mg m^-3 for the CO2 concentrations (about 28 ppm), 100 Pa for the vapour pressures (about
  5 % RH at 20 C), and 5 % of the reset state for the crop pools cLeaf, cStem, cFruit and tSum (cBuf starts at 0: 1000 mg m^-2).
- q_std: the per-state standard deviation of the nominal model's one-step error against envs with uncertainty_scale = 0.1 under
  the rule-based controller, measured with tools/estimate_q.py (DESIGN.md, "State estimation").
- r_std: sensor-like values: 20 ppm CO2, 0.2 K air temperature, 2 % RH, 0.5 K pipe and 24 h canopy temperature, 1 % of the reset
  fruit weight (553 mg m^-2) and 10 C d for the temperature sum.

DeviceStateSmoother -- an unscented Rauch-Tung-Striebel smoother over the estimator's last `window` estimates
(csrc/glg_smooth.cuh behind glg_smooth_* in include/glgym.h).  The filter's estimate at step k uses the observations up to k; the
smoothed one uses every observation in the window, which is what analysing a logged season or an EM fit of the noise wants:

    smoother = DeviceStateSmoother(est, window=192)   # records from the estimator's next reset on
    est.reset()
    for step in range(192):
        env.step_rule_based_tensor()
        est.update(est.measurements() + sensor_noise)
    s = smoother.smooth()                             # s.mean [L, B, 28], s.cov and s.gain [L, B, 28, 28], oldest first
"""
import collections
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .vec_env import OBSERVATION_MODULES, _EnvCompanion

# h(x): the seven state-dependent observation entries, in glg_obs_head order, and the observation module each is read from
MEASUREMENT_NAMES = ("co2_air", "temp_air", "rh_air", "pipe_temp", "24CanTemp", "cFruit", "tSum")
_SOURCE = [("IndoorClimateObservations", 0), ("IndoorClimateObservations", 1), ("IndoorClimateObservations", 2),
           ("IndoorClimateObservations", 3), ("BasicCropObservations", 0), ("BasicCropObservations", 1), ("BasicCropObservations", 2)]
MAX_SIGMA_POINTS = 4194304  # num_envs * 57: the largest batch the step kernels were run at

_TEMPS = (2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 17, 18, 19, 20, 21)
_P0 = np.zeros(28)
_P0[list(_TEMPS)] = 1.0
_P0[[0, 1]] = 50.0
_P0[[15, 16]] = 100.0
_P0[22] = 1000.0
_P0[[23, 24, 25, 26]] = 0.05 * np.array([9.5283e4, 2.5107e5, 5.5338e4, 3.0978e3])
DEFAULT_P0_STD = tuple(float(v) for v in _P0)
# tools/estimate_q.py: 256 envs (uncertainty_scale 0.1, the default weather tables), rule-based, 960 steps: 245 760 one-step errors
DEFAULT_Q_STD = (4.36, 3.733, 0.01738, 0.01204, 0.02273, 0.008972, 0.008528, 0.003531, 0.006428, 0.00216, 0.001275, 4.147e-05,
                 2.514e-07, 3.001e-10, 7.489e-14, 4.646, 4.01, 0.01846, 7.105e-15, 0.0008623, 0.009966, 0.0002232, 24.17, 156.9,
                 2.056, 8.163, 0.0002243, 0.0)  # x27, the day counter, is deterministic: its 4e-15 is rounding
DEFAULT_R_STD = (20.0, 0.2, 2.0, 0.5, 0.5, 553.38, 10.0)


def _std_vector(v, n, name):
    a = np.asarray(v, dtype=np.float64).reshape(-1)
    if a.shape != (n,):
        raise ValueError(f"{name} must hold {n} values")
    if not np.all(np.isfinite(a)) or np.any(a < 0):
        raise ValueError(f"{name} must be finite and >= 0")
    return a


def _measured_indices(measured):
    if measured is None:
        return list(range(7))
    items = [measured] if isinstance(measured, (str, int)) else list(measured)
    idx = []
    for m in items:
        if isinstance(m, str):
            if m not in MEASUREMENT_NAMES:
                raise ValueError(f"unknown measurement {m!r}; choose from {MEASUREMENT_NAMES}")
            m = MEASUREMENT_NAMES.index(m)
        elif not (isinstance(m, (int, np.integer)) and 0 <= int(m) < 7):
            raise ValueError(f"measured entries are names out of {MEASUREMENT_NAMES} or indices 0..6; got {m!r}")
        idx.append(int(m))
    if not idx or len(set(idx)) != len(idx):
        raise ValueError("measured must name at least one entry, each once")
    return sorted(idx)


class DeviceStateEstimator(_EnvCompanion):
    _kind, _destroy = "estimator", "glg_est_destroy"
    _e = property(lambda self: self._obj)  # the glg_est object, for calling the C entry points directly

    def __init__(self, env, p0_std=None, q_std=None, r_std=None, measured=None, alpha=1.0, beta=2.0, kappa=0.0):
        p0 = _std_vector(DEFAULT_P0_STD if p0_std is None else p0_std, 28, "p0_std")
        q = _std_vector(DEFAULT_Q_STD if q_std is None else q_std, 28, "q_std")
        r = _std_vector(DEFAULT_R_STD if r_std is None else r_std, 7, "r_std")
        idx = _measured_indices(measured)
        if any(r[i] <= 0 for i in idx):
            raise ValueError("r_std must be > 0 for every measured entry")
        alpha, beta, kappa = float(alpha), float(beta), float(kappa)
        if not (alpha > 0 and math.isfinite(alpha)) or not (beta >= 0 and math.isfinite(beta)) or not math.isfinite(kappa):
            raise ValueError("need alpha > 0, beta >= 0 and a finite kappa")
        if not alpha * alpha * (28 + kappa) > 0:
            raise ValueError("need n + lambda = alpha^2 (28 + kappa) > 0")
        B = int(env.num_envs)
        if B * 57 > MAX_SIGMA_POINTS:
            raise ValueError(f"num_envs * 57 = {B * 57} sigma points exceed {MAX_SIGMA_POINTS}")
        cfg = _lib.GlgEstConfig()
        cfg.alpha, cfg.beta, cfg.kappa = alpha, beta, kappa
        cfg.meas_mask = sum(1 << i for i in idx)
        for i in range(28):
            cfg.p0_std[i], cfg.q_std[i] = float(p0[i]), float(q[i])
        for i in range(7):
            cfg.r_std[i] = float(r[i])
        super().__init__(env, "glg_est_create", cfg)
        self.measured = [MEASUREMENT_NAMES[i] for i in idx]
        self.p0_std, self.q_std, self.r_std = p0, q, r
        e, L = self._obj, self._lib
        self.mean = self._view(L.glg_est_mean_dev(e), (28, B), "<f8").t()        # [B, 28] view of the [28][B] estimate
        self.cov = self._view(L.glg_est_cov_dev(e), (B, 28, 28), "<f8")
        self.innovation = self._view(L.glg_est_innovation_dev(e), (B, 7), "<f8")  # y - ybar; 0 where not measured / updated
        self.status = self._view(L.glg_est_status_dev(e), (B,), "|u1")
        self.sigma = self._view(L.glg_est_sigma_dev(e), (28, B, 57), "<f8")      # propagated sigma points [state][env][point]
        self._y = None

    def reset(self, x0=None):
        """Starts every env's filter: mean <- x0 (float64 [B, 28]; None = the env's current state, e.g. right after the env's
        reset, where the state is init_state(d0) of its weather table), cov <- diag(p0_std^2)."""
        e = self._live()
        ptr, keep = 0, None
        if x0 is not None:
            keep = torch.as_tensor(x0, dtype=torch.float64, device=self.env.device)
            if tuple(keep.shape) != (self.env.num_envs, 28):
                raise ValueError(f"x0 must have shape [{self.env.num_envs}, 28]")
            keep = keep.t().contiguous()
            ptr = keep.data_ptr()
        _lib.check(self._lib.glg_est_reset(e, ptr, self.env._stream()), self.env._h, "glg_est_reset")

    def update(self, y=None):
        """After each env step: predict over the interval the env just took, then update with y (float64 [B, 7] in
        MEASUREMENT_NAMES order; unmeasured columns are not read), or predict only when y is None."""
        e = self._live()
        ptr = 0
        if y is not None:
            yy = torch.as_tensor(y, dtype=torch.float64, device=self.env.device)
            if tuple(yy.shape) != (self.env.num_envs, 7):
                raise ValueError(f"y must have shape [{self.env.num_envs}, 7]")
            self._y = yy.contiguous()  # kept alive until the next update: the kernels read it asynchronously
            ptr = self._y.data_ptr()
        _lib.check(self._lib.glg_est_update(e, ptr, self.env._stream()), self.env._h, "glg_est_update")

    def measurements(self, obs=None):
        """The 7 measurement entries as float64 [B, 7] read from an observation batch (default: the env's current obs_t), zeros in
        unmeasured columns.  Raises ValueError when the env's observation stack lacks a module a measured entry comes from."""
        env = self.env
        mods = env.observation_modules
        sizes = [len(OBSERVATION_MODULES[m][1]) if OBSERVATION_MODULES[m][1] is not None else 5 * env.Np for m in mods]
        offsets = dict(zip(mods, np.cumsum([0] + sizes[:-1])))
        o = env.obs_t if obs is None else torch.as_tensor(obs, device=env.device)
        y = torch.zeros((o.shape[0], 7), dtype=torch.float64, device=env.device)
        for name in self.measured:
            mod, col = _SOURCE[MEASUREMENT_NAMES.index(name)]
            if mod not in offsets:
                raise ValueError(f"the observation stack has no {mod}, which {name} is read from")
            j = MEASUREMENT_NAMES.index(name)
            y[:, j] = o[:, int(offsets[mod]) + col].to(torch.float64)
        return y



Smoothed = collections.namedtuple("Smoothed", "mean cov gain")


class DeviceStateSmoother(_EnvCompanion):
    """Records every glg_est_reset / glg_est_update of `est` into a ring of `window` slots per env and smooths the valid slots on
    demand.  Recording does not change the estimator's outputs.  Keeps the estimator alive; close the smoother before closing the
    estimator explicitly."""
    _kind, _destroy = "smoother", "glg_smooth_destroy"

    def __init__(self, est, window):
        if isinstance(window, bool) or not isinstance(window, (int, np.integer)) or int(window) < 2:
            raise ValueError("window must be an integer >= 2")
        if not isinstance(est, DeviceStateEstimator):
            raise TypeError("est must be a DeviceStateEstimator")
        W, B = int(window), int(est.env.num_envs)
        self.est, self.env, self._lib, self.window = est, est.env, est._lib, W
        self._obj = C.c_void_p()
        _lib.check(self._lib.glg_smooth_create(est._live(), W, C.byref(self._obj)), self.env._h, "glg_smooth_create")
        s, L = self._obj, self._lib
        mean = lambda ptr: self._view(ptr, (W, 28, B), "<f8").permute(0, 2, 1)  # [W, B, 28] view of [W][28][B]
        mat = lambda ptr: self._view(ptr, (W, B, 28, 28), "<f8")
        self._out = Smoothed(mean(L.glg_smooth_mean_dev(s)), mat(L.glg_smooth_cov_dev(s)), mat(L.glg_smooth_gain_dev(s)))
        self._rec = {"filtered_mean": mean(L.glg_smooth_filtered_mean_dev(s)), "filtered_cov": mat(L.glg_smooth_filtered_cov_dev(s)),
                     "prior_mean": mean(L.glg_smooth_prior_mean_dev(s)), "prior_cov": mat(L.glg_smooth_prior_cov_dev(s)),
                     "cross_cov": mat(L.glg_smooth_cross_dev(s)),
                     "status": self._view(L.glg_smooth_status_dev(s), (W, B), "|u1"),
                     "timestep": self._view(L.glg_smooth_timestep_dev(s), (W, B), "<i4")}
        self.bytes = int(L.glg_smooth_bytes(s))

    def _live(self):
        self.est._live()
        return super()._live()

    @property
    def length(self):
        """The number of valid slots: min(estimates recorded since the estimator's last reset, window)."""
        return int(self._lib.glg_smooth_length(self._live()))

    def smooth(self):
        """Runs the backward pass and returns Smoothed(mean [L, B, 28], cov [L, B, 28, 28], gain [L, B, 28, 28]), float64 views
        of the smoother's output, oldest first (L = length).  gain[k] is G_k; it is 0 at the last slot of a segment, and
        cov[k + 1] @ gain[k].transpose(-1, -2) is the lag-one cross-covariance."""
        s = self._live()
        _lib.check(self._lib.glg_smooth_run(s, self.env._stream()), self.env._h, "glg_smooth_run")
        n = self.length
        return Smoothed(*(v[:n] for v in self._out))

    def _rolled(self, name):
        """A recorded quantity, oldest first (a copy: the record is a ring)."""
        s = self._live()
        n, first = self.length, int(self._lib.glg_smooth_first(s))
        return torch.roll(self._rec[name], -first, 0)[:n]

    filtered_mean = property(lambda self: self._rolled("filtered_mean"), doc="x^ [L, B, 28]: the estimator's means")
    filtered_cov = property(lambda self: self._rolled("filtered_cov"), doc="P [L, B, 28, 28]: the estimator's covariances")
    prior_mean = property(lambda self: self._rolled("prior_mean"), doc="xbar [L, B, 28]; 0 where no prediction leads to the slot")
    prior_cov = property(lambda self: self._rolled("prior_cov"), doc="P- [L, B, 28, 28]; 0 where no prediction leads to the slot")
    cross_cov = property(lambda self: self._rolled("cross_cov"), doc="D [L, B, 28, 28]: sum Wc (chi - x^)(chi' - xbar)^T")
    status = property(lambda self: self._rolled("status"), doc="[L, B] the estimator's status bits of each slot")
    timestep = property(lambda self: self._rolled("timestep"), doc="[L, B] the env's timestep of each slot")
