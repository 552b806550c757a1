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

DeviceNoiseEM -- an EM fit of the estimator's diagonal process and measurement noise (q_std, r_std) from the observations alone,
over a smoother's window (csrc/glg_em.cuh behind glg_em_* in include/glgym.h).  It logs, beside the smoother's record, what a replay
of the run needs (the controls, tables and measurements) and each update's log-likelihood term; its E-step steps the sigma points of
every (env, slot) transition of the window in a few wide launches:

    em = DeviceNoiseEM(smoother)                      # logs from the estimator's next reset on
    start = env.state_dict()
    est.reset()
    for step in range(192):
        env.step_rule_based_tensor()
        est.update(est.measurements() + sensor_noise)
    history = em.fit(start, iterations=10)            # estimate, set_noise, replay; history[-1].q_std / .r_std
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
        self._staged = None  # set_noise's settings until the next reset
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
        self._reset_noise()

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

    def set_noise(self, p0_std=None, q_std=None, r_std=None):
        """Stages new noise settings (None keeps a setting); they take effect at the next reset(), so one smoother record never
        mixes two noise models.  Validated as in the constructor."""
        p0 = None if p0_std is None else _std_vector(p0_std, 28, "p0_std")
        q = None if q_std is None else _std_vector(q_std, 28, "q_std")
        r = None if r_std is None else _std_vector(r_std, 7, "r_std")
        if r is not None and any(r[MEASUREMENT_NAMES.index(n)] <= 0 for n in self.measured):
            raise ValueError("r_std must be > 0 for every measured entry")
        e = self._live()
        ptr = lambda a: 0 if a is None else a.ctypes.data
        _lib.check(self._lib.glg_est_set_noise(e, ptr(p0), ptr(q), ptr(r)), self.env._h, "glg_est_set_noise")
        cur = self._staged or (self.p0_std, self.q_std, self.r_std)
        self._staged = tuple(old if new is None else new for new, old in zip((p0, q, r), cur))

    def _reset_noise(self):
        if self._staged is not None:
            self.p0_std, self.q_std, self.r_std = self._staged
            self._staged = None

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


EMStep = collections.namedtuple("EMStep", "q_std r_std loglik transitions measurements")


def _mask(v, n, name, default):
    if v is None:
        return default.copy()
    a = np.asarray(v)
    if a.shape != (n,) or a.dtype != np.bool_:
        raise ValueError(f"{name} must be a boolean mask of {n} entries")
    return a.copy()


class DeviceNoiseEM(_EnvCompanion):
    """EM of the estimator's diagonal Q and R over `smoother`'s window.  Logs every reset / update of the estimator from its next
    reset on; estimate() is one E-step and M-step over the logged window, replay() re-runs the logged window under the estimator's
    current (staged) noise, fit() alternates them.  Keeps the smoother alive; close the EM object before closing the smoother.

    fit_q / fit_r: boolean masks of the fitted entries (defaults: every state that takes part in smoothing, p0_std or q_std > 0,
    except x27; every measured entry).  q_floor / r_floor: lower bounds of the fitted values (defaults: 1e-3 x the estimator
    defaults).  max_points: sigma points per E-step launch (it bounds the memory of the internal handle that steps them)."""
    _kind, _destroy = "EM object", "glg_em_destroy"

    def __init__(self, smoother, fit_q=None, fit_r=None, q_floor=None, r_floor=None, max_points=MAX_SIGMA_POINTS):
        if not isinstance(smoother, DeviceStateSmoother):
            raise TypeError("smoother must be a DeviceStateSmoother")
        if isinstance(max_points, bool) or not isinstance(max_points, (int, np.integer)) or not 57 <= int(max_points) <= MAX_SIGMA_POINTS:
            raise ValueError(f"max_points must be an integer in 57 .. {MAX_SIGMA_POINTS}")
        est = smoother.est
        active = (np.asarray(est.p0_std) > 0) | (np.asarray(est.q_std) > 0)
        active[27] = False
        measured = np.zeros(7, dtype=bool)
        measured[[MEASUREMENT_NAMES.index(n) for n in est.measured]] = True
        self.fit_q = _mask(fit_q, 28, "fit_q", active)
        self.fit_r = _mask(fit_r, 7, "fit_r", measured)
        if self.fit_q[27]:
            raise ValueError("fit_q: x27, the day counter, is deterministic and never fitted")
        if np.any(self.fit_r & ~measured):
            raise ValueError("fit_r may only select measured entries")
        self.q_floor = _std_vector(1e-3 * np.asarray(DEFAULT_Q_STD) if q_floor is None else q_floor, 28, "q_floor")
        self.r_floor = _std_vector(1e-3 * np.asarray(DEFAULT_R_STD) if r_floor is None else r_floor, 7, "r_floor")
        W, B = smoother.window, int(est.env.num_envs)
        self.smoother, self.est, self.env, self._lib, self.window = smoother, est, est.env, est._lib, W
        self._obj = C.c_void_p()
        _lib.check(self._lib.glg_em_create(smoother._live(), int(max_points), C.byref(self._obj)), self.env._h, "glg_em_create")
        m, L = self._obj, self._lib
        self._log = {"controls": self._view(L.glg_em_controls_dev(m), (W, 6, B), "<f8").permute(0, 2, 1),
                     "table": self._view(L.glg_em_table_dev(m), (W, B), "<i4"),
                     "measurements": self._view(L.glg_em_measurements_dev(m), (W, 7, B), "<f8").permute(0, 2, 1),
                     "flags": self._view(L.glg_em_flags_dev(m), (W, B), "|u1"),
                     "loglik": self._view(L.glg_em_loglik_dev(m), (W, B), "<f8")}
        self._expectation = self._view(L.glg_em_expectation_dev(m), (W, B, 35), "<f8")
        self._prediction = self._view(L.glg_em_prediction_dev(m), (W, 28, B), "<f8").permute(0, 2, 1)
        self._used = self._view(L.glg_em_used_dev(m), (W, B), "|u1")
        self.env_stats = self._view(L.glg_em_env_stats_dev(m), (B, 38), "<f8")  # 35 sums, transitions, measured slots, sum of l
        self.totals = self._view(L.glg_em_totals_dev(m), (38,), "<f8")
        self.bytes = int(L.glg_em_bytes(m))
        self.chunk_pairs = int(L.glg_em_chunk_pairs(m))

    def _live(self):
        self.smoother._live()
        return super()._live()

    def _rolled(self, name):
        """A logged quantity, oldest first (a copy: the log is a ring)."""
        m = self._live()
        n, first = self.smoother.length, int(self._lib.glg_smooth_first(self.smoother._obj))
        return torch.roll(self._log[name], -first, 0)[:n]

    controls = property(lambda self: self._rolled("controls"), doc="[L, B, 6] the controls each env applied; 0 at a reset slot")
    tables = property(lambda self: self._rolled("table"), doc="[L, B] the weather table of each slot's step")
    measurements = property(lambda self: self._rolled("measurements"), doc="[L, B, 7] y as given; 0 where not measured")
    flags = property(lambda self: self._rolled("flags"), doc="[L, B] bit 0: y was given; bit 1: the update was applied")
    loglik = property(lambda self: self._rolled("loglik"), doc="[L, B] each update's log-likelihood term; 0 where none applied")

    @property
    def prediction(self):
        """[L, B, 28] fbar of the last estimate(): the smoothed one-step prediction (0 where no transition leads to the slot)."""
        return self._prediction[:self.smoother.length]

    @property
    def expectation(self):
        """[L, B, 35] of the last estimate(): the 28 Q terms E_k, then the 7 R terms; 0 where a slot does not enter a sum."""
        return self._expectation[:self.smoother.length]

    @property
    def used(self):
        """[L, B] of the last estimate(): bit 0: the slot's transition entered the Q sums; bit 1: its measurement the R sums."""
        return self._used[:self.smoother.length]

    def estep(self):
        """Runs the smoother, then the E-step over its output (device views expectation, prediction, used, env_stats, totals)."""
        self.smoother.smooth()
        _lib.check(self._lib.glg_em_estep(self._live(), self.env._stream()), self.env._h, "glg_em_estep")

    def estimate(self):
        """One E-step and M-step: EMStep(q_std, r_std, loglik, transitions, measurements).  loglik is the log-likelihood of the
        logged window under the noise it was filtered with; q_std and r_std are the maximisers for the fitted entries, floored, and
        the estimator's current values elsewhere."""
        self.estep()
        tot = self.totals.cpu().numpy()
        ntr, nme = int(round(tot[35])), int(round(tot[36]))
        q, r = np.array(self.est.q_std, dtype=np.float64), np.array(self.est.r_std, dtype=np.float64)
        if ntr > 0:
            q[self.fit_q] = np.maximum(np.sqrt(np.maximum(tot[:28] / ntr, 0.0)), self.q_floor)[self.fit_q]
        if nme > 0:
            r[self.fit_r] = np.maximum(np.sqrt(np.maximum(tot[28:35] / nme, 0.0)), self.r_floor)[self.fit_r]
        return EMStep(q, r, float(tot[37]), ntr, nme)

    def replay(self, env_state, x0=None):
        """Re-runs the logged window: restores the env from env_state (its state_dict() taken before the logged reset), resets the
        estimator (x0 as given to that reset), then steps the env with the logged controls and updates the estimator with the
        logged measurements (None where the logged update had none).  A run can be replayed when each update followed one env step
        and the log holds the whole run (at most `window` slots since the reset)."""
        m = self._live()
        n = int(self._lib.glg_em_logged(m))
        if n == 0:
            raise RuntimeError("nothing logged yet: the log starts with the estimator's first reset after the EM object's creation")
        if n > self.window:
            raise RuntimeError(f"the run has {n} slots and the log keeps the last {self.window}: it cannot be replayed")
        u, y, flags = self.controls.clone(), self.measurements.clone(), self.flags.cpu().numpy()
        self.env.load_state_dict(env_state)
        self.est.reset(x0)
        for k in range(1, n):
            self.env.step_raw_control_tensor(u[k])
            self.est.update(y[k] if np.any(flags[k] & 1) else None)

    def fit(self, env_state, iterations, x0=None):
        """`iterations` rounds of estimate(), set_noise(q_std, r_std) and replay(); returns the list of EMSteps (the loglik of step
        i is that of the noise the step started from)."""
        if isinstance(iterations, bool) or not isinstance(iterations, (int, np.integer)) or int(iterations) < 1:
            raise ValueError("iterations must be an integer >= 1")
        history = []
        for _ in range(int(iterations)):
            step = self.estimate()
            history.append(step)
            self.est.set_noise(q_std=step.q_std, r_std=step.r_std)
            self.replay(env_state, x0)
        return history
