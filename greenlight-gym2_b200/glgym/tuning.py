"""Tuning of the rule-based controller's settings: CEM over the 29 settings of rule_based.yml, scored by the env's own season
return.

`RuleControllerTuner` owns one `GreenLightVecEnv` of K S envs without auto-reset: env c = k S + s runs candidate k on scenario s
(a weather table of the env's bank).  A generation samples K candidates, resets every env onto its scenario, runs `horizon` steps
of `rule_controls_tensor` (per-env settings, csrc glg_rule_controls) followed by `step_raw_control_tensor`, and moves the sampling
distribution to the E best candidates.  The tuner's own arithmetic is 29 K numbers per generation next to seconds of simulation,
so it is torch, not kernels.

With uncertainty_scale > 0 the parametric noise is one fixed sample, n ~ U(-scale/2, scale/2) per (scenario, step, parameter),
passed to the step as external noise and shared by all K candidates and all generations (common random numbers): candidates are
compared on identical weather and parameter paths, and the objective is deterministic.
"""
import numpy as np
import torch

from .controller import DEFAULT_SETTINGS, SETTING_NAMES
from .vec_env import DEFAULT_BASE_ENV_PARAMS, GreenLightVecEnv

# Default search box: the settings a grower would adjust, each range keeping its band's sign.
DEFAULT_BOUNDS = dict(
    temp_setpoint_day=(16.0, 24.0), temp_setpoint_night=(12.0, 20.0), heat_deadzone=(1.0, 10.0), co2_day=(400.0, 1200.0),
    vent_heat_Pband=(1.0, 10.0), rh_max=(75.0, 95.0), vent_rh_Pband=(1.0, 10.0), thScrSpDay=(0.0, 15.0),
    thScrSpNight=(0.0, 15.0), lamps_off_sun=(100.0, 600.0), lamp_rad_sum_limit=(5.0, 20.0),
)
# proportional bands: glg_prop_ctrl divides by the band, so a tuned range must not contain 0
PBAND_SETTINGS = ("vent_heat_Pband", "vent_rh_Pband", "vent_cold_Pband", "thScrPband", "thScrRhPband", "tHeatBand", "co2Band")


class SeasonFitness:
    """Streaming fitness of K candidates over S scenarios each (env c = k S + s).  add() takes one step's reward and done of
    every env; a reward counts up to and including the env's first done.  result(): the mean over its S envs of each candidate's
    undiscounted return, or -inf when one of its envs ended before the last step or had a non-finite reward."""

    def __init__(self, n_candidates, n_scenarios, device):
        B = n_candidates * n_scenarios
        self.K, self.S = n_candidates, n_scenarios
        self.ret = torch.zeros(B, dtype=torch.float64, device=device)
        self.alive = torch.ones(B, dtype=torch.bool, device=device)
        self.ok = torch.ones(B, dtype=torch.bool, device=device)

    def add(self, reward, done, last):
        r = torch.where(self.alive, reward, 0.0)
        self.ret += r
        self.ok &= torch.isfinite(r)
        done = done.bool()
        if not last:
            self.ok &= ~(self.alive & done)
        self.alive &= ~done

    def result(self):
        ok = self.ok.view(self.K, self.S).all(dim=1)
        fit = self.ret.view(self.K, self.S).mean(dim=1)
        return torch.where(ok, fit, -torch.inf)


def elite_update(candidates, fitness, n_elites, tuned):
    """CEM update: the n_elites largest fitnesses (ties to the lower index, -inf last) -> (elite indices, mean, population
    std) of the columns `tuned` of candidates [K, 29], in float64."""
    order = torch.sort(fitness, descending=True, stable=True).indices
    elites = order[:n_elites]
    x = candidates[elites][:, tuned]
    return elites, x.mean(dim=0), x.std(dim=0, correction=0)


def _env_shape(env_kwargs):
    """(N, number of weather tables) of the GreenLightVecEnv env_kwargs would build, before building it."""
    bp = dict(DEFAULT_BASE_ENV_PARAMS)
    bp.update(env_kwargs.get("base_env_params") or {})
    N = int(bp["season_length"] * 86400 / bp["dt"])
    w = env_kwargs.get("weather_tables")
    if w is not None:
        w = np.asarray(w)
        return N, 1 if w.ndim == 2 else w.shape[0]
    if bp["training"]:
        years = range(bp["start_train_year"], bp["end_train_year"] + 1)
        days = range(bp["start_train_day"], bp["end_train_day"] + 1)
    else:
        years, days = env_kwargs["eval_options"]["eval_years"], env_kwargs["eval_options"]["eval_days"]
    return N, len(years) * len(days)


class RuleControllerTuner:
    """CEM over the rule-based controller's settings; see the module docstring.

    n_candidates K, n_elites E; scenarios: S table ids of the env's weather bank (default: every table; a table may repeat, and
    under uncertainty each repeat gets its own noise draw); horizon: steps per rollout, 1 .. N + 1 (default N + 1, the season);
    bounds: {name: (lo, hi)} of the tuned settings (default DEFAULT_BOUNDS); base: values of every other setting (default the
    shipped rule_based.yml); init_std: initial std as a fraction of each range; env_kwargs: passed to GreenLightVecEnv.

    After generation(): best_settings (dict), best_fitness, history (one dict per generation), and the last generation's
    candidates [K, 29] / fitness [K] (CUDA float64) and the distribution mean / std [29] (0 std for fixed settings)."""

    def __init__(self, n_candidates=256, n_elites=32, scenarios=None, horizon=None, bounds=None, base=None, init_std=0.3,
                 uncertainty_scale=0.0, seed=0, **env_kwargs):
        K, E = int(n_candidates), int(n_elites)
        if K < 1 or not 1 <= E <= K:
            raise ValueError(f"need 1 <= n_elites <= n_candidates; got n_elites={E}, n_candidates={K}")
        base_s = dict(DEFAULT_SETTINGS)
        unknown = [k for k in (base or {}) if k not in base_s]
        if unknown:
            raise ValueError(f"unknown settings in base: {unknown}")
        base_s.update({k: float(v) for k, v in (base or {}).items()})
        bounds = dict(DEFAULT_BOUNDS if bounds is None else bounds)
        unknown = [k for k in bounds if k not in base_s]
        if unknown or not bounds:
            raise ValueError(f"bounds must name at least one of {list(SETTING_NAMES)}; unknown: {unknown}")
        for name, (lo, hi) in bounds.items():
            lo, hi = float(lo), float(hi)
            if not lo < hi:
                raise ValueError(f"bounds of {name}: need lo < hi, got ({lo}, {hi})")
            if not lo <= base_s[name] <= hi:
                raise ValueError(f"base value {base_s[name]} of {name} is outside its bounds ({lo}, {hi})")
            if name in PBAND_SETTINGS and lo <= 0.0 <= hi:
                raise ValueError(f"{name} is a proportional band (the controller divides by it): its range ({lo}, {hi}) "
                                 "must not contain 0")
        if not init_std > 0:
            raise ValueError("init_std must be > 0")
        if uncertainty_scale < 0:
            raise ValueError("uncertainty_scale must be >= 0")
        N, n_tables = _env_shape(env_kwargs)
        scenarios = list(range(n_tables)) if scenarios is None else [int(s) for s in scenarios]
        if not scenarios or min(scenarios) < 0 or max(scenarios) >= n_tables:
            raise ValueError(f"scenarios must be a non-empty list of table ids in 0 .. {n_tables - 1}; got {scenarios}")
        horizon = N + 1 if horizon is None else int(horizon)
        if not 1 <= horizon <= N + 1:
            raise ValueError(f"horizon must be in 1 .. N + 1 = {N + 1}; got {horizon}")

        S = len(scenarios)
        self.n_candidates, self.n_elites, self.n_scenarios, self.horizon = K, E, S, horizon
        self.scenarios, self.base, self.bounds = scenarios, base_s, bounds
        self.uncertainty_scale = float(uncertainty_scale)
        self.env = GreenLightVecEnv(K * S, auto_reset=False, uncertainty_scale=0.0, **env_kwargs)
        dev = self.device = self.env.device
        f64 = dict(dtype=torch.float64, device=dev)
        self.tuned = torch.tensor([SETTING_NAMES.index(k) for k in bounds], dtype=torch.long, device=dev)
        base_v = torch.tensor([base_s[k] for k in SETTING_NAMES], **f64)
        # fixed settings have lo = hi = base, so the clamp of the sampling step keeps them at their base value exactly
        self.lo, self.hi = base_v.clone(), base_v.clone()
        self.lo[self.tuned] = torch.tensor([float(b[0]) for b in bounds.values()], **f64)
        self.hi[self.tuned] = torch.tensor([float(b[1]) for b in bounds.values()], **f64)
        self.mean = base_v.clone()
        self.std = torch.zeros(len(SETTING_NAMES), **f64)
        self.std[self.tuned] = float(init_std) * (self.hi - self.lo)[self.tuned]
        self._gen = torch.Generator(device=dev)
        self._gen.manual_seed(int(seed))
        self._table_ids = torch.tensor(scenarios, dtype=torch.int32, device=dev).repeat(K)
        self._noise = None
        if self.uncertainty_scale > 0:  # one draw per (scenario, step), reused by every candidate and generation
            u = torch.rand((horizon, S, 34), generator=self._gen, **f64)
            self._noise = (u - 0.5) * self.uncertainty_scale
        self.candidates = self.fitness = None
        self.best_settings, self.best_fitness, self.history = None, -float("inf"), []

    def _sample(self):
        K = self.n_candidates
        z = torch.randn((K, len(SETTING_NAMES)), generator=self._gen, dtype=torch.float64, device=self.device)
        z[0] = 0.0
        return torch.minimum(torch.maximum(self.mean + self.std * z, self.lo), self.hi)

    def _rollout(self, candidates):
        """Fitness [K] of candidates [K, 29] on the scenarios."""
        env, K, S = self.env, self.n_candidates, self.n_scenarios
        settings = candidates.repeat_interleave(S, dim=0).contiguous()
        env.reset_tensor(table_ids=self._table_ids)
        acc = SeasonFitness(K, S, self.device)
        for t in range(self.horizon):
            u = env.rule_controls_tensor(settings)
            noise = None if self._noise is None else self._noise[t].repeat(K, 1)
            _, reward, done = env.step_raw_control_tensor(u, noise=noise)
            acc.add(reward, done, last=t == self.horizon - 1)
        return acc.result()

    def generation(self):
        """One CEM generation.  Returns (mean fitness of the elites, best fitness of this generation)."""
        cand = self._sample()
        fit = self._rollout(cand)
        elites, mean_t, std_t = elite_update(cand, fit, self.n_elites, self.tuned)
        self.mean[self.tuned] = mean_t
        self.std[self.tuned] = std_t
        self.candidates, self.fitness = cand, fit
        best, elite_fit = float(fit[elites[0]]), fit[elites]
        if self.best_settings is None or best > self.best_fitness:
            v = cand[elites[0]].tolist()
            self.best_settings, self.best_fitness = dict(zip(SETTING_NAMES, v)), best
        mean_fit = float(elite_fit.mean())
        self.history.append(dict(mean_fitness=mean_fit, best_fitness=best, mean=self.mean.tolist(), std=self.std.tolist()))
        return mean_fit, best

    def evaluate(self, settings):
        """Fitness (numpy float64) of each settings dict (at most K of them; missing keys take the tuner's base values) on the
        tuner's scenarios, horizon and noise sample."""
        settings = list(settings)
        if not 1 <= len(settings) <= self.n_candidates:
            raise ValueError(f"evaluate takes 1 .. {self.n_candidates} settings; got {len(settings)}")
        rows = []
        for s in settings:
            unknown = [k for k in s if k not in self.base]
            if unknown:
                raise ValueError(f"unknown settings: {unknown}")
            full = dict(self.base)
            full.update(s)
            rows.append([float(full[k]) for k in SETTING_NAMES])
        rows += [rows[0]] * (self.n_candidates - len(rows))
        cand = torch.tensor(rows, dtype=torch.float64, device=self.device)
        return self._rollout(cand)[:len(settings)].cpu().numpy()

    def close(self):
        if getattr(self, "env", None) is not None:
            self.env.close()
            self.env = None
