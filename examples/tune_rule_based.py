"""Tune the rule-based controller's settings for this weather, reward and prices, and check the result on held-out start days.

CEM (glgym.tuning.RuleControllerTuner) over the 11 settings of DEFAULT_BOUNDS, scored by the full-season return on the GL2009
start days 0-15 (K = 256 candidates x 16 days = 4096 envs in one batch, E = 32 elites, 10 generations).  Then the shipped and the
tuned settings are each run through a full season on the held-out start days 16-18 with `evaluate_rule_based`, and the tuned
settings are written as YAML in rule_based.yml key order, loadable by the reference's evaluate_baseline.py.

    python examples/tune_rule_based.py [--out data/rule_based_tuned.yml] [--generations 10] [--candidates 256] [--elites 32]
"""
import argparse, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import yaml

from glgym.controller import DEFAULT_SETTINGS, SETTING_NAMES
from glgym.evaluation import RESULT_INFO, evaluate_rule_based
from glgym.tuning import RuleControllerTuner
from glgym.vec_env import GreenLightVecEnv

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="data/rule_based_tuned.yml")
ap.add_argument("--generations", type=int, default=10)
ap.add_argument("--candidates", type=int, default=256)
ap.add_argument("--elites", type=int, default=32)
ap.add_argument("--horizon", type=int, default=None, help="steps per rollout (default: the season, N + 1)")
ap.add_argument("--seed", type=int, default=0)
a = ap.parse_args()

t0 = time.time()
tuner = RuleControllerTuner(n_candidates=a.candidates, n_elites=a.elites, horizon=a.horizon, seed=a.seed,
                            base_env_params=dict(start_train_day=0, end_train_day=15))
print(f"tuning on GL2009 start days 0-15: {a.candidates} candidates x {tuner.n_scenarios} days = {tuner.env.num_envs} envs, "
      f"{tuner.horizon} steps per rollout", flush=True)
shipped_fit = tuner.evaluate([{}])[0]
print(f"shipped settings: fitness {shipped_fit:.4f}", flush=True)
for g in range(a.generations):
    tg = time.time()
    mean_fit, best_fit = tuner.generation()
    print(f"generation {g}: elite mean {mean_fit:.4f}, generation best {best_fit:.4f}, best so far {tuner.best_fitness:.4f} "
          f"({time.time() - tg:.1f} s)", flush=True)
best = tuner.best_settings
tuner.close()
print("tuned settings (changed from rule_based.yml):")
for k in SETTING_NAMES:
    if best[k] != DEFAULT_SETTINGS[k]:
        print(f"  {k:22s} {DEFAULT_SETTINGS[k]:>8g} -> {best[k]:.4f}")


def held_out(settings):
    """Full season on each of the start days 16-18 (one env per day): [days, steps, 32]."""
    out = []
    for day in (16, 17, 18):
        env = GreenLightVecEnv(1, base_env_params=dict(start_train_day=day, end_train_day=day), info_mode="minimal")
        out.append(evaluate_rule_based(env, settings)[0])
        env.close()
    return np.stack(out)


print("held-out GL2009 start days 16-18, one full season each (mean over the days):")
print(f"  {'':8s} {'reward/step':>12s} {'EPI':>10s} {'temp viol':>10s} {'co2 viol':>10s} {'rh viol':>10s}")
for name, s in (("shipped", None), ("tuned", best)):
    d = held_out(s)
    col = lambda key: 24 + RESULT_INFO.index(key)
    season = lambda key: d[:, :, col(key)].sum(axis=1).mean()
    print(f"  {name:8s} {d[:, :, 23].mean():12.5f} {season('EPI'):10.3f} {season('temp_violation'):10.2f} "
          f"{season('co2_violation'):10.2f} {season('rh_violation'):10.2f}", flush=True)

os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    yaml.safe_dump({k: float(best[k]) for k in SETTING_NAMES}, f, sort_keys=False)
print(f"tuned settings -> {a.out}; total {time.time() - t0:.1f} s")
