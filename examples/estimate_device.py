"""State estimation on the batched GPU env: an unscented Kalman filter (`glgym.estimation.DeviceStateEstimator`) that tracks every
env's 28-state from its noisy observations, and model-predictive control from that estimate (output feedback).

The true envs run with parametric uncertainty (uncertainty_scale 0.2) for one January day; the filter starts from a deliberately
wrong prior for the unobserved states (temperatures 1.5 K off, crop pools 10 % off) and receives the seven measured quantities
with seeded Gaussian sensor noise added in torch.

    python examples/estimate_device.py [--n-envs 16] [--days 1] [--horizon 8] [--candidates 64] [--elites 8] [--iters 2]

Prints the per-state RMS error of the filter and of the open-loop prediction (update(None)) over the run, and the mean reward
per step of full-state MPC, MPC from the estimate and the rule-based controller.
"""
import argparse, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch
from glgym.estimation import DeviceStateEstimator
from glgym.planning import DevicePlanner
from glgym.vec_env import GreenLightVecEnv

ap = argparse.ArgumentParser()
ap.add_argument("--n-envs", type=int, default=16)
ap.add_argument("--days", type=float, default=1.0)
ap.add_argument("--horizon", type=int, default=8)
ap.add_argument("--candidates", type=int, default=64)
ap.add_argument("--elites", type=int, default=8)
ap.add_argument("--iters", type=int, default=2)
ap.add_argument("--seed", type=int, default=0)
a = ap.parse_args()
B = a.n_envs
mk = lambda: GreenLightVecEnv(B, seed=a.seed, uncertainty_scale=0.2, base_env_params=dict(start_train_day=0, end_train_day=0))
steps = int(round(a.days * 86400 / 900))


def wrong_prior(env):
    x0 = env.state_t.T.clone()
    x0[:, 2:15] += 1.5
    x0[:, 22:26] *= 1.1
    return x0


def run(controller):
    """One day from the reset state; controller in ("rule", "mpc-full", "mpc-est").  Returns (reward per step, filter RMS per
    state, open-loop RMS per state)."""
    env = mk()
    env.reset_tensor()
    est, olp = DeviceStateEstimator(env), DeviceStateEstimator(env)
    x0 = wrong_prior(env)
    est.reset(x0)
    olp.reset(x0)
    planner = None if controller == "rule" else DevicePlanner(env, a.horizon, a.candidates, a.elites, a.iters, seed=a.seed)
    gen = torch.Generator(device="cuda").manual_seed(a.seed)
    rstd = torch.as_tensor(est.r_std, device="cuda")
    rew, e_f, e_o = 0.0, [], []
    for _ in range(steps):
        if controller == "rule":
            env.step_rule_based_tensor()
        else:
            env.step_tensor(planner.plan(est.mean if controller == "mpc-est" else None))
            planner.shift()
        rew += float(env.reward_t.mean())
        y = est.measurements() + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen) * rstd
        est.update(y)
        olp.update(None)
        e_f.append((est.mean - env.state_t.T).cpu().numpy())
        e_o.append((olp.mean - env.state_t.T).cpu().numpy())
    rms = lambda e: np.sqrt(np.mean(np.square(np.stack(e)), axis=(0, 1)))
    out = (rew / steps, rms(e_f), rms(e_o))
    for o in (planner, est, olp):
        if o is not None:
            o.close()
    env.close()
    return out


results = {c: run(c) for c in ("rule", "mpc-full", "mpc-est")}
_, rf, ro = results["rule"]
print(f"per-state RMS error over {steps} steps under the rule-based controller ({B} envs, uncertainty_scale 0.2):")
print(f"{'state':>5} {'filter':>12} {'open loop':>12}")
for i in range(28):
    print(f"{i:5d} {rf[i]:12.4g} {ro[i]:12.4g}")
print("mean reward per step:")
print(f"  full-state MPC      {results['mpc-full'][0]:.4f}")
print(f"  MPC from estimate   {results['mpc-est'][0]:.4f}")
print(f"  rule-based          {results['rule'][0]:.4f}")
