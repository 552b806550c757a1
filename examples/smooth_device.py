"""State smoothing on the batched GPU env: an unscented Rauch-Tung-Striebel smoother (`glgym.estimation.DeviceStateSmoother`) over the
estimates of the state estimator, reconstructing every env's 28-state from a logged run of noisy observations.

The setting is examples/estimate_device.py's: the true envs run with parametric uncertainty (uncertainty_scale 0.2) under the
rule-based controller; the filter starts from a deliberately wrong prior for the unobserved states (temperatures 1.5 K off, crop
pools 10 % off) and receives the seven measured quantities with seeded Gaussian sensor noise added in torch.

    python examples/smooth_device.py [--n-envs 16] [--days 2]

Prints the per-state RMS error against the true state over the run of three estimates: open loop (update(None)), filtered and
smoothed.
"""
import argparse, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch
from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
from glgym.vec_env import GreenLightVecEnv

ap = argparse.ArgumentParser()
ap.add_argument("--n-envs", type=int, default=16)
ap.add_argument("--days", type=float, default=2.0)
ap.add_argument("--seed", type=int, default=0)
a = ap.parse_args()
B = a.n_envs
steps = int(round(a.days * 86400 / 900))

env = GreenLightVecEnv(B, seed=a.seed, uncertainty_scale=0.2, base_env_params=dict(start_train_day=0, end_train_day=0))
env.reset_tensor()
est, olp = DeviceStateEstimator(env), DeviceStateEstimator(env)
smoother = DeviceStateSmoother(est, steps + 1)  # the whole run: the reset and every update
x0 = env.state_t.T.clone()
x0[:, 2:15] += 1.5
x0[:, 22:26] *= 1.1
est.reset(x0)
olp.reset(x0)
gen = torch.Generator(device="cuda").manual_seed(a.seed)
rstd = torch.as_tensor(est.r_std, device="cuda")
truth, open_loop = [env.state_t.T.clone()], [olp.mean.clone()]
for _ in range(steps):
    env.step_rule_based_tensor()
    est.update(est.measurements() + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen) * rstd)
    olp.update(None)
    truth.append(env.state_t.T.clone())
    open_loop.append(olp.mean.clone())
smoothed = smoother.smooth()
truth = torch.stack(truth)
rms = lambda m: torch.sqrt(torch.mean(torch.square(m - truth), dim=(0, 1))).cpu().numpy()
r_o, r_f, r_s = rms(torch.stack(open_loop)), rms(smoother.filtered_mean), rms(smoothed.mean)
assert np.all(smoother.status.cpu().numpy() == 0)
print(f"per-state RMS error against the true state over {steps + 1} estimates ({B} envs, uncertainty_scale 0.2, rule-based):")
print(f"{'state':>5} {'open loop':>12} {'filtered':>12} {'smoothed':>12} {'smoothed/filtered':>18}")
for i in range(28):
    ratio = f"{r_s[i] / r_f[i]:18.3f}" if r_f[i] > 0 else f"{'-':>18}"
    print(f"{i:5d} {r_o[i]:12.4g} {r_f[i]:12.4g} {r_s[i]:12.4g} {ratio}")
for o in (smoother, est, olp):
    o.close()
env.close()
