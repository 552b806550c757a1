"""Linearise the greenhouse along a controlled trajectory on the device.

16 envs run one January day (GL2009 start day 0, 96 steps) under the device rule-based controller.  At each step the example
asks the library for:
  - df/dx of the continuous-time model at every env's state (glg_rhs_jacobian_batch) and prints the largest |Re lambda| over the
    batch: the stiffness trace tests/golden/make_truth.py computes on the CPU with forward differences;
  - the step Jacobian of the coming control interval (glg_linearize) and prints the linear prediction Bu . du of the climate states'
    response to a +0.1 boiler step, beside the response a twin env shows when it takes the perturbed step.

    python examples/linearize_device.py [--envs 16] [--steps 96]
"""
import argparse, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym.model import GreenLight
from glgym.vec_env import GreenLightVecEnv

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=16)
ap.add_argument("--steps", type=int, default=96)
a = ap.parse_args()

CLIMATE = {"co2Air": 0, "tAir": 2, "vpAir": 15}  # the controlled climate states
kw = dict(base_env_params=dict(start_train_day=0, end_train_day=0), seed=0)
env, twin = GreenLightVecEnv(a.envs, **kw), GreenLightVecEnv(a.envs, **kw)
env.reset_tensor()
twin.reset_tensor()
model = GreenLight(integrator=env.integrator, n_sub=env.n_sub)
p = torch.as_tensor(np.asarray(env.p, dtype=np.float64), device="cuda")
W = torch.as_tensor(env.weather_tables, device="cuda")
du = torch.zeros((a.envs, 6), dtype=torch.float64, device="cuda")
du[:, 0] = 0.1  # boiler
print(f"{'step':>4} {'max|Re l|':>9} " + " ".join(f"{n + ' lin':>12} {n + ' sim':>12}" for n in CLIMATE))
for k in range(a.steps):
    u = env.rule_controls_tensor().clone()
    x = env.state_t.T.contiguous()
    kw_ = torch.clamp(env.timestep_t.long(), max=W.shape[1] - env.Np - 1)
    d = W[env.table_t.long(), kw_].contiguous()
    _, jx, _ = model.rhs_jacobian_batch(x, u, d, p)
    lam = torch.linalg.eigvals(jx).real.abs().amax().item()
    u_up = torch.clamp(u + du, 0.0, 1.0)
    x_next, A, Bu = env.linearize_tensor(u)
    lin = (Bu @ (u_up - u)[:, :, None])[:, :, 0]
    twin.load_state_dict(env.state_dict())
    twin.step_raw_control_tensor(u_up)
    env.step_raw_control_tensor(u)
    sim = twin.state_t.T - env.state_t.T
    cols = " ".join(f"{lin[:, i].mean().item():>12.4e} {sim[:, i].mean().item():>12.4e}" for i in CLIMATE.values())
    print(f"{k:>4} {lam:>9.4f} {cols}", flush=True)
env.close()
twin.close()
