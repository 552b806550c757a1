"""Model-predictive control on the batched GPU env: a receding-horizon CEM planner (`glgym.planning.DevicePlanner`) that scores
candidate control sequences with the env's own step kernels and reward, against the on-device rule-based controller
(configs/agents/rule_based.yml) and the hold policy (a = 0: keep the controls), all three from the same start states.

    python examples/mpc_device.py [--n-envs 16] [--days 1] [--horizon 12] [--candidates 256] [--elites 32] [--iters 3]

Prints per controller the mean reward per step, and per env over the run the summed EPI (economic performance indicator) and the
temperature, CO2 and relative-humidity violations; for the planner also the time per decision.
"""
import argparse, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import torch
from glgym.planning import DevicePlanner
from glgym.vec_env import GreenLightVecEnv

ap = argparse.ArgumentParser()
ap.add_argument("--n-envs", type=int, default=16)
ap.add_argument("--days", type=float, default=1.0)
ap.add_argument("--horizon", type=int, default=12)
ap.add_argument("--candidates", type=int, default=256)
ap.add_argument("--elites", type=int, default=32)
ap.add_argument("--iters", type=int, default=3)
ap.add_argument("--gamma", type=float, default=1.0)
ap.add_argument("--seed", type=int, default=0)
a = ap.parse_args()

env = GreenLightVecEnv(a.n_envs, seed=a.seed)
steps = int(round(a.days * 86400 / env.dt))
env.reset_tensor()
start = env.state_dict()
planner = DevicePlanner(env, a.horizon, a.candidates, a.elites, a.iters, gamma=a.gamma, seed=a.seed)


def run(name, act):
    env.load_state_dict(start)
    rew = torch.zeros(env.num_envs, dtype=torch.float64, device=env.device)
    info = torch.zeros_like(env.info_t)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        _, r, _ = act()
        rew += r
        info += env.info_t
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    info = info.mean(dim=1).cpu().numpy()  # per env over the run, averaged over envs
    print(f"{name:11s} reward/step {rew.mean().item() / steps:+.5f}   EPI {info[0]:+.4f}   temp viol {info[7]:8.3f}   "
          f"co2 viol {info[8]:9.2f}   rh viol {info[9]:7.3f}   {1e3 * dt:8.2f} ms per step", flush=True)


def mpc_step():
    out = env.step_tensor(planner.plan())
    planner.shift()
    return out


print(f"{a.n_envs} envs, {steps} steps from the same start states; planner H = {a.horizon}, K = {a.candidates}, E = {a.elites}, "
      f"I = {a.iters} ({a.n_envs * a.candidates} planning envs); ms per step includes the decision")
run("planner", mpc_step)
run("rule-based", env.step_rule_based_tensor)
zero = torch.zeros(a.n_envs, 6, device=env.device)
run("hold", lambda: env.step_tensor(zero))
planner.close()
env.close()
