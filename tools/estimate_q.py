"""Default process-noise std of DeviceStateEstimator (glgym/estimation.py DEFAULT_Q_STD): the per-state standard deviation of
the nominal model's one-step error against envs with uncertainty_scale = 0.1 under the rule-based controller.

Each step the estimator is restarted at the true state with zero covariance, so all its sigma points coincide and update(None)
is one nominal step from the true state; the error is the true env's state after its step minus that prediction.  Envs that
finished (auto-reset) are left out of that step.

    python tools/estimate_q.py [--envs 256] [--steps 960]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym.estimation import DeviceStateEstimator
from glgym.vec_env import GreenLightVecEnv

assert torch.cuda.is_available(), "this measurement needs the GPU"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--steps", type=int, default=960)
    args = ap.parse_args()
    B = args.envs
    env = GreenLightVecEnv(B, seed=11, uncertainty_scale=0.1)
    env.reset_tensor()
    est = DeviceStateEstimator(env, p0_std=np.zeros(28), q_std=np.zeros(28))
    err = []
    for _ in range(args.steps):
        est.reset()
        env.step_rule_based_tensor()
        est.update(None)
        ok = est.status == 0
        err.append((env.state_t.T - est.mean)[ok].cpu().numpy())
    e = np.concatenate(err)
    q = np.sqrt(np.mean(np.square(e), axis=0))
    print(f"{len(e)} one-step errors, {B} envs x {args.steps} steps")
    print("DEFAULT_Q_STD = (" + ", ".join(f"{v:.4g}" for v in q) + ")")
    est.close()
    env.close()


if __name__ == "__main__":
    main()
