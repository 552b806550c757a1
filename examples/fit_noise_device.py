"""Fit the state estimator's process and measurement noise from observations alone (glgym.estimation.DeviceNoiseEM).

64 envs with uncertainty_scale 0.1 run two days under the rule-based controller; the measurements carry Gaussian sensor noise at
DEFAULT_R_STD.  EM starts from a 4x mis-set noise model and alternates the E-step on the device, the M-step and a replay of the
logged run.  Printed: the log-likelihood per iteration, the fitted r_std against the true one, the fitted q_std beside the values
tools/estimate_q.py measures with the true state, and the smoothed per-state RMS error under the fitted, the default and the
4x-mis-set noise.

    python examples/fit_noise_device.py [--iterations 10]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym.estimation import DEFAULT_Q_STD, DEFAULT_R_STD, DeviceNoiseEM, DeviceStateEstimator, DeviceStateSmoother
from glgym.vec_env import GreenLightVecEnv

NAMES = ["co2Air", "co2Top", "tAir", "tTop", "tCan", "tCovIn", "tCovE", "tThScr", "tFlr", "tPipe", "tSo1", "tSo2", "tSo3", "tSo4",
         "tSo5", "vpAir", "vpTop", "tLamp", "tIntLamp", "tGroPipe", "tBlScr", "tCan24", "cBuf", "cLeaf", "cStem", "cFruit", "tCanSum",
         "time"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iterations", type=int, default=10)
    args = ap.parse_args()
    B, steps = 64, 192
    env = GreenLightVecEnv(B, seed=2, uncertainty_scale=0.1)
    env.reset_tensor()
    start = env.state_dict()
    q0, r0 = 4 * np.array(DEFAULT_Q_STD), 4 * np.array(DEFAULT_R_STD)
    est = DeviceStateEstimator(env, q_std=q0, r_std=r0)
    sm = DeviceStateSmoother(est, steps + 1)
    em = DeviceNoiseEM(sm)
    est.reset()
    gen = torch.Generator(device="cuda").manual_seed(0)
    truth = [env.state_t.T.cpu().numpy().copy()]
    for _ in range(steps):
        env.step_rule_based_tensor()
        y = est.measurements() + torch.randn(B, 7, device="cuda", dtype=torch.float64, generator=gen) * torch.as_tensor(
            DEFAULT_R_STD, device="cuda")
        est.update(y)
        truth.append(env.state_t.T.cpu().numpy().copy())
    truth = np.stack(truth)

    def smoothed_rms():
        return np.sqrt(np.mean(np.square(sm.smooth().mean.cpu().numpy() - truth), axis=(0, 1)))

    rms_mis = smoothed_rms()
    history = em.fit(start, args.iterations)
    fitted = em.estimate()
    print("log-likelihood per iteration:", " ".join(f"{h.loglik:.6e}" for h in history + [fitted]))
    print(f"{'entry':>10s} {'fitted r_std':>13s} {'true':>10s}")
    for n, a, b in zip(("co2_air", "temp_air", "rh_air", "pipe_temp", "24CanTemp", "cFruit", "tSum"), fitted.r_std, DEFAULT_R_STD):
        print(f"{n:>10s} {a:13.4g} {b:10.4g}")
    est.set_noise(q_std=fitted.q_std, r_std=fitted.r_std)  # the printed fit, applied to the window
    em.replay(start)
    rms_fit = smoothed_rms()
    est.set_noise(q_std=DEFAULT_Q_STD, r_std=DEFAULT_R_STD)
    em.replay(start)
    rms_def = smoothed_rms()
    print(f"{'state':>9s} {'fitted q':>10s} {'estimate_q':>10s} | smoothed RMS error: {'fitted':>10s} {'default':>10s} "
          f"{'4x':>10s}")
    for j in range(28):
        print(f"{NAMES[j]:>9s} {fitted.q_std[j]:10.4g} {DEFAULT_Q_STD[j]:10.4g} | {'':20s}{rms_fit[j]:10.4g} {rms_def[j]:10.4g} "
              f"{rms_mis[j]:10.4g}")
    for o in (em, sm, est, env):
        o.close()


if __name__ == "__main__":
    main()
