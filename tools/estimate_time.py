"""State estimation (glg_est_update) against the bare step of its B * 57 sigma points and against glg_linearize, in one command, on
one GPU, at B = 64, 1024 and 4096 (default env: fp64, graded integrator, n_sub 260, rule-based controller):

  - glg_est_update after each env step, CUDA events around the update alone (the env's step is outside the window);
  - glg_step_raw_control of a bare handle of B * 57 envs configured like the estimator's internal handle (no auto-reset, the
    IndoorClimateObservations stack), and of one with the default observation stack;
  - glg_linearize of the env (the extended Kalman filter's predict step) at the same B;
  - the estimator's own kernels (sigma, UT) from torch.profiler in a separate pass.
The paths alternate within each of ROUNDS rounds of REPS calls; the median round is reported.

    python tools/estimate_time.py [--out profiles/estimate_kernels.txt] [--sizes 64,1024,4096]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym.estimation import DeviceStateEstimator
from glgym.vec_env import GreenLightVecEnv

REPS, ROUNDS = 10, 5
assert torch.cuda.is_available(), "this measurement needs the GPU"


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def event_ms(before, fn, n):
    """Mean device time of fn over n calls, each preceded by before() outside the timed window."""
    tot = 0.0
    for _ in range(n):
        before()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        tot += a.elapsed_time(b)
    return tot / n


def measure(B):
    env = GreenLightVecEnv(B, seed=1, uncertainty_scale=0.1)
    env.reset_tensor()
    for _ in range(8):
        env.step_rule_based_tensor()
    est = DeviceStateEstimator(env)
    est.reset()
    y = est.measurements()
    bare = {s: GreenLightVecEnv(B * 57, seed=1, auto_reset=False, observation_modules=m)
            for s, m in (("shadow-like", ["IndoorClimateObservations"]), ("default stack", None))}
    for h in bare.values():
        h.reset_tensor()
    u = torch.rand(B * 57, 6, device="cuda", dtype=torch.float64)
    nothing = lambda: None
    paths = {"glg_est_update": (env.step_rule_based_tensor, lambda: est.update(y)),
             "glg_linearize": (nothing, lambda: env.linearize_tensor(None))}
    for s, h in bare.items():
        paths[f"bare B*57 step ({s})"] = (nothing, lambda h=h: h.step_raw_control_tensor(u))
    for name, (pre, fn) in paths.items():  # warm-up
        event_ms(pre, fn, 2)
    rounds = {n: [] for n in paths}
    for _ in range(ROUNDS):
        for name, (pre, fn) in paths.items():
            rounds[name].append(event_ms(pre, fn, REPS))
    med = {n: float(np.median(v)) for n, v in rounds.items()}
    assert np.all(est.status.cpu().numpy() == 0)
    # the estimator's kernels alone
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(REPS):
            env.step_rule_based_tensor()
            est.update(y)
        torch.cuda.synchronize()
    own = {}
    for ev in prof.key_averages():
        if "glg_est_" in ev.key:
            own[ev.key.split("(")[0]] = ev.device_time_total / 1e3 / REPS if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3 / REPS
    est.close()
    env.close()
    for h in bare.values():
        h.close()
    return med, own


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="64,1024,4096")
    args = ap.parse_args()
    lines = [f"# tools/estimate_time.py on {card()}",
             "# default env (fp64, graded integrator, n_sub 260), uncertainty_scale 0.1, rule-based controller; CUDA events,",
             f"# median of {ROUNDS} alternating rounds of {REPS} calls; times in ms per call"]
    for B in [int(s) for s in args.sizes.split(",")]:
        med, own = measure(B)
        ref = med["bare B*57 step (shadow-like)"]
        lines.append(f"B = {B} ({B * 57} sigma points)")
        for n, v in med.items():
            lines.append(f"  {n:40s} {v:9.4f} ms   {v / ref:7.3f} x bare shadow-like step")
        for n, v in sorted(own.items()):
            lines.append(f"  kernel {n:33s} {v:9.4f} ms   {v / med['glg_est_update'] * 100:6.2f} % of glg_est_update")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
