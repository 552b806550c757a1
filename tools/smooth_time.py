"""State smoothing: the cost of recording (glg_est_update with and without a smoother) and of the backward pass (glg_smooth_run over
a full 96-slot window), in one command, on one GPU, at B = 64, 1024 and 4096 (default env: fp64, graded integrator, n_sub 260,
rule-based controller, uncertainty_scale 0.1):

  - two envs alike, each with an estimator; the second estimator has a smoother of WINDOW slots.  glg_est_update after each env
    step, CUDA events around the update alone (the env's step is outside the window); the two alternate within each of ROUNDS
    rounds of REPS calls, and the median round is reported;
  - glg_smooth_run once the ring is full, CUDA events, median of ROUNDS rounds of REPS calls;
  - the smoother's device bytes per env-slot (glg_smooth_bytes / (B W));
  - the record and backward kernels alone from torch.profiler in a separate pass.

    python tools/smooth_time.py [--out profiles/smooth_kernels.txt] [--sizes 64,1024,4096]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym.estimation import DeviceStateEstimator, DeviceStateSmoother
from glgym.vec_env import GreenLightVecEnv

REPS, ROUNDS, WINDOW = 10, 5, 96
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
    envs = [GreenLightVecEnv(B, seed=1, uncertainty_scale=0.1) for _ in range(2)]
    ests = []
    for env in envs:
        env.reset_tensor()
        for _ in range(8):
            env.step_rule_based_tensor()
        ests.append(DeviceStateEstimator(env))
    sm = DeviceStateSmoother(ests[1], WINDOW)
    for e in ests:
        e.reset()
    y = ests[0].measurements()
    paths = {"glg_est_update": (envs[0].step_rule_based_tensor, lambda: ests[0].update(y)),
             f"glg_est_update with a smoother (W {WINDOW})": (envs[1].step_rule_based_tensor, lambda: ests[1].update(y))}
    for pre, fn in paths.values():  # warm-up
        event_ms(pre, fn, 2)
    rounds = {n: [] for n in paths}
    for _ in range(ROUNDS):
        for name, (pre, fn) in paths.items():
            rounds[name].append(event_ms(pre, fn, REPS))
    med = {n: float(np.median(v)) for n, v in rounds.items()}
    while sm.length < WINDOW:
        envs[1].step_rule_based_tensor()
        ests[1].update(y)
    nothing = lambda: None
    event_ms(nothing, sm.smooth, 2)
    med[f"glg_smooth_run (W {WINDOW}, full ring)"] = float(np.median([event_ms(nothing, sm.smooth, REPS) for _ in range(ROUNDS)]))
    assert np.all(sm.status.cpu().numpy() == 0) and bool(torch.isfinite(sm.smooth().cov).all())
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(REPS):
            for pre, fn in paths.values():
                pre()
                fn()
            sm.smooth()
        torch.cuda.synchronize()
    own = {}
    for ev in prof.key_averages():
        if "glg_est_" in ev.key or "glg_smooth" in ev.key:
            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            own[ev.key.split("(")[0]] = t / 1e3 / REPS
    per_slot = sm.bytes / (B * WINDOW)
    sm.close()
    for e in ests:
        e.close()
    for env in envs:
        env.close()
    return med, own, per_slot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="64,1024,4096")
    args = ap.parse_args()
    lines = [f"# tools/smooth_time.py on {card()}",
             "# default env (fp64, graded integrator, n_sub 260), uncertainty_scale 0.1, rule-based controller; CUDA events,",
             f"# median of {ROUNDS} rounds of {REPS} calls (the two update paths alternate); times in ms per call; kernel times from",
             "# torch.profiler per call (the <true> instantiations run only with a smoother)"]
    for B in [int(s) for s in args.sizes.split(",")]:
        med, own, per_slot = measure(B)
        ref = med["glg_est_update"]
        lines.append(f"B = {B}: smoother device bytes per env-slot {per_slot:.0f} ({per_slot * B * WINDOW / 2 ** 30:.3f} GiB)")
        for n, v in med.items():
            lines.append(f"  {n:44s} {v:9.4f} ms   {v / ref:7.3f} x glg_est_update")
        for n, v in sorted(own.items()):
            lines.append(f"  kernel {n:37s} {v:9.4f} ms")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
