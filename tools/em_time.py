"""Noise identification: the cost of one E-step (glg_em_estep over a full W-slot window) against the bare step launches of its own
sigma points, the W-update forward pass and glg_smooth_run, in one command, on one GPU, at B = 128, 1024 and 4096 (default env:
fp64, graded integrator, n_sub 260, rule-based controller, uncertainty_scale 0.1):

  - an env with an estimator, a smoother of W slots and an EM object; W - 1 updates fill the window (the forward pass, timed with
    CUDA events around the whole loop of env steps and updates, and the updates alone);
  - glg_smooth_run and glg_em_estep (the smoother's output is left as it is), CUDA events, median of ROUNDS rounds of REPS calls;
  - the bare step of the E-step's points: glg_step_raw_control of handles the size of the E-step's chunks (balanced, at most
    max_points points each), one launch per chunk, so exactly the B W 57 points the E-step steps;
  - the E-step's own kernels (everything but the step) from torch.profiler in a separate pass.

    python tools/em_time.py [--out profiles/em_kernels.txt] [--sizes 128,1024,4096]
"""
import argparse
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym import _lib
from glgym.estimation import DeviceNoiseEM, DeviceStateEstimator, DeviceStateSmoother
from glgym.vec_env import GreenLightVecEnv

REPS, ROUNDS, WINDOW = 3, 3, 96
assert torch.cuda.is_available(), "this measurement needs the GPU"


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def event_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def measure(B):
    env = GreenLightVecEnv(B, seed=1, uncertainty_scale=0.1)
    env.reset_tensor()
    for _ in range(8):
        env.step_rule_based_tensor()
    est = DeviceStateEstimator(env)
    sm = DeviceStateSmoother(est, WINDOW)
    em = DeviceNoiseEM(sm)
    est.reset()
    y = est.measurements()
    torch.cuda.synchronize()
    upd = []

    def step_update():
        env.step_rule_based_tensor()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        est.update(y)
        b.record()
        upd.append((a, b))

    forward = event_ms(step_update, WINDOW - 1)
    torch.cuda.synchronize()
    updates = sum(a.elapsed_time(b) for a, b in upd)
    assert sm.length == WINDOW
    out = {f"forward pass ({WINDOW - 1} env steps + updates)": forward * (WINDOW - 1),
           f"  of which glg_est_update ({WINDOW - 1} calls)": updates}
    sm.smooth()
    estep = lambda: _lib.check(env._lib.glg_em_estep(em._obj, env._stream()), env._h, "glg_em_estep")
    estep()
    event_ms(sm.smooth, 1)
    out[f"glg_smooth_run (W {WINDOW})"] = float(np.median([event_ms(sm.smooth, REPS) for _ in range(ROUNDS)]))
    out[f"glg_em_estep (W {WINDOW})"] = float(np.median([event_ms(estep, REPS) for _ in range(ROUNDS)]))
    assert bool(torch.isfinite(em.totals).all())
    # the bare step of exactly the E-step's points: its balanced chunks of at most chunk_pairs pairs, each a batch of its own
    pairs = B * WINDOW
    chunks = math.ceil(pairs / em.chunk_pairs)
    per = math.ceil(pairs / chunks)
    sizes = [min(per, pairs - i * per) for i in range(chunks)]
    bare = {n: GreenLightVecEnv(n * 57, seed=1, uncertainty_scale=0.0) for n in set(sizes)}
    ctrl = {}
    for n, benv in bare.items():
        benv.reset_tensor()
        ctrl[n] = torch.full((n * 57, 6), 0.5, device="cuda", dtype=torch.float64)

    def bare_steps():
        for n in sizes:
            bare[n].step_raw_control_tensor(ctrl[n])

    bare_steps()
    label = " + ".join(f"{sizes.count(n)} x {n * 57}" for n in sorted(set(sizes), reverse=True))
    out[f"bare step of the E-step's {pairs * 57} points ({label} envs)"] = float(
        np.median([event_ms(bare_steps, 1) for _ in range(ROUNDS)]))
    for benv in bare.values():
        benv.close()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(REPS):
            estep()
        torch.cuda.synchronize()
    own = {}
    for ev in prof.key_averages():
        if "glg_em_" in ev.key:
            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            own[ev.key.split("(")[0]] = t / 1e3 / REPS
    em_bytes = em.bytes
    for o in (em, sm, est, env):
        o.close()
    return out, own, chunks, em_bytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="128,1024,4096")
    args = ap.parse_args()
    lines = [f"# tools/em_time.py on {card()}",
             "# default env (fp64, graded integrator, n_sub 260), uncertainty_scale 0.1, rule-based controller, W = 96; CUDA events,",
             f"# median of {ROUNDS} rounds of {REPS} calls; times in ms per call; the E-step's own kernels from torch.profiler"]
    for B in [int(s) for s in args.sizes.split(",")]:
        out, own, chunks, em_bytes = measure(B)
        es = out[f"glg_em_estep (W {WINDOW})"]
        lines.append(f"B = {B}: {chunks} chunk(s); EM object device bytes {em_bytes} ({em_bytes / 2 ** 30:.3f} GiB)")
        for n, v in out.items():
            lines.append(f"  {n:58s} {v:10.3f} ms   {v / es:7.3f} x glg_em_estep")
        ownt = sum(own.values())
        for n, v in sorted(own.items()):
            lines.append(f"  kernel {n:51s} {v:10.3f} ms")
        lines.append(f"  E-step kernels other than the step: {ownt:.3f} ms = {100 * ownt / es:.1f} % of glg_em_estep")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
