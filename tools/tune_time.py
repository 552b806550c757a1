"""Per-env rule-based controls (glg_rule_controls) and the settings tuner (glgym.tuning.RuleControllerTuner): what they cost
against the fused rule-based step, in one command.

  - time per step of glg_rule_controls + glg_step_raw_control (per-env settings) against glg_step_rule_based, alternating in
    the same run, at B = 4096 and 65 536 (default env: fp64, graded integrator), CUDA events over STEPS steps per round;
  - the controls kernel alone, CUDA events over many launches;
  - one tuner generation (K = 256 candidates x 16 start days = 4096 envs, the season) against its horizon bare
    glg_step_rule_based launches of a handle of the same size.

    python tools/tune_time.py [--out profiles/tune_rule_based.txt]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import torch

from glgym.controller import RuleBasedController
from glgym.tuning import RuleControllerTuner
from glgym.vec_env import GreenLightVecEnv

STEPS, ROUNDS, KERNEL_LAUNCHES = 200, 3, 2000
assert torch.cuda.is_available(), "this measurement needs the GPU"


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tune_rule_based.txt"))
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"card: {card()}")
    say(f"torch {torch.__version__}; default env (fp64, graded integrator, n_sub 260), January start states, no auto-reset")
    say(f"per step: CUDA events over {STEPS} steps, {ROUNDS} rounds alternating the two paths on twin handles; "
        "per-env settings = 4 distinct settings vectors spread over the envs")
    say()
    for B in (4096, 65536):
        fused = GreenLightVecEnv(B, auto_reset=False)
        split = GreenLightVecEnv(B, auto_reset=False)
        vecs = torch.stack([torch.as_tensor(RuleBasedController(temp_setpoint_day=18.0 + i, co2_day=600 + 100 * i).settings_vector())
                            for i in range(4)]).to("cuda")
        settings = vecs[torch.arange(B, device="cuda") % 4].contiguous()
        for env in (fused, split):
            env.reset_tensor()
        step_fused = fused.step_rule_based_tensor
        step_split = lambda: split.step_raw_control_tensor(split.rule_controls_tensor(settings))
        step_split_none = lambda: split.step_raw_control_tensor(split.rule_controls_tensor())
        for f in (step_fused, step_split, step_split_none):
            timed(f, 5)
        tf, ts, tn = [], [], []
        for _ in range(ROUNDS):
            tf.append(timed(step_fused, STEPS))
            ts.append(timed(step_split, STEPS))
            tn.append(timed(step_split_none, STEPS))
        t_k = timed(lambda: split.rule_controls_tensor(settings), KERNEL_LAUNCHES)
        say(f"B = {B}")
        say(f"  fused glg_step_rule_based                     {' '.join(f'{t:8.4f}' for t in tf)} ms/step (min {min(tf):.4f})")
        say(f"  glg_rule_controls (per-env) + raw step        {' '.join(f'{t:8.4f}' for t in ts)} ms/step (min {min(ts):.4f})"
            f"  -> {100 * (min(ts) / min(tf) - 1):+.2f} %")
        say(f"  glg_rule_controls (handle settings) + raw step {' '.join(f'{t:8.4f}' for t in tn)} ms/step (min {min(tn):.4f})"
            f"  -> {100 * (min(tn) / min(tf) - 1):+.2f} %")
        say(f"  glg_rule_controls alone (per-env settings)     {1e3 * t_k:8.2f} us per launch ({KERNEL_LAUNCHES} back-to-back launches)")
        say()
        fused.close()
        split.close()
    # one tuner generation against the bare steps it is made of
    tuner = RuleControllerTuner(n_candidates=256, n_elites=32, base_env_params=dict(start_train_day=0, end_train_day=15))
    B, H = tuner.env.num_envs, tuner.horizon
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tuner.generation()
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    tuner.close()
    bare = GreenLightVecEnv(B, auto_reset=False, base_env_params=dict(start_train_day=0, end_train_day=15))
    bare.reset_tensor()
    t_bare = timed(bare.step_rule_based_tensor, H) * H / 1e3
    bare.close()
    say(f"tuner generation: K = 256, S = 16 (GL2009 start days 0-15), {B} envs, horizon {H} (the season)")
    say(f"  one generation (host clock, ends in a synchronise) {t_gen:8.3f} s")
    say(f"  {H} bare glg_step_rule_based launches of {B} envs  {t_bare:8.3f} s   (generation / bare = {t_gen / t_bare:.3f})")
    say()
    say(f"card (read again): {card()}")
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
