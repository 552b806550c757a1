"""Receding-horizon planner (glgym.planning.DevicePlanner, csrc/glg_plan.cuh): time per decision against the step launches it is
made of, in one command.

For (B, K) = (16, 256), (64, 1024), (256, 1024) with H = 12, I = 3, E = K / 8, default env (fp64, graded integrator):
  - time per decision (plan() + shift(), CUDA events around DECISIONS warmed-up decisions);
  - time of H I bare glg_step launches of a separate B K env handle in the same run (what a decision cannot go below);
  - the new kernels' share of a decision: torch.profiler (CUDA activities) over one decision in a pass of its own, glg_plan_* kernel
    time against all kernel time;
  - a bytes model of the new kernels per decision and the rate it implies.

    python tools/plan_time.py [--out profiles/plan_kernels.txt]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import torch

from glgym.planning import DevicePlanner
from glgym.vec_env import GreenLightVecEnv

H, I = 12, 3
CASES = ((16, 256), (64, 1024), (256, 1024))
WARM, DECISIONS = 1, 3
assert torch.cuda.is_available(), "this measurement needs the GPU"


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def plan_bytes(B, K, E):
    """HBM bytes the glg_plan_* kernels move per decision (I iterations).  Per iteration: fan-out (read the B source states:
    36 doubles + 3 words; write B K planning states, zeroed accumulators, return and alive flag), sample (read mean / std, write
    H B K 6 floats), H accumulations (read reward, done, return, alive; write return, alive), update (read B K returns and the
    elites' candidates twice; write mean, std and, once, the actions)."""
    BK = B * K
    fan = B * (36 * 8 + 12) + BK * (36 * 8 + 12 + 8 + 4 + 11 * 8 + 1 + 8 + 1)
    sample = 2 * H * B * 6 * 4 + H * BK * 6 * 4
    accum = H * BK * (8 + 1 + 8 + 1 + 8 + 1)
    update = BK * 8 + 2 * B * E * H * 6 * 4 + 2 * H * B * 6 * 4
    return I * (fan + sample + accum + update) + B * 6 * 4


def ev():
    return torch.cuda.Event(enable_timing=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plan_kernels.txt"))
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"card: {card()}")
    say(f"torch {torch.__version__}; H = {H}, I = {I}, E = K / 8; default env (fp64, graded integrator, n_sub 260), January start states")
    say(f"decision = plan() + shift(), CUDA events over {DECISIONS} decisions after {WARM} warm-up; bare steps = H I = {H * I} "
        "glg_step launches of a B K handle, events, same run; kernel share from torch.profiler over one decision")
    say()
    for B, K in CASES:
        E = K // 8
        env = GreenLightVecEnv(B)
        env.reset_tensor()
        planner = DevicePlanner(env, H, K, E, I, seed=0)
        for _ in range(WARM):
            planner.plan()
            planner.shift()
        a, b = ev(), ev()
        a.record()
        for _ in range(DECISIONS):
            planner.plan()
            planner.shift()
        b.record()
        torch.cuda.synchronize()
        t_dec = a.elapsed_time(b) / DECISIONS
        # the same work's floor: H I bare steps of a B K handle
        bare = GreenLightVecEnv(B * K, auto_reset=False)
        bare.reset_tensor()
        acts = torch.zeros(B * K, 6, device="cuda")
        bare.step_tensor(acts)
        a, b = ev(), ev()
        a.record()
        for _ in range(H * I):
            bare.step_tensor(acts)
        b.record()
        torch.cuda.synchronize()
        t_bare = a.elapsed_time(b)
        bare.close()
        # kernel split of one decision
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            planner.plan()
            planner.shift()
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA":
                per[e.name] = per.get(e.name, 0.0) + e.time_range.elapsed_us()
        total = sum(per.values())
        new = {n: t for n, t in per.items() if "glg_plan_" in n}
        t_new = sum(new.values())
        nb = plan_bytes(B, K, E)
        say(f"B = {B}, K = {K} ({B * K} planning envs), E = {E}")
        say(f"  decision                      {t_dec:10.2f} ms   ({B / (t_dec * 1e-3):.0f} env decisions/s)")
        say(f"  {H * I} bare steps of {B * K} envs  {t_bare:10.2f} ms   (decision / bare = {t_dec / t_bare:.3f})")
        say(f"  profiled decision: kernels {total / 1e3:.2f} ms, glg_plan_* {t_new / 1e3:.3f} ms = {100 * t_new / total:.2f} %")
        for n, t in sorted(new.items(), key=lambda kv: -kv[1]):
            short = n.split("(")[0].replace("void ", "")
            say(f"      {short:28s} {t / 1e3:9.3f} ms")
        say(f"  bytes model glg_plan_* {nb / 1e6:8.2f} MB per decision -> {nb / (t_new * 1e-6) / 1e9:.0f} GB/s over their kernel time")
        say()
        planner.close()
        env.close()
    say(f"card (read again): {card()}")
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
