"""Linearisation (glg_linearize, glg_rhs_jacobian_batch) against the step and against the forward-difference alternative, in
one command, on one GPU:

  - glg_linearize of a handle against glg_step of the same handle, alternating in one run, at B = 256, 4096 and 65 536
    (default env: fp64, graded integrator, n_sub 260), CUDA events over REPS calls per round;
  - glg_rhs_jacobian_batch at the same sizes;
  - the forward-difference alternative: 35 B rows (the point and one step per state and control) through glg_evalf_batch_ex;
  - accuracy of forward differences (step 1e-6 max(|x|, 1e-3)) against the AD Jacobian at B = 256, scaled D^-1 J D.

    python tools/linearize_time.py [--out profiles/linearize_kernels.txt] [--sizes 256,4096,65536]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import numpy as np
import torch

from glgym.model import GreenLight
from glgym.vec_env import GreenLightVecEnv

REPS, ROUNDS = 5, 3
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


def fd_rows(x, u):
    """[35 B] rows: the point, then one forward step per state and control."""
    B = x.shape[0]
    D = torch.cat([x.abs().clamp_min(1e-3), torch.ones_like(u)], 1)
    h = 1e-6 * D
    X = x[:, None].repeat(1, 35, 1)
    U = u[:, None].repeat(1, 35, 1)
    for j in range(34):
        if j < 28:
            X[:, 1 + j, j] += h[:, j]
        else:
            U[:, 1 + j, j - 28] += h[:, j]
    return X.reshape(-1, 28).contiguous(), U.reshape(-1, 6).contiguous(), h, D


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "linearize_kernels.txt"))
    ap.add_argument("--sizes", default="256,4096,65536")
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"card: {card()}")
    say(f"torch {torch.__version__}; default env (fp64, graded integrator, n_sub 260), states after 20 rule-based steps of a "
        f"January start; CUDA events, {ROUNDS} rounds x {REPS} calls, paths alternating in each round")
    say()
    say(f"{'B':>7} {'step ms':>9} {'linearize ms':>13} {'ratio':>6} {'rhs_jac ms':>11} {'FD 35B evalF ms':>16} {'FD/AD':>6}")
    for B in [int(s) for s in args.sizes.split(",")]:
        env = GreenLightVecEnv(B, seed=1)
        env.reset_tensor()
        for _ in range(20):
            env.step_rule_based_tensor()
        m = GreenLight(integrator=env.integrator, n_sub=env.n_sub)
        u = env.rule_controls_tensor().clone()
        x = env.state_t.T.contiguous()
        st = env.state_dict()
        W = env.weather_tables
        rows = torch.as_tensor(np.stack([W[st["table"][e], min(st["timestep"][e], W.shape[1] - env.Np - 1)] for e in range(B)]),
                               device="cuda")
        p = torch.as_tensor(np.asarray(env.p, dtype=np.float64), device="cuda")
        X, U, h, D = fd_rows(x, u)
        Dd = rows.repeat_interleave(35, 0).contiguous()
        snap = env.state_dict()
        # warm-up of every path
        env.linearize_tensor(u)
        m.rhs_jacobian_batch(x, u, rows, p)
        m.evalF_batch(X, U, Dd, p)
        env.step_raw_control_tensor(u)
        env.load_state_dict(snap)
        torch.cuda.synchronize()
        ts, tl, tr, tf = [], [], [], []
        for _ in range(ROUNDS):
            env.load_state_dict(snap)
            ts.append(timed(lambda: env.step_raw_control_tensor(u), REPS))
            env.load_state_dict(snap)
            tl.append(timed(lambda: env.linearize_tensor(u), REPS))
            tr.append(timed(lambda: m.rhs_jacobian_batch(x, u, rows, p), REPS))
            tf.append(timed(lambda: m.evalF_batch(X, U, Dd, p), max(1, REPS // 2)))
        s, l, r, f = (float(np.median(v)) for v in (ts, tl, tr, tf))
        say(f"{B:>7} {s:>9.3f} {l:>13.3f} {l / s:>6.2f} {r:>11.3f} {f:>16.3f} {f / l:>6.2f}")
        if B == 256:
            env.load_state_dict(snap)
            _, A, Bu = env.linearize_tensor(u)
            out = m.evalF_batch(X, U, Dd, p).reshape(B, 35, 28)
            Jfd = ((out[:, 1:] - out[:, :1]) / h[:, :, None]).transpose(1, 2)  # [B, 28, 34]
            J = torch.cat([A, Bu], 2)
            E = ((J - Jfd) * D[:, None, :] / D[:, :28, None]).abs()
            acc = (f"accuracy at B = 256: forward differences (step 1e-6 max(|x|, 1e-3)) against the AD Jacobian, scaled "
                   f"entries: median {E.median().item():.2e}, 99th percentile {torch.quantile(E.flatten().float(), 0.99).item():.2e}, "
                   f"max {E.max().item():.2e}")
        env.close()
    say()
    say(acc)
    with open(args.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
