"""Device replay buffer (glgym.replay.DeviceReplayBuffer, csrc/glg_replay.cuh) against the host pipeline it replaces, in one command.

Device: CUDA-event times of glg_replay_store (the VecNormalize statistics + the transition write, after each env step) at
B = 4096 and 65 536, and of glg_replay_sample at n = 256, 4096 and 65 536 (warmed up, 200 calls each), next to the bytes each call
must move and the achieved rate; device bytes per transition against SB3's raw-row layout.
Host alternative at B = 4096 (SAC through SB3 today): env.step(numpy) + a numpy restatement of VecNormalize.step_wait and of
ReplayBuffer.add (tests/test_gpu_replay.py), and ReplayBuffer.sample(n) with VecNormalize + SB3's copy of the batch to the GPU.

    python tools/replay_time.py            # prints the record kept as profiles/replay_kernels.txt
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

from glgym.replay import DeviceReplayBuffer
from glgym.vec_env import GreenLightVecEnv
from test_gpu_replay import NpReplayBuffer
from test_normalize import NpVecNormalize

WARM, CALLS = 20, 200
SAMPLE_N = (256, 4096, 65536)
CAP = {4096: 256, 65536: 64}  # slots per env: 0.23 / 0.93 GB of device buffer, both above the 126 MB L2
dev = torch.device("cuda", 0)
assert torch.cuda.is_available(), "this measurement needs the GPU"


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def store_bytes(B, D, H):
    """HBM bytes one store must move: statistics (obs read twice, normalised obs written, returns) + the transition write (heads of
    the observation kept from the last store and of the new one, action, reward, done, keys, anchors)."""
    stats = B * (3 * D * 4 + 8 + 8 + 1 + 8)
    write = B * (2 * H * 4 + 6 * 4 + 8 + 1 + 8 + 8 + 2 * H * 4 + 2 * 4 + 6 * 4 + 4 + 1 + H * 4 + 8)
    return stats + write


def sample_bytes(n, D, H):
    """Per sampled transition: two heads, two keys, action, reward, done read; two [obs_dim] rows, action, reward, done written.
    The forecast blocks' bank rows (2 x Np x 5 doubles) are read from L2 and not counted."""
    return n * (2 * H * 4 + 2 * 4 + 6 * 4 + 4 + 1 + 2 * D * 4 + 6 * 4 + 4 + 4)


def ev():
    return torch.cuda.Event(enable_timing=True)


print(f"card: {card()}")
print(f"torch {torch.__version__}, {WARM} warm-up calls, {CALLS} timed calls per row, CUDA events\n")
host_ref = {}
for B in (4096, 65536):
    cap = CAP[B]
    env = GreenLightVecEnv(B)
    D, Np = env.obs_dim, env.Np
    H = D - 5 * Np
    rb = DeviceReplayBuffer(env, cap * B, gamma=0.99, seed=1)
    rb.reset()
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    for _ in range(cap):  # fill the ring, so samples spread over the whole buffer
        rb.step(torch.rand(B, 6, device=dev, generator=g) * 2 - 1)
    acts = [torch.rand(B, 6, device=dev, generator=g) * 2 - 1 for _ in range(8)]
    for i in range(WARM):
        rb.step(acts[i % 8])
    e = [(ev(), ev(), ev()) for _ in range(CALLS)]
    for i in range(CALLS):
        e[i][0].record()
        env.step_tensor(acts[i % 8])
        e[i][1].record()
        rb.store(acts[i % 8])
        e[i][2].record()
    torch.cuda.synchronize()
    t_step = np.mean([a.elapsed_time(b) for a, b, _ in e]) * 1e3
    t_store = np.mean([b.elapsed_time(c) for _, b, c in e]) * 1e3
    nb = store_bytes(B, D, H)
    print(f"B = {B}, {cap} slots per env ({cap * B:.3g} transitions), default stack (obs_dim {D}, {H} stored columns + key)")
    print(f"  env step (default integrator)   {t_step:9.1f} us")
    print(f"  glg_replay_store                {t_store:9.1f} us  = {100 * t_store / t_step:.1f} % of the step;  "
          f"bytes model {nb / 1e6:.1f} MB -> {nb / (t_store * 1e-6) / 1e12:.2f} TB/s")
    per_tr = rb.nbytes / (cap * B)
    raw = 2 * D * 4 + 6 * 4 + 3 * 4
    print(f"  device bytes per transition     {per_tr:9.1f} B  (incl. per-env state; SB3 raw rows {raw} B: {raw / per_tr:.1f}x less), "
          f"buffer {rb.nbytes / 1e9:.2f} GB")
    for n in SAMPLE_N:
        for _ in range(WARM):
            rb.sample(n)
        a, b = ev(), ev()
        a.record()
        for _ in range(CALLS):
            rb.sample(n)
        b.record()
        torch.cuda.synchronize()
        t = a.elapsed_time(b) / CALLS * 1e3
        nb = sample_bytes(n, D, H)
        host_ref[(B, n)] = t
        print(f"  glg_replay_sample n = {n:6d}     {t:9.1f} us;  bytes model {nb / 1e6:7.2f} MB -> {nb / (t * 1e-6) / 1e12:.2f} TB/s")
    host_ref[(B, "step")] = t_step + t_store
    rb.close()
    env.close()
    print()

# ---- host alternative at B = 4096: numpy VecEnv step + numpy VecNormalize + numpy ReplayBuffer (SB3's data path)
B, cap = 4096, CAP[4096]
env = GreenLightVecEnv(B)
D = env.obs_dim
vn, buf = NpVecNormalize(B, D, 0.99), NpReplayBuffer(cap * B, B, D)
rng = np.random.default_rng(0)
infos_empty = [{"TimeLimit.truncated": False} for _ in range(B)]
last = env.reset().astype(np.float32)
vn.reset(last.astype(np.float64))


def host_step(actions):
    global last
    obs, rew, dones, infos = env.step(actions)
    obs = obs.copy()
    vn.step(obs.astype(np.float64), rew.astype(np.float64), dones)  # VecNormalize.step_wait
    nxt = obs.copy()
    for i in np.nonzero(dones)[0]:
        nxt[i] = infos[i]["terminal_observation"]
    buf.add(last, nxt, actions, rew, dones, infos_empty)
    last = obs


for _ in range(cap):
    host_step(rng.uniform(-1, 1, (B, 6)).astype(np.float32))
steps = 50
acts = rng.uniform(-1, 1, (steps, B, 6)).astype(np.float32)
t0 = time.perf_counter()
for i in range(steps):
    host_step(acts[i])
t_host_step = (time.perf_counter() - t0) / steps * 1e6
print(f"host alternative, B = {B}, {cap} slots per env ({buf.observations.nbytes * 2 / 1e9:.2f} GB of observation arrays in host memory)")
print(f"  env.step(numpy) + VecNormalize + ReplayBuffer.add   {t_host_step:9.1f} us per step (wall clock, {steps} steps; "
      f"device step + store: {host_ref[(B, 'step')]:.1f} us)")


def host_sample(n):
    b, e = rng.integers(0, buf.size(), n), rng.integers(0, B, n)
    out = [torch.as_tensor(x, device=dev) for x in buf.get_samples(b, e, vn)]  # SB3 ReplayBuffer.to_torch
    torch.cuda.synchronize()
    return out


for n in SAMPLE_N:
    reps = 50 if n < 65536 else 20
    for _ in range(3):
        host_sample(n)
    t0 = time.perf_counter()
    for _ in range(reps):
        host_sample(n)
    t = (time.perf_counter() - t0) / reps * 1e6
    print(f"  ReplayBuffer.sample n = {n:6d} + copy to the GPU     {t:9.1f} us  (device: {host_ref[(B, n)]:.1f} us, {t / host_ref[(B, n)]:.0f}x)")
env.close()
print(f"\ncard (read again): {card()}")
