#!/usr/bin/env python
"""bench.py -- GreenLight env-steps/sec on B200 (BASELINE.json metric), fp64 parity mode.

Headline workload (config.workload): BASELINE.json configs[1] -- "TomatoEnv 4096 batched envs fp64 parity mode, nominal
parameters, fixed weather year": 4096 envs PER GPU (weak scaling: every rank owns its own 4096-env shard, no collective on
the step path), Bleiswijk GL2009 weather table (start day 0), the package's default integrator contract (graded RK4 with
zero-order hold, n_sub = 260 nominal substeps, 300 RK4 steps per 900 s control interval; DESIGN.md "Integrator contract"),
U(-1,1) float32 actions through the rate-limited action->control map, observations (263 f32), reward, info, termination and
auto-reset all inside the one fused kernel launch per step.

One "step" = one vector env step (B env-steps per GPU).
  value      whole-job env-steps/s with inputs resident in HBM (actions pre-generated on the device, CUDA-event timing per
             step on the launching stream, L2 flushed between steps, max over ranks).
  e2e        the same metric through the numpy SB3-VecEnv call (`env.step(actions)`: host actions -> pinned -> device, kernel,
             obs / reward / done -> host), wall clock around K calls.
  roofline   FP64 pipe (this path is FP64-bound by > 100x over HBM, SURVEY.md 8d): achieved = env-steps/s x algorithmic
             flop per env-step, F = 3968 x (RK4 steps the kernel reports having executed) + 529; peak = DFMA throughput
             measured live on the same GPU (MEASURED_PEAKS.json carries no FP64 figure).  `traffic` / `ncu` come from the
             committed ncu capture and are attached only if that capture was taken with the kernel sources now in the tree.
  configs    further workloads timed inside the same run, each with its own ms_per_step / value / roofline: the equal-
             substep RK4(600) contract at B = 4096 (round 1's headline), the saturated regime B = 262 144 in fp64, BASELINE
             configs[2] (B = 262 144, fp32 throughput mode, uncertainty_scale 0.3, start day randomised over 19 tables), and
             under --gpus 8 also 65 536 envs per GPU.
  cpu_baseline  both CPU arms on the box's host cores over bounded samples: "port" = the oracle with the same RK4 contract,
             "port-implicit" = the oracle's right-hand side under an adaptive variable-order BDF at rtol = atol = 1e-6 (the
             class of solver the reference uses, CasADi CVODES, which is not installable here) -- the faster one is `value`.
  --impl reference  times that faster CPU arm alone (rank 0), sample sized for >= 10 s whatever --steps is.
  --dump-outputs DIR  after the timed steps, writes what the headline's last timed step returned (rank 0's envs) as .npy files, so
             that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs B] [--integrator graded|fixed]
                    [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...      (one rank per GPU)
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "GreenLight env-steps/sec (fp64 parity)"
UNIT = "env-steps/s"
F_RHS, F_SUBSTEP_OVERHEAD, F_STEP_CONST = 880, 448, 529  # SURVEY.md 8d: algorithmic flop model
F_RK4_STEP = 4 * F_RHS + F_SUBSTEP_OVERHEAD               # 3968 per RK4 step


def flop_per_env_step(rk4_steps):
    return F_RK4_STEP * rk4_steps + F_STEP_CONST


def algorithmic_bytes_per_env_step(obs_dim):
    # SURVEY.md 8d: read x,u,action,scalars ; write x,u,obs,reward,done,info (+ per-CTA weather tile, amortised)
    return (224 + 48 + 24 + 16) + (224 + 48 + obs_dim * 4 + 8 + 1 + 88) + 16


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much, all files together


def dump_outputs(path, obs, reward, done):
    """Writes one step's outputs to `path`: obs.npy [n, obs_dim] f32, reward.npy [n] f64, done.npy [n] f32 (0 / 1) and
    env_index.npy [n] f64, the env each row belongs to.  All rows if they fit in DUMP_BYTES, else a sample of rows drawn with a
    fixed seed, so that the same batch size always selects the same envs."""
    B = obs.shape[0]
    row_bytes = obs.shape[1] * 4 + 8 + 4 + 8
    idx = np.arange(B)
    if B * row_bytes > DUMP_BYTES - 4096:  # 4096: room for the four .npy headers
        idx = np.sort(np.random.default_rng(0).choice(B, (DUMP_BYTES - 4096) // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    out = {"obs": obs[idx].astype(np.float32), "reward": reward[idx].astype(np.float64), "done": done[idx].astype(np.float32),
           "env_index": idx.astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def csrc_hash():
    """sha256 (first 16 hex digits) of the kernel sources: an ncu capture is only quoted for the sources it was taken with."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "greenlight-gym2_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def result(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


_REAL_STDOUT = None


def quiet_stdout():
    """Everything this process (or a library it loads: NCCL prints a version banner to stdout when the first communicator is
    created) writes to fd 1 goes to stderr from here on; the one JSON line is written to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def load_inputs():
    from glgym.params import init_default_params
    from glgym.weather import load_weather_data
    return init_default_params().astype(np.float64), load_weather_data(None, "Bleiswijk", "GL", 2009, 0, 60, 49, 900, 10)


# ---------------------------------------------------------------------------------------------------- CPU arms
def oracle_cfg(kind, integrator, n_sub):
    """glgo_env_cfg of a CPU arm: "port" = the same RK4 contract as the GPU arm, "port-implicit" = adaptive BDF at 1e-6."""
    import oracle_binding as ob
    if kind == "port-implicit":
        return ob.default_cfg(n_sub=n_sub, stiff_guard=ob.INTEGRATOR_BDF)
    return ob.default_cfg(n_sub=n_sub, stiff_guard=ob.INTEGRATOR_GRADED if integrator == "graded" else ob.INTEGRATOR_RK4)


def cpu_rate(kind, integrator, n_sub, B, n_steps, threads, warmup=0):
    """(env-steps/s, seconds, right-hand-side evaluations per env-step) of a CPU arm: B envs stepped by `threads` host threads"""
    import oracle_binding as ob
    p, W = load_inputs()
    batch = ob.OracleBatch(W, p, B, oracle_cfg(kind, integrator, n_sub), n_threads=threads)
    rng = np.random.default_rng(0)
    acts = rng.uniform(-1, 1, (warmup + n_steps, B, 6)).astype(np.float32)
    for s in range(warmup):
        batch.step(acts[s])
    w0 = batch.work()
    t0 = time.perf_counter()
    for s in range(n_steps):
        batch.step(acts[warmup + s])
    dt = time.perf_counter() - t0
    work = (batch.work() - w0) / (B * n_steps)
    batch.close()
    return B * n_steps / dt, dt, work * (1 if kind == "port-implicit" else 4)


def cpu_arm(kind, integrator, n_sub, seconds, cores):
    """One CPU arm over a bounded sample sized for about `seconds` of work: 4 envs per thread, as many steps as fit."""
    B = 4 * cores
    probe, _, _ = cpu_rate(kind, integrator, n_sub, B, 2, cores)
    steps = max(3, int(seconds * probe / B))
    rate, dt, rhs = cpu_rate(kind, integrator, n_sub, B, steps, cores)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "rhs_evals_per_env_step": rhs,
            "sample": f"{B} envs x {steps} steps on {cores} threads ({dt:.1f} s), same weather / action distribution"}


def workload_config(args):
    """The `config` both arms report."""
    nominal = 260 if args.integrator == "graded" else 600
    n_sub = args.n_sub or nominal
    integ = (f"graded RK4, zero-order hold: {n_sub} nominal substeps, the first 12 split 16/8/4x4/2x6, transient-stiffness rule "
             f"(300 RK4 steps per interval at n_sub 260)" if args.integrator == "graded" else f"RK4, {n_sub} equal substeps, zero-order hold")
    return {"workload": f"TomatoEnv {args.envs} batched envs per GPU, fp64 parity mode, nominal parameters, fixed weather year "
                        "(BASELINE configs[1])",
            "envs_per_gpu": args.envs, "n_sub": n_sub, "dt": 900, "integrator": integ, "obs_dim": 263,
            "parallelism": f"env-shard x{args.gpus}, no collective on the step path",
            "l2": "GPU arm: flushed between timed steps (256 MiB memset outside the event pair); CPU arm: not applicable",
            "kernel": {0: "GPU arm: glg_step_units_kernel (auto: latency layout, 4 owner + 12 flux-unit warps per 32 envs, up to 2*SMs*32 envs; "
                          "else throughput layout, 4 fused warps per 32 envs x 4 CTAs per SM)",
                       1: "GPU arm: glg_step_kernel (thread per env)", 2: "GPU arm: glg_step_units_kernel latency layout",
                       3: "GPU arm: glg_step_units_kernel throughput layout"}[args.role_warps]}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's CPU implementation of the path.  CasADi / SUNDIALS cannot be installed in this image
    (no wheel, no network), so this is the CPU oracle -- its right-hand side under the adaptive implicit BDF solver at the
    reference's tolerances ("port-implicit", the faster of the two CPU arms) -- on all host threads; rank 0 only.  Each of the
    --steps steps advances a bounded sample of the workload's envs, sized so that the run takes >= 10 s."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_sub = args.n_sub or (260 if args.integrator == "graded" else 600)
    kind = "port-implicit"
    probe, _, _ = cpu_rate(kind, args.integrator, n_sub, 16 * cores, 3, cores, warmup=1)
    sample = max(4 * cores, int(np.ceil(15.0 * probe / max(args.steps, 1) / cores)) * cores)  # envs per step: >= 10 s in total
    rate, dt, rhs = cpu_rate(kind, args.integrator, n_sub, sample, args.steps, cores, warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic actions; Bleiswijk GL2009 weather table shipped with the reference",
        "config": workload_config(args),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "rhs_evals_per_env_step": rhs,
                         "sample": f"each step advances {sample} envs of the workload (the per-env work of the {args.envs}-env batch; the count is "
                                   f"sized for >= 10 s of CPU work) on {cores} host threads; {args.steps} steps in {dt:.1f} s",
                         "note": "CPU oracle right-hand side under an adaptive variable-order BDF (rtol = atol = 1e-6, finite-difference "
                                 "Jacobian, cold start per control interval like CasADi's integrator); the reference's CasADi CVODES "
                                 "extension is not installable here"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------- GPU arm
def time_steps(env, actions, K, Wm, flush, barrier, dev, world):
    """W warm-up steps, then K steps timed one by one with CUDA events on the launching stream (L2 flushed between steps).
    Returns (sum of step times [ms] max over ranks, mean step time of this rank [ms], RK4 steps per env-step, launches)."""
    import torch
    from glgym.distributed import max_over_ranks
    for s in range(Wm):
        env.step_tensor(actions[s % actions.shape[0]])
    env.episode_stats(clear=True)
    launches0 = env.launch_count()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for s in range(K):
        flush.zero_()
        ev[s][0].record()
        env.step_tensor(actions[(Wm + s) % actions.shape[0]])
        ev[s][1].record()
    barrier()
    ms = [a.elapsed_time(b) for a, b in ev]
    micro = env.stats_t[15].item() / (env.num_envs * K)
    return max_over_ranks(sum(ms), dev), float(np.mean(ms)), micro, env.launch_count() - launches0


def extra_config(name, desc, ctor_kwargs, B, K, Wm, flush, barrier, dev, world, rank, local, peak):
    """One entry of the line's `configs` object."""
    import torch
    from glgym.vec_env import GreenLightVecEnv
    try:
        env = GreenLightVecEnv(B, device=local, seed=0, env_id_offset=rank * B, **ctor_kwargs)
        env.reset_tensor()
        g = torch.Generator(device=dev)
        g.manual_seed(99 + rank)
        actions = torch.rand(4, B, 6, device=dev, generator=g) * 2 - 1
        total_ms, mean_ms, micro, _ = time_steps(env, actions, K, Wm, flush, barrier, dev, world)
        finite = bool(torch.isfinite(env.state_t).all().item())
        env.close()
        F = flop_per_env_step(micro)
        per_gpu = B / (mean_ms * 1e-3)
        return {"workload": desc, "envs_per_gpu": B, "value": world * B * K / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / K,
                "steps": K, "warmup": Wm, "rk4_steps_per_env_step": micro, "flop_per_env_step": F, "state_finite": finite,
                "roofline": {"bound": peak[0], "achieved": per_gpu * F / 1e12, "peak": peak[1], "unit": "TFLOP/s",
                             "frac": per_gpu * F / 1e12 / peak[1] if peak[1] else None}}
    except Exception as exc:  # never lose the headline because of an extra measurement
        return {"workload": desc, "error": str(exc)[:300]}


def run_ours(args, rank, world, local):
    import ctypes as C
    import torch
    from glgym import _lib
    from glgym.distributed import max_over_ranks
    from glgym.vec_env import GreenLightVecEnv
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B, K, Wm = args.envs, args.steps, args.warmup
    ctor = dict(device=local, seed=0, env_id_offset=rank * B, role_warps=args.role_warps, precision=args.precision,
                integrator=args.integrator, n_sub=args.n_sub)
    env = GreenLightVecEnv(B, **ctor)
    obs_dim = env.obs_dim
    env.reset_tensor()
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    actions = torch.rand(Wm + K, B, 6, device=dev, generator=g) * 2 - 1
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    L = _lib.load()
    pk64, pk32 = C.c_double(), C.c_double()
    L.glg_measure_fp64_peak(local, C.byref(pk64))
    L.glg_measure_fp32_peak(local, C.byref(pk32))
    peak64, peak32 = ("fp64", pk64.value / 1e12), ("fp32", pk32.value / 1e12)

    # ---- device-resident throughput
    sampler = ClockSampler(local)
    sampler.start()
    total_ms, kernel_ms, micro, launches = time_steps(env, actions, K, Wm, flush, barrier, dev, world)
    value = world * B * K / (total_ms * 1e-3)
    finite = bool(torch.isfinite(env.state_t).all().item())
    # what step_tensor returned in the last timed step (device views the next step overwrites): host copies, written at the end
    last_step = (env.obs_t.cpu().numpy(), env.reward_t.cpu().numpy(), env.done_t.cpu().numpy()) if args.dump_outputs and rank == 0 else None

    # ---- end to end through the numpy VecEnv API (host buffers, copies inside the timed region)
    a_host = actions[Wm:].cpu().numpy()
    for s in range(min(2, K)):
        env.step(a_host[s])
    barrier()
    t0 = time.perf_counter()
    for s in range(K):
        obs, rew, done, infos = env.step(a_host[s])
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_s = max_over_ranks(e2e_s, dev)
    e2e_value = world * B * K / e2e_s
    sampler.stop_flag = True  # clocks are sampled over both timed regions (device-resident and end-to-end)
    sampler.join(timeout=1.0)
    # the opt-in split observation layout (per-env columns over PCIe, forecast block from the host's weather bank)
    e2e_split = None
    try:
        for s in range(min(2, K)):
            env.step_split(a_host[s])
        barrier()
        t0 = time.perf_counter()
        for s in range(K):
            env.step_split(a_host[s])
        e2e_split = world * B * K / max_over_ranks(time.perf_counter() - t0, dev)
    except Exception:
        pass
    # the same loop (a) returning a fresh pageable copy per step (obs_ring = 0: the reference's array semantics), (b) with one
    # device->host copy of the whole observation array instead of the overlapped host-side forecast fill (host_obs="copy")
    def e2e_variant(**kw):
        try:
            cenv = GreenLightVecEnv(B, **dict(ctor, **kw))
            cenv.reset()
            for s in range(min(2, K)):
                cenv.step(a_host[s])
            barrier()
            t0 = time.perf_counter()
            for s in range(K):
                cenv.step(a_host[s])
            rate = world * B * K / max_over_ranks(time.perf_counter() - t0, dev)
            cenv.close()
            return rate
        except Exception:
            return None
    e2e_copy = e2e_variant(obs_ring=0)
    e2e_full_d2h = e2e_variant(host_obs="copy")

    # ---- the one collective of the path, on hardware: episode statistics summed over the ranks' handles (SURVEY 8e)
    stats_allreduce = None
    try:
        x, u, k = env.get_state()
        env.set_state(timestep=np.full(B, env.N, dtype=np.int32))  # forced episode end: the next step terminates every env
        env.episode_stats(clear=True)
        env.step_tensor(actions[0])
        env.init_stats_allreduce()
        barrier()
        local_eps = float(env.stats_t[0].item())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        env.allreduce_stats()  # first call: communicator warm-up
        torch.cuda.synchronize(dev)
        glob_eps = float(env.stats_t[0].item())
        reps = 20
        zero = torch.zeros_like(env.stats_t)
        env.stats_t.copy_(zero)
        barrier()
        e0.record()
        for _ in range(reps):
            env.allreduce_stats()
        e1.record()
        torch.cuda.synchronize(dev)
        us = max_over_ranks(e0.elapsed_time(e1) / reps * 1e3, dev)
        stats_allreduce = {"us": us, "episodes_local": local_eps, "episodes_global": glob_eps, "ranks": world,
                           "ok": bool(local_eps == B and glob_eps == world * B),
                           "api": "glg_allreduce_stats: ncclAllReduce(sum, 16 x f64) on the handle's statistics buffer"}
    except Exception as exc:
        stats_allreduce = {"error": str(exc)[:300]}
    env.close()

    # ---- further workloads inside the same run, K timed steps each like the headline
    Wx = 3
    configs = {}
    other = "fixed" if args.integrator == "graded" else "graded"
    configs[f"config2_{other}"] = extra_config(
        f"config2_{other}", f"BASELINE configs[1] with integrator='{other}' (" + ("RK4, 600 equal substeps: round 1's headline contract)" if other == "fixed"
                                                                                   else "graded RK4, n_sub 260)"),
        dict(integrator=other, precision="fp64"), B, K, Wm, flush, barrier, dev, world, rank, local, peak64)
    configs["saturated_fp64"] = extra_config(
        "saturated_fp64", "262 144 envs per GPU, fp64 parity mode, nominal parameters, one weather table (the regime the one-CTA-per-32-envs "
        "design is built for; BASELINE configs[4] sweep point)", dict(integrator=args.integrator, precision="fp64"), 262144, K, Wx, flush,
        barrier, dev, world, rank, local, peak64)
    configs["config3_fp32_uncertainty"] = extra_config(
        "config3_fp32_uncertainty", "BASELINE configs[2]: 262 144 envs per GPU, fp32 throughput mode (flux units fp32, RK4 state fp64), "
        "uncertainty_scale 0.3 (device Philox, 34 draws per env-step), start day randomised over the 19 Bleiswijk GL2009 tables; 24 warm-up "
        "steps: in the first steps after a reset ~10 % of the envs are pruned by the harvest terms (cLeafMax redrawn below the initial "
        "leaf mass) and their CTAs run twice the RK4 steps (27.5 ms per step; 20.5 after 12 steps); a whole season averages 18.2 ms per "
        "step (profiles/r2_season_throughput.txt)",
        dict(integrator=args.integrator, precision="fp32", uncertainty_scale=0.3, base_env_params=dict(start_train_day=0, end_train_day=18)),
        262144, K, 24, flush, barrier, dev, world, rank, local, peak32)
    if world >= 8:
        configs["config4_65536_per_gpu"] = extra_config(
            "config4_65536_per_gpu", "BASELINE configs[3] shape: 65 536 envs per GPU x 8 GPUs, fp64, U(-1,1) actions resident on the device",
            dict(integrator=args.integrator, precision="fp64"), 65536, K, Wx, flush, barrier, dev, world, rank, local, peak64)

    if rank == 0:
        peak = peak64 if args.precision == "fp64" else peak32
        per_gpu_rate = B / (kernel_ms * 1e-3)
        F = flop_per_env_step(micro)
        achieved_tf = per_gpu_rate * F / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_gbs = per_gpu_rate * algorithmic_bytes_per_env_step(obs_dim) / 1e9
        traffic, ncu_info = None, None
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            ent = prof.get(f"{args.integrator}_{args.precision}_B{B}")
            if ent and prof.get("csrc_sha16") == csrc_hash():
                traffic = ent.get("dram_bytes_per_launch")
                ncu_info = {k: ent.get(k) for k in ("fp64_pipe_active_pct", "issue_active_pct", "kernel", "source")}
            elif ent:
                ncu_info = {"stale": "profiles/r2_traffic.json was captured with other kernel sources (csrc hash differs); not quoted"}
        except Exception:
            pass
        cores = os.cpu_count() or 1
        n_sub = env.n_sub
        arm_rk4 = cpu_arm("port", args.integrator, n_sub, 8.0, cores)
        arm_bdf = cpu_arm("port-implicit", args.integrator, n_sub, 10.0, cores)
        best = arm_bdf if arm_bdf["value"] >= arm_rk4["value"] else arm_rk4
        line = {
            "metric": METRIC if args.precision == "fp64" else "GreenLight env-steps/sec (fp32 throughput mode)",
            "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if args.precision == "fp64" else "f32 (RK4 state f64)",
            "data": "synthetic actions; Bleiswijk GL2009 weather table shipped with the reference",
            "config": workload_config(args),  # identical in both arms
            "run": {"state_finite": finite, "rk4_steps_per_env_step": micro},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 6 * 4,
                    "d2h_bytes_per_step": B * (obs_dim - 240) * 4 + 2 * B * 4 + B * 8 + B,
                    "api": "GreenLightVecEnv(...).step(numpy) -> glg_step_host with the constructor's defaults: host actions in, observations "
                           "[B, 263] / rewards / dones out as numpy arrays (observations are page-locked buffers of a ring of 4: valid for the "
                           "next 3 steps).  Default host_obs='overlap': the 240-float forecast block of every row is written by the host from "
                           "its copy of the weather bank while the kernel runs and verified after it; the 23 other columns, timestep, table, "
                           "reward and done cross PCIe",
                    "value_full_d2h_copy": e2e_full_d2h, "full_d2h_copy_bytes_per_step": B * obs_dim * 4 + B * 8 + B,
                    "value_with_copy_per_step": e2e_copy,
                    "value_split_layout": e2e_split, "split_layout_d2h_bytes_per_step": B * (obs_dim - 240) * 4 + B * 8 + B * 8 + B,
                    "split_layout_note": "opt-in env.step_split(): every column but the 240-float forecast block crosses PCIe; the forecast is "
                                         "read from the host's copy of the weather bank"},
            "gpu_launches": int(launches), "configs": configs, "stats_allreduce": stats_allreduce,
            "clocks": sampler.result(),
            "roofline": {"bound": args.precision, "achieved": achieved_tf, "peak": peak[1], "unit": "TFLOP/s",
                         "frac": achieved_tf / peak[1] if peak[1] else None, "traffic": traffic,
                         "peak_source": ("glg_measure_fp64_peak: DFMA" if args.precision == "fp64" else "glg_measure_fp32_peak: FFMA")
                                        + " micro-benchmark measured live on this GPU (MEASURED_PEAKS.json has no FP64/FP32 pipe entry)",
                         "flop_per_env_step": F, "flop_model": "3968 x RK4 steps executed (kernel counter) + 529", "kernel_ms": kernel_ms,
                         "ncu": ncu_info, "csrc_sha16": csrc_hash(),
                         "hbm": {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                                 "bytes_per_env_step": algorithmic_bytes_per_env_step(obs_dim),
                                 "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650"}},
            "cpu_baseline": dict(best, arms={"port": arm_rk4, "port-implicit": arm_bdf},
                                 note="value = the faster CPU arm; 'port' runs the GPU arm's RK4 contract, 'port-implicit' an adaptive BDF at the "
                                      "reference solver's tolerances (rtol = atol = 1e-6) on the same right-hand side"),
        }
        if last_step is not None:
            dump_outputs(args.dump_outputs, *last_step)
        emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="envs per GPU")
    ap.add_argument("--integrator", default=None, choices=["graded", "fixed"], help="default: the package's default contract")
    ap.add_argument("--n-sub", type=int, default=None, help="nominal RK4 substeps (default 260 graded / 600 fixed)")
    ap.add_argument("--role-warps", type=int, default=0)
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"],
                    help="fp64 = parity mode (the BASELINE metric); fp32 = throughput mode (flux groups in fp32, RK4 state in fp64)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's last timed step (observations, rewards, dones of rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the CPU arm's sample size follows its measured speed, so its inputs vary")
    if args.integrator is None:
        args.integrator = "graded"  # == glgym.vec_env.DEFAULT_INTEGRATOR (not imported here: --impl reference must not need torch)
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        from glgym.distributed import init_from_env
        import torch
        torch.cuda.set_device(local)
        init_from_env("nccl")
    run_ours(args, rank, world, local)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
