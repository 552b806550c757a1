"""CPU tier: host-side mirror of the reference interface (parameters, weather, controller), the host build of the
kernel math against the oracle, and the C-ABI library's exported surface."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle_binding as ob
from conftest import GOLDEN, ROOT, rel_err

DP = C.POINTER(C.c_double)


def P(a):
    return a.ctypes.data_as(DP)


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(os.path.join(ROOT, "tests", "hostmath", "libhostmath.so"))
    lib.hm_evalf.argtypes = [DP, DP, DP, DP, C.c_double, C.c_int, C.c_int, DP]
    lib.hm_rhs_units.argtypes = [DP, DP, DP, DP, C.c_int, C.c_int, C.c_int, DP]
    lib.hm_rhs_stiffness.argtypes = [DP, DP, DP, DP]
    lib.hm_rhs_stiffness.restype = C.c_double
    return lib


def test_parameter_table_matches_reference():
    from glgym.params import init_default_params, PARAM_NAMES
    ref = np.load(os.path.join(GOLDEN, "params_numpy2.npy"))
    assert init_default_params(208, legacy_promotion=False).dtype == np.float32
    assert np.array_equal(init_default_params(208, legacy_promotion=False), ref)  # what the reference yields under numpy 2
    legacy = init_default_params(208)
    assert list(np.nonzero(legacy != ref)[0]) == [169, 171]  # SURVEY.md B.4: numpy-1.26 promotion changes exactly these
    assert float(legacy[169]) == 0.18197675049304962 and float(legacy[171]) == 6746.373046875
    assert len(PARAM_NAMES) == 208 and PARAM_NAMES[46] == "aFlr" and PARAM_NAMES[154] == "rgFruit"
    with pytest.raises(ValueError):
        init_default_params(100)


def test_weather_builder_matches_reference(weather0):
    from glgym.weather import load_weather_data, init_state
    g = np.load(os.path.join(GOLDEN, "weather_golden.npz"))
    assert tuple(g["shape"]) == weather0.shape == (10464, 10)
    assert np.array_equal(weather0[::97], g["sample_sd0"])
    assert np.array_equal(init_state(weather0[0]), g["x0"])
    for sd in (0, 7, 18):
        W = weather0 if sd == 0 else load_weather_data(None, "Bleiswijk", "GL", 2009, sd, 60, 49, 900, 10)
        assert np.array_equal(W[0], g["first"][sd]) and np.array_equal(W[-1], g["last"][sd])
        assert np.allclose([W.sum(), (W * np.arange(1, 11)).sum(), np.abs(W).max()], g["sums"][sd], rtol=1e-14, atol=0)
    with pytest.raises(ValueError):  # start day 19 runs out of rows even with GL2010 appended (SURVEY B.5)
        load_weather_data(None, "Bleiswijk", "GL", 2009, 19, 60, 49, 900, 10)


def test_rule_based_controller_matches_reference(shell_trace, weather0):
    from glgym.controller import RuleBasedController
    from glgym.weather import init_state
    t, c = shell_trace, RuleBasedController()
    x, hod, doy = init_state(weather0[0]), 0.0, 0.0
    for s in range(t["rb_u"].shape[0]):
        assert np.array_equal(c.predict(x, weather0[s], hod, doy)[0], t["rb_u"][s]), s
        x, hod, doy = t["rb_x"][s], (hod + 0.25) % 24, doy + 900 / 86400
    # batch form = row-wise form
    X = np.stack([t["rb_x"][3], t["rb_x"][30]])
    U = c.predict(X, np.stack([weather0[4], weather0[31]]), np.array([1.0, 7.75]), np.array([0.04, 0.32]))
    assert np.array_equal(U[1], c.predict(X[1], weather0[31], 7.75, 0.32)[0])


def test_rule_based_controller_known_answers():
    """Oracle restatement and host port of RuleBasedController.predict against 800 known-answer vectors produced by the
    reference's own class (tests/golden/make_golden.py: shipped settings, wrapping lamp window, day-of-year window,
    lamps_on == lamps_off, non-default thresholds)."""
    import oracle_binding as ob
    from glgym.controller import RuleBasedController, DEFAULT_SETTINGS
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "ctrl_golden.npz"))
    names = [str(n) for n in z["names"]]
    assert names == list(DEFAULT_SETTINGS)  # the settings-vector order of the C-ABI
    assert (z["u"][:, 4] > 0).sum() > 50 and (z["u"][:, 5] > 0).sum() > 20  # lamps / blackout screen exercised
    worst = 0.0
    for i in range(z["u"].shape[0]):
        u = ob.rule_control(z["settings"][i], z["x"][i], z["d"][i], z["hod"][i], z["doy"][i])
        worst = max(worst, np.abs(u - z["u"][i]).max())
        c = RuleBasedController(**dict(zip(names, z["settings"][i])))
        assert np.array_equal(c.settings_vector(), z["settings"][i])
        with np.errstate(all="ignore"):
            assert np.array_equal(c.predict(z["x"][i], z["d"][i], z["hod"][i], z["doy"][i])[0], z["u"][i]), i
    assert worst <= 4e-16  # glibc exp vs numpy exp: one rounding of a value in [0, 1]


def test_oracle_rule_based_step_matches_reference_trace(shell_trace, weather0, params64):
    """Controller in the loop (glgo_env_step_rule) reproduces the reference's rule-based episode prefix."""
    import oracle_binding as ob
    from glgym.controller import RuleBasedController
    t = shell_trace
    env = ob.OracleEnv(weather0, params64, ob.default_cfg(n_sub=int(t["n_sub"])))
    s29 = RuleBasedController().settings_vector()
    for s in range(t["rb_u"].shape[0]):
        obs, r, done, info = env.step_rule(s29)
        assert np.abs(env.u - t["rb_u"][s]).max() <= 1e-11, s  # closed loop: 1e-15 state differences times the sigmoid gains
        assert abs(r - t["rb_reward"][s]) <= 1e-9
    assert np.max(np.abs(env.x - t["rb_x"][-1]) / np.maximum(np.abs(t["rb_x"][-1]), 1e-3)) <= 1e-9


def test_kernel_math_restructuring_matches_oracle(hm, rhs_golden):
    """The hoisted / streaming RHS of csrc/glg_model.h (host build) and its unit-split form (csrc/glg_units.h, every unit ->
    warp assignment the kernel can be built with) against the oracle."""
    g = rhs_golden
    worst = np.zeros(28)
    for i in range(g["x"].shape[0]):
        x, u, d, p = (g[k][i].copy() for k in ("x", "u", "d", "p"))
        general = 0 if hm.hm_nominal_structure(P(p)) else 1
        assert general == (1 if i % 4 == 3 else 0)
        f, s1 = g["f"][i], np.zeros(28)
        hm.hm_rhs(P(x), P(u), P(d), P(p), general, P(s1))
        scale = np.maximum(np.abs(f), 1e-12 * np.maximum(1.0, np.abs(x)))
        worst = np.maximum(worst, np.abs(s1 - f) / scale)
        lam = hm.hm_rhs_stiffness(P(x), P(u), P(d), P(p))
        for ng in (4, 8, 12, 13):
            s2 = np.zeros(30)
            hm.hm_rhs_units(P(x), P(u), P(d), P(p), general, ng, 0, P(s2))
            assert np.all(np.abs(s1 - s2[:28]) <= 1e-12 * np.maximum(np.abs(s1), 1e-9 * np.maximum(1, np.abs(x)))), (i, ng)
            assert abs(s2[29] - lam) <= 1e-12 * abs(lam), (i, ng)  # transient-stiffness estimate of the graded integrator
    # derivative-level agreement; the two carbohydrate balances cancel to ~1e-8 of their terms (see DESIGN.md)
    assert np.all(np.delete(worst, [22, 23, 25]) <= 1e-9) and np.all(worst <= 1e-6), worst


def test_kernel_rk4_matches_oracle_per_step(hm, weather0, params64):
    """Teacher-forced: identical (x,u,d,p) into both; gate 1e-9 relative per state per step (measured ~2e-15)."""
    from glgym.weather import init_state
    rng = np.random.default_rng(5)
    x, u, worst = init_state(weather0[0]), np.zeros(6), 0.0
    for k in range(12):
        u = np.clip(u + (rng.uniform(-1, 1, 6).astype(np.float32) * np.float32(0.1)), 0, 1)
        ya, bad = ob.evalf(x, u, weather0[k], params64, 900.0, 600)
        yb = np.zeros(28)
        assert hm.hm_evalf(P(x), P(u), P(weather0[k].copy()), P(params64), 900.0, 600, 0, P(yb)) == 0 and not bad
        worst = max(worst, rel_err(yb, ya))
        x = ya
    assert worst <= 1e-9, worst


def test_branch_free_math_accuracy(hm):
    rng = np.random.default_rng(0)

    def run(op, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros_like(x)
        hm.hm_math(op, P(x), P(y), len(x))
        return y
    x = np.concatenate([rng.uniform(-700, 700, 200000), rng.uniform(-2, 2, 200000)])
    assert np.max(np.abs(run(0, x) / np.exp(x) - 1) - 1.2e-16 * np.abs(x)) <= 2e-15  # 8-instruction exp: one-constant reduction
    assert np.max(np.abs(run(10, x) / np.exp(x) - 1)) <= 4e-16  # glg_exp_acc (controller)
    sat = run(0, np.array([-1e4, 1e4]))
    assert 0 < sat[0] < 1e-300 and 1e300 < sat[1] < np.inf  # saturates, never 0 / inf
    x = np.exp(rng.uniform(-40, 40, 200000))
    assert np.max(np.abs(run(1, x) - np.log(x))) <= 4e-16 * 40
    x = np.exp(rng.uniform(-25, 6, 200000))
    assert np.max(np.abs(run(4, x) / np.cbrt(x) - 1)) <= 4e-16
    assert np.max(np.abs(run(5, x) / x ** 0.66 - 1)) <= 4e-15 and np.max(np.abs(run(6, x) / x ** 0.32 - 1)) <= 2e-15
    # branch-free per-lane root (floor convection): x^(1/3) / x^(1/4), no final correction step => a few ulp
    assert np.max(np.abs(run(8, x) / np.cbrt(x) - 1)) <= 1e-15 and np.max(np.abs(run(9, x) / x ** 0.25 - 1)) <= 1e-15
    assert run(4, np.array([0.0]))[0] == 0.0


def test_capi_exports_every_declared_symbol():
    """Every function include/glgym.h declares is exported by the built library and bound in glgym._lib."""
    from glgym import _lib
    hdr = open(os.path.join(ROOT, "include", "glgym.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(glg_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 30
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()  # raises if the CUDA extension has not been built
    for name in declared:
        assert hasattr(lib, name), name


def test_capi_config_defaults_and_no_cpu_fallback():
    from glgym import _lib
    lib = _lib.load()
    cfg = _lib.GlgConfig()
    lib.glg_default_config(C.byref(cfg))
    assert (cfg.n_sub, cfg.N, cfg.Np, cfg.dt, cfg.auto_reset) == (600, 5760, 48, 900.0, 1)
    assert cfg.delta_u_max == float(np.float32(0.1)) and list(cfg.con_high) == [1600.0, 34.0, 85.0]
    assert abs(cfg.fixed_costs - (15 + 0.015 + 0.07 * 116 + 2) / 365 / 96) < 1e-18 and cfg.env_id_offset == 0
    import torch
    if not torch.cuda.is_available():
        h = C.c_void_p()
        assert lib.glg_create(C.byref(cfg), C.byref(h)) == _lib.GLG_ERR_CUDA  # loud failure, no CPU path
        assert b"no CPU fallback" in lib.glg_last_error(None)
        with pytest.raises(_lib.GlgError):
            _lib.check(_lib.GLG_ERR_CUDA, None, "glg_create")
    cfg.num_envs = 0
    h = C.c_void_p()
    assert lib.glg_create(C.byref(cfg), C.byref(h)) == _lib.GLG_ERR_ARG


def test_results_frame_layout():
    """glgym.evaluation.to_results_frame: one row per step, the reference's Results columns plus `episode` (common/results.py,
    experiments/evaluate_baseline.py:63-67)."""
    from glgym.evaluation import RESULT_COLUMNS_TAIL, to_results_frame
    from glgym.vec_env import obs_names
    cols = obs_names(48)[:23] + RESULT_COLUMNS_TAIL + ["episode"]
    assert len(cols) == 33 and cols[23:29] == ["Rewards", "EPI", "Revenue", "Heat costs", "CO2 costs", "Elec costs"]
    data = np.arange(2 * 3 * 32, dtype=np.float64).reshape(2, 3, 32)
    df = to_results_frame(data, cols)
    assert df.shape == (6, 33) and df["episode"].tolist() == [0, 0, 0, 1, 1, 1]
    assert df["Rewards"].tolist() == data[:, :, 23].ravel().tolist() and df["co2_air"].iloc[4] == data[1, 1, 0]


def test_role_loops_fit_the_instruction_cache():
    """The latency layout's role loops (10 group loops + the owner loop) must together span less than the SM's ~32 KB
    instruction cache: measured on B200, a build whose loops span 32.0-32.5 KB is 3-20 % slower at B = 4096 whatever else
    changed (DESIGN.md "Round-2 kernel experiments").  A code change that grows the loops shows up here, at build time."""
    import shutil
    import subprocess
    import sys
    from glgym import _lib
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    dump = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    path = os.path.join(os.path.dirname(__file__), "..", "tools")
    out = subprocess.run([sys.executable, os.path.join(path, "sass_loop_size.py"), "/dev/stdin"], input=dump, capture_output=True, text=True).stdout
    import re
    m = re.search(r"loops (0x[0-9a-f]+)\.\.(0x[0-9a-f]+)", out)
    assert m, out
    span = int(m.group(2), 16) - int(m.group(1), 16) + 16
    assert span <= 32 * 1024 - 64, f"role loops span {span} B"


def test_bench_contract_helpers():
    """bench.py's workload description, flop model and source hash (the pieces both arms and the committed ncu record depend on)."""
    import argparse
    import json
    import sys
    sys.path.insert(0, ROOT)
    import bench
    args = argparse.Namespace(integrator="graded", n_sub=None, envs=4096, gpus=1, role_warps=0)
    cfg = bench.workload_config(args)
    assert cfg["n_sub"] == 260 and cfg["envs_per_gpu"] == 4096 and "300 RK4 steps" in cfg["integrator"] and "model" not in cfg
    assert "BASELINE configs[1]" in cfg["workload"]
    args.integrator = "fixed"
    assert bench.workload_config(args)["n_sub"] == 600
    assert bench.flop_per_env_step(300) == 3968 * 300 + 529 and bench.flop_per_env_step(600) == 2381329
    assert bench.algorithmic_bytes_per_env_step(263) == 1749
    h = bench.csrc_hash()
    assert len(h) == 16 and int(h, 16) >= 0
    prof = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
    assert {"csrc_sha16", "graded_fp64_B4096", "fixed_fp64_B4096", "graded_fp64_B262144"} <= set(prof)
    assert prof["csrc_sha16"] == open(os.path.join(ROOT, "profiles", "r2_csrc_sha16.txt")).read().strip()


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every row while the files fit the byte limit, above it a fixed seeded sample of rows that stays
    under the limit; float32 / float64 files only."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(0)
    B, D = 300, 263
    obs, rew, done = rng.random((B, D), dtype=np.float32), rng.random(B), (rng.random(B) < 0.1).astype(np.uint8)
    bench.dump_outputs(str(tmp_path / "all"), obs, rew, done)
    z = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in ("obs", "reward", "done", "env_index")}
    assert {a.dtype for a in z.values()} <= {np.dtype(np.float32), np.dtype(np.float64)}
    assert np.array_equal(z["obs"], obs) and np.array_equal(z["reward"], rew) and np.array_equal(z["done"], done)
    assert np.array_equal(z["env_index"], np.arange(B))
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 100 * (D * 4 + 20))
    samples = []
    for tag in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / tag), obs, rew, done)
        assert sum(f.stat().st_size for f in (tmp_path / tag).iterdir()) <= bench.DUMP_BYTES
        samples.append({n: np.load(tmp_path / tag / f"{n}.npy") for n in ("obs", "reward", "done", "env_index")})
    idx = samples[0]["env_index"].astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0)
    assert all(np.array_equal(samples[0][n], samples[1][n]) for n in samples[0])
    assert np.array_equal(samples[0]["obs"], obs[idx]) and np.array_equal(samples[0]["reward"], rew[idx])
