"""GreenLightVecEnv -- the batched, GPU-resident replacement for the reference's
`SubprocVecEnv([TomatoEnv ...])` stack (gl_gym/RL/utils.py:44-69, gl_gym/environments/tomato_env.py).

One object = B greenhouse envs on one B200; every `step` is ONE fused CUDA kernel launch (csrc/glg_kernels.cuh)
behind the C-ABI in include/glgym.h.  Two ways to drive it:

  * SB3 `VecEnv` protocol with numpy in/out (`reset`, `step_async`/`step_wait`/`step`, `get_attr`, `env_method`,
    ...): drop-in for code written against the reference.  Host<->device copies happen inside `glg_step_host`.
  * tensor fast path (`reset_tensor`, `step_tensor`, `step_raw_control_tensor`): actions are CUDA tensors, the
    returned obs/reward/done are zero-copy torch views of handle-owned device memory; nothing touches the host.

Constructor arguments mirror the reference's YAML (`gl_gym/configs/envs/TomatoEnv.yml`): `base_env_params` =
the GreenLightEnv section, `constraints`, `reward_params`, `observation_modules`, `uncertainty_scale`.
"""
import ctypes as C
from os.path import join

import types

import numpy as np
import torch

from . import _lib
from .params import init_default_params
from .spaces import Box
from .weather import DEFAULT_WEATHER_DIR, load_weather_data

# Integrator contract of a freshly constructed env: "graded" = classical RK4 with zero-order hold on a grid refined at the start
# of every control interval and wherever the transient-stiffness estimate asks for it (n_sub = 260 nominal substeps, 300 RK4
# steps per interval).  Chosen on accuracy grounds (DESIGN.md "Integrator contract"): against tight-tolerance solutions of 250
# rule-based control intervals its worst-step error sits inside the reference solver's 1e-6 band, the fixed 600-substep grid's
# does not.  integrator="fixed" keeps the equal-substep contract (n_sub = 600).
DEFAULT_INTEGRATOR = "graded"

DEFAULT_OBSERVATION_MODULES = [
    "IndoorClimateObservations", "BasicCropObservations", "ControlObservations", "WeatherObservations",
    "TimeObservations", "WeatherForecastObservations",
]
DEFAULT_BASE_ENV_PARAMS = dict(
    weather_data_dir=DEFAULT_WEATHER_DIR, location="Bleiswijk", data_source="GL", num_params=208, nx=28, nu=6, nd=10,
    dt=900, u_min=[0, 0, 0, 0, 0, 0], u_max=[1, 1, 1, 1, 1, 1], delta_u_max=0.1, pred_horizon=0.5, season_length=60,
    start_train_year=2009, end_train_year=2009, start_train_day=0, end_train_day=0, training=True,
)
DEFAULT_CONSTRAINTS = dict(co2_min=300.0, co2_max=1600.0, temp_min=15.0, temp_max=34.0, rh_min=50.0, rh_max=85.0)
DEFAULT_REWARD_PARAMS = dict(
    fixed_greenhouse_cost=15.0, fixed_co2_cost=0.015, fixed_lamp_cost=0.07, fixed_screen_cost=2.0, elec_price=0.3,
    heating_price=0.09, co2_price=0.3, fruit_price=1.6, dmfm=0.065, pen_weights=[4.0e-4, 5.0e-3, 7.0e-4], pen_lamp=0.1,
)
_EMPTY_INFO = types.MappingProxyType({})

INFO_KEYS = ("EPI", "revenue", "variable_costs", "fixed_costs", "co2_cost", "heat_cost", "elec_cost",
             "temp_violation", "co2_violation", "rh_violation", "lamp_violation")


def _raw_stream(device_index):
    """cudaStream_t of torch's current stream on the device (the cheap accessor where this torch has it)."""
    try:
        return torch._C._cuda_getCurrentRawStream(device_index)
    except AttributeError:
        return torch.cuda.current_stream(device_index).cuda_stream


class _DevArray:
    """Zero-copy view of handle-owned device memory through __cuda_array_interface__."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


class _EnvCompanion:
    """Base of the device objects created on an env (DeviceRollout, DeviceReplayBuffer, DevicePlanner).  Each owns one C object
    (`create(env._h, &cfg, &obj)`), so several may share an env; close() frees it, before or after the env is closed."""
    _kind = ""     # what the error messages call it
    _destroy = ""  # name of the C destructor

    def __init__(self, env, create, cfg):
        self.env, self._lib = env, env._lib
        self._obj = C.c_void_p()
        _lib.check(getattr(self._lib, create)(env._h, C.byref(cfg), C.byref(self._obj)), env._h, create)

    def _view(self, ptr, shape, typestr):
        return torch.as_tensor(_DevArray(ptr, shape, typestr), device=self.env.device)

    def _live(self):
        if not self._obj:
            raise RuntimeError(f"the {self._kind} is closed")
        if not self.env._h:
            raise RuntimeError(f"the env of this {self._kind} is closed")
        return self._obj

    def close(self):
        if getattr(self, "_obj", None):
            getattr(self._lib, self._destroy)(self._obj)
            self._obj = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# observation modules (observations.py:35-182): name -> (id in glg_config.obs_modules, names, (low, high) of its Box)
_WEATHER_NAMES = ["glob_rad", "temp_out", "rh_out", "co2_out", "wind_speed"]
OBSERVATION_MODULES = {
    "StateObservations": (1, ["co2_air", "co2_top", "temp_air", "temp_top", "can_temp", "covin_temp", "covex_temp", "thScr_temp",
                              "flr_temp", "pipe_temp", "soil1_temp", "soil2_temp", "soil3_temp", "soil4_temp", "soil5_temp",
                              "vp_air", "vp_top", "lamp_temp", "intlamp_temp", "grow_pipe_temp", "blscr_temp", "24_can_temp",
                              "cBuf", "cleaves", "cstem", "cFruit", "tsum"], (-np.inf, np.inf)),
    "IndoorClimateObservations": (2, ["co2_air", "temp_air", "rh_air", "pipe_temp"], (-1e-4, 1e4)),
    "BasicCropObservations": (3, ["24CanTemp", "cFruit", "tSum"], (-1e-4, 1e4)),
    "ControlObservations": (4, ["uBoil", "uCo2", "uThScr", "uVent", "uLamp", "uBlScr"], (0.0, 1.0)),
    "WeatherObservations": (5, list(_WEATHER_NAMES), (-1e-4, 1e4)),
    "TimeObservations": (6, ["timestep", "day of year sin", "day of year cos", "hour of day sin", "hour of day cos"], (-1e-4, 1e4)),
    "WeatherForecastObservations": (7, None, (-1e-4, 1e4)),  # 5 Np entries
}


def obs_names(Np, modules=None):
    """Same names as TomatoEnv.get_obs_names() (tomato_env.py:200-206) for an ordered module list (default stack if None)."""
    names = []
    for m in (modules or DEFAULT_OBSERVATION_MODULES):
        n = OBSERVATION_MODULES[m][1]
        names += list(n) if n is not None else _WEATHER_NAMES * Np
    return names


class SplitObs:
    """Observation batch in split form (GreenLightVecEnv.step_split): the per-env columns as they came over PCIe plus what is
    needed to read each row's forecast block from the host's copy of the weather bank."""

    def __init__(self, head, timestep, table, w32, Np, fc_off, obs_dim):
        self.head, self.timestep, self.table = head, timestep, table
        self._w32, self.Np, self.fc_off, self.obs_dim = w32, Np, fc_off, obs_dim

    def forecast(self, i):
        """float32 [5 Np] view of row i's WeatherForecastObservations block: weather rows k+1 .. k+Np of the step's pre-increment
        timestep k (observations.py:179-182), i.e. rows max(timestep, 1) .. of the timestep after the step."""
        k0 = max(int(self.timestep[i]), 1)
        return self._w32[int(self.table[i]), k0:k0 + self.Np].reshape(-1)

    def full(self, idx=None):
        """Rows assembled in the configured module order (a host gather: use it for the rows you need)."""
        idx = np.arange(self.head.shape[0]) if idx is None else np.atleast_1d(idx)
        out = np.empty((len(idx), self.obs_dim), dtype=np.float32)
        if self.fc_off < 0:
            out[:] = self.head[idx]
            return out
        nf = 5 * self.Np
        out[:, :self.fc_off] = self.head[idx, :self.fc_off]
        out[:, self.fc_off + nf:] = self.head[idx, self.fc_off:]
        for j, i in enumerate(idx):
            out[j, self.fc_off:self.fc_off + nf] = self.forecast(i)
        return out


try:  # pragma: no cover - stable-baselines3 is pinned by the reference (requirements.txt:49) but absent from this image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase  # a real subclass where SB3 exists (isinstance checks)
except Exception:
    _VecEnvBase = object


class GreenLightVecEnv(_VecEnvBase):
    """B TomatoEnv instances advanced in lock-step on one GPU.  See the module docstring.  Subclasses SB3's `VecEnv` when
    stable-baselines3 is importable (every abstract method of SB3 2.6.0's VecEnv is implemented below: reset, step_async,
    step_wait, close, get_attr, set_attr, env_method, env_is_wrapped; plus seed / step / get_images-free render_mode)."""

    metadata = {"render_modes": []}

    def __init__(self, num_envs, reward_function="GreenhouseReward", observation_modules=None, constraints=None,
                 eval_options=None, reward_params=None, base_env_params=None, uncertainty_scale=0.0,
                 n_sub=None, device=0, seed=0, auto_reset=True, env_id_offset=0, weather_tables=None,
                 table_start_days=None, params=None, info_mode=None, role_warps=0, role_lanes=0, precision="fp64",
                 reuse_output_buffers=False, integrator=None, obs_ring=4, host_obs="overlap"):
        if reward_function != "GreenhouseReward":
            raise ValueError("only GreenhouseReward exists in the reference (tomato_env.py:14)")
        mods = list(observation_modules or DEFAULT_OBSERVATION_MODULES)
        unknown = [m for m in mods if m not in OBSERVATION_MODULES]
        if unknown or len(set(mods)) != len(mods):
            raise ValueError(f"observation_modules must be distinct names out of {list(OBSERVATION_MODULES)}; got {mods}")
        bp = dict(DEFAULT_BASE_ENV_PARAMS)
        bp.update(base_env_params or {})
        self.base_env_params = bp
        con = dict(DEFAULT_CONSTRAINTS)
        con.update(constraints or {})
        rp = dict(DEFAULT_REWARD_PARAMS)
        rp.update(reward_params or {})
        self.eval_options = eval_options
        self.uncertainty_scale = float(uncertainty_scale)
        self.num_envs = int(num_envs)
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        # --- derived quantities, base_env.py:65-88
        self.c = 86400
        self.nx, self.nu, self.nd, self.num_params = bp["nx"], bp["nu"], bp["nd"], bp["num_params"]
        self.dt = bp["dt"]
        self.u_min = np.array(bp["u_min"], dtype=np.float32)
        self.u_max = np.array(bp["u_max"], dtype=np.float32)
        self.delta_u_max = np.ones(self.nu, dtype=np.float32) * bp["delta_u_max"]
        self.Np = int(bp["pred_horizon"] * self.c / self.dt)
        self.N = int(bp["season_length"] * self.c / self.dt)
        self.season_length = bp["season_length"]
        self.location, self.data_source = bp["location"], bp["data_source"]
        self.weather_data_dir = bp["weather_data_dir"]
        self.training = bp["training"]
        self.train_years = list(range(bp["start_train_year"], bp["end_train_year"] + 1))
        self.train_days = list(range(bp["start_train_day"], bp["end_train_day"] + 1))
        # integrator: "fixed" = n_sub equal RK4 substeps (default 600, the parity contract); "graded" = RK4 with a refined
        # start of every control interval and a transient-stiffness rule (default n_sub 260; DESIGN.md "Graded integrator")
        integrator = integrator or DEFAULT_INTEGRATOR
        if integrator not in ("fixed", "graded"):
            raise ValueError("integrator must be 'fixed' or 'graded'")
        self.integrator = integrator
        self.n_sub = int(n_sub) if n_sub is not None else (600 if integrator == "fixed" else 260)
        self.observation_modules = mods
        # spaces: tomato_env.py:83-98 / observations.py observation_space() of each module, concatenated in stack order
        sizes = [len(OBSERVATION_MODULES[m][1]) if OBSERVATION_MODULES[m][1] is not None else 5 * self.Np for m in mods]
        self.obs_dim = int(sum(sizes))
        if self.obs_dim < 3:
            raise ValueError("the reward reads obs[0:3] (rewards.py:191-198): the observation stack needs at least 3 entries")
        low = np.concatenate([np.full(n, OBSERVATION_MODULES[m][2][0]) for m, n in zip(mods, sizes)]).astype(np.float32)
        high = np.concatenate([np.full(n, OBSERVATION_MODULES[m][2][1]) for m, n in zip(mods, sizes)]).astype(np.float32)
        self.observation_space = Box(low=low, high=high, dtype=np.float32)
        self.forecast_offset = int(sum(sizes[:mods.index("WeatherForecastObservations")])) if "WeatherForecastObservations" in mods else -1
        self.action_space = Box(low=-1, high=1, shape=(self.nu,), dtype=np.float32)
        self.constraints_low = np.array([con["co2_min"], con["temp_min"], con["rh_min"]])
        self.constraints_high = np.array([con["co2_max"], con["temp_max"], con["rh_max"]])
        self.render_mode = None
        self.reset_infos = [{} for _ in range(self.num_envs)]
        self._seeds = [None for _ in range(self.num_envs)]      # attributes SB3's VecEnv.__init__ would set
        self._options = [{} for _ in range(self.num_envs)]
        self.info_mode = info_mode or ("full" if self.num_envs <= 256 else "minimal")

        # --- parameters (parameters.py) : float32 table widened to float64, as pybind does for evalF
        self.p = np.asarray(params if params is not None else init_default_params(self.num_params), dtype=np.float32)
        # --- weather bank: one table per (year, start_day) the env may be reset to (tomato_env.py:236-260)
        if weather_tables is None:
            years = self.train_years if self.training else list(eval_options["eval_years"])
            days = self.train_days if self.training else list(eval_options["eval_days"])
            loc = self.location if self.training else eval_options["location"]
            src = self.data_source if self.training else eval_options["data_source"]
            tabs, sdays, keys = [], [], []
            for y in years:
                for sd in days:
                    tabs.append(load_weather_data(self.weather_data_dir, loc, src, y, sd, self.season_length,
                                                  self.Np + 1, self.dt, self.nd))
                    sdays.append(float(sd))
                    keys.append((y, sd))
            self.table_keys = keys
            weather_tables = np.stack(tabs)
            table_start_days = np.array(sdays)
        weather_tables = np.ascontiguousarray(weather_tables, dtype=np.float64)
        if weather_tables.ndim == 2:
            weather_tables = weather_tables[None]
        self.weather_tables = weather_tables
        n_tables, rows, _ = weather_tables.shape
        self.table_start_days = np.ascontiguousarray(
            table_start_days if table_start_days is not None else np.zeros(n_tables), dtype=np.float64)

        # --- handle
        self._lib = _lib.load()
        cfg = _lib.GlgConfig()
        self._lib.glg_default_config(C.byref(cfg))
        cfg.num_envs, cfg.device, cfg.dt, cfg.n_sub, cfg.N, cfg.Np = self.num_envs, self.device_index, float(self.dt), \
            self.n_sub, self.N, self.Np
        if precision not in ("fp64", "fp32"):
            raise ValueError("precision must be 'fp64' (parity mode) or 'fp32' (throughput mode)")
        self.precision = precision
        cfg.precision = 0 if precision == "fp64" else 1
        cfg.auto_reset = 1 if auto_reset else 0
        for i in range(self.nu):
            cfg.u_min[i], cfg.u_max[i] = float(self.u_min[i]), float(self.u_max[i])
        cfg.delta_u_max = float(np.float32(bp["delta_u_max"]))
        for i in range(3):
            cfg.con_low[i], cfg.con_high[i] = float(self.constraints_low[i]), float(self.constraints_high[i])
        cfg.elec_price, cfg.heating_price, cfg.co2_price = rp["elec_price"], rp["heating_price"], rp["co2_price"]
        cfg.fruit_price, cfg.dmfm = rp["fruit_price"], rp["dmfm"]
        yearly = rp["fixed_greenhouse_cost"] + rp["fixed_co2_cost"] + rp["fixed_lamp_cost"] * 116 + rp["fixed_screen_cost"]
        cfg.fixed_costs = yearly / 365 / (86400 // self.dt)  # rewards.py:69-70,154
        cfg.uncertainty_scale = self.uncertainty_scale
        cfg.seed = int(seed) & (2**64 - 1)
        cfg.env_id_offset = int(env_id_offset)
        cfg.integrator = 0 if integrator == "fixed" else 1
        cfg.role_lanes = int(role_lanes)  # kernel C envs-per-CTA override (0 = auto)
        for i, m in enumerate(mods):
            cfg.obs_modules[i] = OBSERVATION_MODULES[m][0]
        cfg.role_warps = int(role_warps)  # 0 auto, 1 = one thread per env, 2 / 3 = warp-specialised kernel (latency layout, 1 CTA per SM / throughput layout, 4 CTAs per SM)
        self.reward_params = rp
        self._seed = int(seed)
        self._h = C.c_void_p()
        _lib.check(self._lib.glg_create(C.byref(cfg), C.byref(self._h)), None, "glg_create")
        p64 = np.ascontiguousarray(self.p, dtype=np.float64)
        _lib.check(self._lib.glg_set_params(self._h, p64.ctypes.data), self._h, "glg_set_params")
        _lib.check(self._lib.glg_set_weather(self._h, weather_tables.ctypes.data, n_tables, rows,
                                             self.table_start_days.ctypes.data), self._h, "glg_set_weather")
        assert int(self._lib.glg_obs_dim(self._h)) == self.obs_dim
        B, dev = self.num_envs, self.device
        view = lambda ptr, shape, ts: torch.as_tensor(_DevArray(ptr, shape, ts), device=dev)
        L = self._lib
        self.obs_t = view(L.glg_obs_dev(self._h), (B, self.obs_dim), "<f4")
        self.terminal_obs_t = view(L.glg_terminal_obs_dev(self._h), (B, self.obs_dim), "<f4")
        self.reward_t = view(L.glg_reward_dev(self._h), (B,), "<f8")
        self.done_t = view(L.glg_done_dev(self._h), (B,), "|u1")
        self.info_t = view(L.glg_info_dev(self._h), (_lib.NINFO, B), "<f8")
        self.state_t = view(L.glg_state_dev(self._h), (_lib.NX, B), "<f8")
        self.controls_t = view(L.glg_controls_dev(self._h), (_lib.NU, B), "<f8")
        self.timestep_t = view(L.glg_timestep_dev(self._h), (B,), "<i4")
        self.table_t = view(L.glg_table_dev(self._h), (B,), "<i4")
        self.time_t = view(L.glg_time_dev(self._h), (2, B), "<f8")
        self.stats_t = view(L.glg_stats_dev(self._h), (_lib.NSTATS,), "<f8")
        self._actions = None
        # page-locked result buffers: glg_step_host copies device -> these directly (no staging copy)
        self._pin = [torch.empty((B, self.obs_dim), dtype=torch.float32).pin_memory(), torch.empty(B, dtype=torch.float64).pin_memory(),
                     torch.empty(B, dtype=torch.uint8).pin_memory(), torch.empty((B, self.nu), dtype=torch.float32).pin_memory()]
        self._obs_host, self._rew_host, self._done_host, self._act_host = (t.numpy() for t in self._pin)
        # addresses of the fixed host buffers (`ndarray.ctypes.data` costs ~2 us per access: 9 us of a 0.86 ms step otherwise)
        self._rew_ptr, self._done_ptr, self._act_ptr = (a.ctypes.data for a in (self._rew_host, self._done_host, self._act_host))
        # Observation arrays returned by `step()` (numpy path) -- explicit ownership, no reference counting:
        #   obs_ring = n >= 2 (default 4): the arrays ARE page-locked buffers of a ring of n, handed out round-robin; the array
        #       returned by step k stays untouched until step k + n (no host copy: 0.29 ms per step at B = 4096).  Safe for SB3's
        #       collect loop (it copies `new_obs` into its rollout buffer before the next step) and for any consumer that is done
        #       with an observation within n - 1 further steps -- including asynchronous ones (non_blocking H2D from this pinned
        #       memory), which reference counting cannot see.
        #   obs_ring = 0: a fresh pageable copy every step (the reference's semantics, for callers that keep observations).
        #   reuse_output_buffers=True is the old name of obs_ring = 2.
        self.reuse_output_buffers = bool(reuse_output_buffers)
        self.obs_ring = 2 if self.reuse_output_buffers else int(obs_ring)
        if self.obs_ring == 1 or self.obs_ring < 0:
            raise ValueError("obs_ring must be 0 (copy every step) or >= 2")
        # host_obs: how step() (numpy path) gets the observation rows into host memory (glg_set_host_obs_mode): "overlap" (default)
        # = the forecast block of every row is written by the host from its own copy of the weather bank while the kernel runs
        # and only the other columns cross PCIe; "copy" = one device->host copy of the whole array.  Same array either way.
        if host_obs not in ("overlap", "copy"):
            raise ValueError("host_obs must be 'overlap' or 'copy'")
        self.host_obs = host_obs
        _lib.check(self._lib.glg_set_host_obs_mode(self._h, 0 if host_obs == "overlap" else 1), self._h, "glg_set_host_obs_mode")
        self._split = None
        self._ring = self._ring_np = None  # page-locked, allocated by the first numpy step (the tensor path never needs them)
        self._ring_pos = 0

    # ------------------------------------------------------------------ tensor fast path
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def reset_tensor(self, mask=None, table_ids=None):
        m = 0 if mask is None else mask.to(torch.uint8).contiguous().data_ptr()
        t = 0 if table_ids is None else table_ids.to(torch.int32).contiguous().data_ptr()
        _lib.check(self._lib.glg_reset(self._h, m, t, self._stream()), self._h, "glg_reset")
        return self.obs_t

    def step_tensor(self, actions, noise=None):
        """actions: CUDA float32 [B,6].  Returns (obs [B,obs_dim] f32, reward [B] f64, done [B] u8) device views
        that are overwritten by the next step."""
        a = actions.to(device=self.device, dtype=torch.float32).contiguous()
        n = 0 if noise is None else noise.to(device=self.device, dtype=torch.float64).contiguous().data_ptr()
        _lib.check(self._lib.glg_step(self._h, a.data_ptr(), n, self._stream()), self._h, "glg_step")
        return self.obs_t, self.reward_t, self.done_t

    def step_raw_control_tensor(self, controls, noise=None):
        """TomatoEnv.step_raw_control (tomato_env.py:148-173) for the batch: controls CUDA float64 [B,6]."""
        u = controls.to(device=self.device, dtype=torch.float64).contiguous()
        n = 0 if noise is None else noise.to(device=self.device, dtype=torch.float64).contiguous().data_ptr()
        _lib.check(self._lib.glg_step_raw_control(self._h, u.data_ptr(), n, self._stream()), self._h, "glg_step_raw_control")
        return self.obs_t, self.reward_t, self.done_t

    def set_rule_controller(self, controller=None):
        """Settings of the on-device rule-based controller: a `glgym.controller.RuleBasedController`, a dict of
        rule_based.yml keys, or None for the shipped values."""
        from .controller import RuleBasedController
        if controller is None:
            vec = None
        else:
            c = controller if isinstance(controller, RuleBasedController) else RuleBasedController(**controller)
            vec = np.ascontiguousarray(c.settings_vector())
        _lib.check(self._lib.glg_set_rule_controller(self._h, None if vec is None else vec.ctypes.data), self._h,
                   "glg_set_rule_controller")

    def step_rule_based_tensor(self, noise=None):
        """One step with RuleBasedController.predict (baseline.py:68-227) evaluated on the device from each env's own
        state, weather row and clock, then applied like step_raw_control (evaluate_baseline.py:21-23) -- no host round trip."""
        n = 0 if noise is None else noise.to(device=self.device, dtype=torch.float64).contiguous().data_ptr()
        _lib.check(self._lib.glg_step_rule_based(self._h, n, self._stream()), self._h, "glg_step_rule_based")
        return self.obs_t, self.reward_t, self.done_t

    def rule_controls_tensor(self, settings=None):
        """RuleBasedController.predict for every env on its current state, weather row and clock: the controls
        `step_rule_based_tensor` would apply.  settings: CUDA float64 [B, 29] in rule_based.yml order, one row per env, or None
        for the env's own settings (`set_rule_controller`).  Returns a float64 [B, 6] view of a buffer the env owns, overwritten
        by the next call; `step_raw_control_tensor` with it steps exactly as `step_rule_based_tensor` would."""
        s = 0
        if settings is not None:
            if tuple(settings.shape) != (self.num_envs, 29):
                raise ValueError(f"settings must have shape ({self.num_envs}, 29); got {tuple(settings.shape)}")
            settings = settings.to(device=self.device, dtype=torch.float64).contiguous()
            s = settings.data_ptr()
        if getattr(self, "_rule_u", None) is None:
            self._rule_u = torch.empty((self.num_envs, self.nu), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.glg_rule_controls(self._h, s, self._rule_u.data_ptr(), self._stream()), self._h, "glg_rule_controls")
        return self._rule_u

    def linearize_tensor(self, controls=None):
        """Linearise the step `step_raw_control_tensor(controls)` would take from every env's current state, without taking it:
        returns (x_next [B,28], A [B,28,28], Bu [B,28,6]) with A = dx_next/dx and Bu = dx_next/du, exact derivatives of the
        integration on its executed grid.  controls: CUDA float64 [B, 6], or None for the envs' current u.  Always fp64 and the
        nominal model (also for precision=1 and under parametric uncertainty); the env's state is not touched."""
        c = 0
        if controls is not None:
            if tuple(controls.shape) != (self.num_envs, self.nu):
                raise ValueError(f"controls must have shape ({self.num_envs}, {self.nu}); got {tuple(controls.shape)}")
            controls = controls.to(device=self.device, dtype=torch.float64).contiguous()
            c = controls.data_ptr()
        B = self.num_envs
        xn = torch.empty((B, 28), dtype=torch.float64, device=self.device)
        A = torch.empty((B, 28, 28), dtype=torch.float64, device=self.device)
        Bu = torch.empty((B, 28, self.nu), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.glg_linearize(self._h, c, xn.data_ptr(), A.data_ptr(), Bu.data_ptr(), self._stream()), self._h,
                   "glg_linearize")
        return xn, A, Bu

    def step_rule_based(self):
        self.step_rule_based_tensor()
        torch.cuda.synchronize(self.device)
        dones = self.done_t.cpu().numpy().astype(bool)
        return self.obs_t.cpu().numpy(), self.reward_t.cpu().numpy(), dones, self._make_infos(dones)

    # ------------------------------------------------------------------ SB3 VecEnv protocol (numpy)
    def reset(self):
        self.reset_tensor()
        torch.cuda.synchronize(self.device)
        self.reset_infos = [{} for _ in range(self.num_envs)]
        return self.obs_t.cpu().numpy()

    def step_async(self, actions):
        np.copyto(self._act_host, np.asarray(actions, dtype=np.float32).reshape(self.num_envs, self.nu))
        self._actions = self._act_host

    def step_wait(self):
        if self._ring_np is None:
            B = self.num_envs
            self._ring = [self._pin[0]] + [torch.empty((B, self.obs_dim), dtype=torch.float32).pin_memory() for _ in range(max(self.obs_ring - 1, 0))]
            self._ring_np = [t.numpy() for t in self._ring]
            self._ring_ptr = [a.ctypes.data for a in self._ring_np]
        n = len(self._ring_np)
        obs_buf, obs_ptr = self._ring_np[self._ring_pos], self._ring_ptr[self._ring_pos]
        self._ring_pos = (self._ring_pos + 1) % n
        # glg_step_host works on the handle's own stream: order it behind whatever the caller enqueued on torch's current
        # stream (reset_tensor / step_tensor / episode_stats(clear=True) followed by step()) -- an event wait, no host sync
        self._lib.glg_host_path_after(self._h, _raw_stream(self.device_index))
        _lib.check(self._lib.glg_step_host(self._h, self._act_ptr, obs_ptr, self._rew_ptr, self._done_ptr), self._h, "glg_step_host")
        dones = self._done_host.astype(bool)
        obs = obs_buf.copy() if self.obs_ring == 0 else obs_buf
        # rewards: float64 on the device (the reference returns a Python float); the VecEnv protocol carries float32
        return obs, self._rew_host.astype(np.float32), dones, self._make_infos(dones)

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    # ------------------------------------------------------------------ split observations (opt-in host path)
    def step_split(self, actions):
        """`step()` with the observation in SPLIT form: returns (SplitObs, rewards, dones, infos).  240 of the default row's 263
        floats are the WeatherForecastObservations block -- raw weather rows that depend on (table, timestep) only and that the
        host already holds -- so only the other columns cross PCIe (0.43 MB instead of 4.35 MB per step at B = 4096) and the
        forecast is read from the host's float32 copy of the weather bank on demand:
            so.head      float32 [B, obs_dim - 5 Np]   every column but the forecast block (page-locked ring buffer)
            so.forecast(i) -> float32 [5 Np] view      row i's forecast block (zero copy)
            so.full([idx]) -> float32 [n, obs_dim]     rows assembled in the configured module order
        Terminal observations of done envs are delivered through infos as in step()."""
        if self._split is None:
            B, nf = self.num_envs, (5 * self.Np if self.forecast_offset >= 0 else 0)
            n = max(self.obs_ring, 2)
            self._split = dict(head=[torch.empty((B, self.obs_dim - nf), dtype=torch.float32).pin_memory() for _ in range(n)],
                               k=[torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(n)],
                               tb=[torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(n)], pos=0,
                               w32=np.ascontiguousarray(self.weather_tables[:, :, :5], dtype=np.float32))
        sp = self._split
        i = sp["pos"]
        sp["pos"] = (i + 1) % len(sp["head"])
        np.copyto(self._act_host, np.asarray(actions, dtype=np.float32).reshape(self.num_envs, self.nu))
        self._lib.glg_host_path_after(self._h, _raw_stream(self.device_index))
        head, k, tb = sp["head"][i].numpy(), sp["k"][i].numpy(), sp["tb"][i].numpy()
        _lib.check(self._lib.glg_step_host_split(self._h, self._act_host.ctypes.data, head.ctypes.data, k.ctypes.data, tb.ctypes.data,
                                                 self._rew_host.ctypes.data, self._done_host.ctypes.data), self._h, "glg_step_host_split")
        dones = self._done_host.astype(bool)
        return (SplitObs(head, k, tb, sp["w32"], self.Np, self.forecast_offset, self.obs_dim), self._rew_host.astype(np.float32), dones,
                self._make_infos(dones))

    def step_raw_control(self, controls):
        u = torch.as_tensor(np.asarray(controls, dtype=np.float64).reshape(self.num_envs, self.nu), device=self.device)
        self.step_raw_control_tensor(u)
        torch.cuda.synchronize(self.device)
        dones = self.done_t.cpu().numpy().astype(bool)
        return self.obs_t.cpu().numpy(), self.reward_t.cpu().numpy(), dones, self._make_infos(dones)

    def _make_infos(self, dones):
        if self.info_mode == "full":
            info = self.info_t.cpu().numpy()
            ctrl = self.controls_t.cpu().numpy()
            infos = [dict(zip(INFO_KEYS, info[:, i].tolist()), controls=ctrl[:, i].copy(), **{"TimeLimit.truncated": False})
                     for i in range(self.num_envs)]
        else:
            # "minimal": envs that are not done share ONE read-only empty mapping (building 4096 dicts costs 0.1 ms per step,
            # 65 536 of them 1.6 ms).  It supports everything SB3's wrappers do with an info (`.get`, `in`, `.copy()`);
            # assigning into it raises TypeError instead of silently leaking into the other envs.
            infos = [_EMPTY_INFO] * self.num_envs
        idx = np.nonzero(dones)[0]
        if idx.size:
            term = self.terminal_obs_t[torch.as_tensor(idx, device=self.device)].cpu().numpy()
            for j, i in enumerate(idx):
                info = dict(infos[i])
                info["terminal_observation"] = term[j]
                info["TimeLimit.truncated"] = False
                infos[i] = info
        return infos

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.glg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _indices(self, indices):
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return indices

    def get_attr(self, attr_name, indices=None):
        idx = list(self._indices(indices))
        if attr_name == "u":
            u = self.controls_t.cpu().numpy()
            return [u[:, i].copy() for i in idx]
        if attr_name == "x":
            x = self.state_t.cpu().numpy()
            return [x[:, i].copy() for i in idx]
        if attr_name == "timestep":
            k = self.timestep_t.cpu().numpy()
            return [int(k[i]) for i in idx]
        if attr_name in ("start_day", "growth_year"):
            tb = self.table_t.cpu().numpy()
            keys = getattr(self, "table_keys", None)
            if attr_name == "start_day":
                return [float(self.table_start_days[tb[i]]) for i in idx]
            return [keys[tb[i]][0] if keys else None for i in idx]
        return [getattr(self, attr_name) for _ in idx]

    def set_attr(self, attr_name, value, indices=None):
        """Per-env attributes that live on the device ("u", "x", "timestep") are written for `indices`; anything else is an
        attribute of the batch as a whole and only accepts indices=None / all envs."""
        idx = list(self._indices(indices))
        if attr_name in ("u", "x", "timestep"):
            x, u, k = self.get_state()
            arr = {"u": u, "x": x, "timestep": k}[attr_name]
            arr[idx] = value
            self.set_state(**{attr_name: arr})
            return
        if len(idx) != self.num_envs:
            raise ValueError(f"attribute {attr_name!r} is shared by all envs of the batch; set it with indices=None")
        setattr(self, attr_name, value)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        idx = list(self._indices(indices))
        if method_name == "get_obs_names":
            return [obs_names(self.Np, self.observation_modules) for _ in idx]
        if method_name == "set_seed":
            # RNG streams are keyed by (seed, global env id): one key for the batch.  SB3 scripts call set_seed(seed + rank) per
            # env; the first env's argument re-keys the handle, the per-env offset is what the global env id already provides.
            if args:
                self.reseed(int(args[0]))
            return [None for _ in idx]
        if method_name in ("_reset_eval_idx", "increase_eval_idx"):
            self.eval_idx = 0 if method_name == "_reset_eval_idx" else getattr(self, "eval_idx", 0) + 1
            return [None for _ in idx]
        raise AttributeError(f"env_method {method_name!r} is not provided by the batched env")

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False for _ in self._indices(indices)]

    def reseed(self, seed):
        """New key for the handle's Philox streams (parametric noise, reset-table choice, StateObservations); takes effect with
        the next launch.  base_env.py:166-170 `set_seed`."""
        self._seed = int(seed)
        _lib.check(self._lib.glg_set_seed(self._h, C.c_uint64(self._seed & (2**64 - 1))), self._h, "glg_set_seed")

    def set_options(self, options=None):  # SB3 VecEnv API; TomatoEnv.reset takes no options
        self._options = [{} for _ in range(self.num_envs)]

    def seed(self, seed=None):
        """SB3 VecEnv.seed: env i is seeded with seed + i.  Here one key re-keys the handle's Philox streams and the per-env offset
        is the global env id those streams are keyed by anyway."""
        if seed is not None:
            self.reseed(int(seed))
        self._seeds = [None if seed is None else seed + i for i in range(self.num_envs)]
        return list(self._seeds)

    def get_obs_names(self):
        return obs_names(self.Np, self.observation_modules)

    # ------------------------------------------------------------------ helpers
    def set_state(self, x=None, u=None, timestep=None):
        """Teacher forcing: x [B,28], u [B,6] float64, timestep [B] int32 (host arrays).  Setting the timestep also moves the
        env clock to it (day of year / hour of day as after `timestep` steps from the env's table start day); for a complete
        checkpoint / restore use state_dict() / load_state_dict()."""
        keep = [None if a is None else np.ascontiguousarray(a, dtype=dt) for a, dt in
                ((x, np.float64), (u, np.float64), (timestep, np.int32))]
        _lib.check(self._lib.glg_set_state(self._h, *[0 if a is None else a.ctypes.data for a in keep]), self._h, "glg_set_state")

    def get_state(self):
        x = np.empty((self.num_envs, _lib.NX))
        u = np.empty((self.num_envs, _lib.NU))
        k = np.empty(self.num_envs, dtype=np.int32)
        _lib.check(self._lib.glg_get_state(self._h, x.ctypes.data, u.ctypes.data, k.ctypes.data), self._h, "glg_get_state")
        return x, u, k

    _STATE_FIELDS = (("x", np.float64, _lib.NX), ("u", np.float64, _lib.NU), ("timestep", np.int32, 0), ("table", np.int32, 0),
                     ("time", np.float64, 2), ("step_ctr", np.uint32, 0), ("ep_return", np.float64, 0), ("ep_len", np.int32, 0),
                     ("ep_info", np.float64, _lib.NINFO))

    def state_dict(self):
        """Everything a step reads besides the parameter table and the weather bank: state, controls, timestep, weather table,
        clock, Philox stream position and the episode accumulators (host arrays)."""
        B = self.num_envs
        out = {n: np.empty((B, w) if w else B, dtype=dt) for n, dt, w in self._STATE_FIELDS}
        st = _lib.GlgEnvState(**{n: out[n].ctypes.data for n, _, _ in self._STATE_FIELDS})
        _lib.check(self._lib.glg_get_state_ex(self._h, C.byref(st)), self._h, "glg_get_state_ex")
        return out

    def load_state_dict(self, state):
        """Restores (a subset of) state_dict(); table ids and timesteps are range-checked by the library."""
        B = self.num_envs
        keep = {}
        for n, dt, w in self._STATE_FIELDS:
            if n in state and state[n] is not None:
                keep[n] = np.ascontiguousarray(state[n], dtype=dt).reshape((B, w) if w else B)
        st = _lib.GlgEnvState(**{n: a.ctypes.data for n, a in keep.items()})
        _lib.check(self._lib.glg_set_state_ex(self._h, C.byref(st)), self._h, "glg_set_state_ex")

    def launch_count(self):
        return int(self._lib.glg_launch_count(self._h))

    def init_stats_allreduce(self):
        """Creates the handle's NCCL communicator over torch.distributed's ranks (the 128-byte NCCL id travels in a
        broadcast); afterwards allreduce_stats() sums the episode statistics of all ranks' handles on the device."""
        import torch.distributed as dist
        ident = torch.zeros(128, dtype=torch.uint8)
        rank, world = (dist.get_rank(), dist.get_world_size()) if dist.is_initialized() else (0, 1)
        if rank == 0:
            buf = np.zeros(128, dtype=np.uint8)
            _lib.check(self._lib.glg_nccl_unique_id(buf.ctypes.data), None, "glg_nccl_unique_id")
            ident = torch.from_numpy(buf)
        if world > 1:
            t = ident.to(self.device) if dist.get_backend() == "nccl" else ident
            dist.broadcast(t, src=0)
            ident = t.cpu()
        buf = np.ascontiguousarray(ident.numpy())
        # NCCL prints its version banner to stdout when a process creates its first communicator: keep stdout clean for callers
        # that emit machine-readable output (bench.py's one JSON line) by pointing fd 1 at stderr for the duration of the call
        import os
        import sys
        sys.stdout.flush()
        saved = os.dup(1)
        try:
            os.dup2(2, 1)
            rc = self._lib.glg_nccl_init(self._h, buf.ctypes.data, rank, world)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        _lib.check(rc, self._h, "glg_nccl_init")

    def allreduce_stats(self):
        """In-place sum over ranks of the 16-entry statistics vector (ncclAllReduce on torch's current stream); stats_t then
        holds the global sums on every rank."""
        _lib.check(self._lib.glg_allreduce_stats(self._h, self._stream()), self._h, "glg_allreduce_stats")
        return self.stats_t

    def episode_stats(self, clear=False):
        s = self.stats_t.cpu().numpy().copy()
        if clear:
            _lib.check(self._lib.glg_clear_stats(self._h, self._stream()), self._h, "glg_clear_stats")
        out = {"episodes": s[0], "return_sum": s[1], "length_sum": s[2], "nonfinite": s[14]}
        out.update({k: s[3 + i] for i, k in enumerate(INFO_KEYS)})
        return out
