"""Rule-based greenhouse climate controller, vectorised over envs (host side, numpy).

Same contract as the reference's `RuleBasedController.predict(x, d, env) -> u[6]`
(gl_gym/environments/baseline.py:68-227, settings gl_gym/configs/agents/rule_based.yml), but for a batch:
`predict(x[B,28], d[B,10], hour_of_day[B], day_of_year[B]) -> u[B,6]`; used with `step_raw_control`
(experiments/evaluate_baseline.py:12-37).  The device-side version (SURVEY.md 8f-1) is csrc/glg_controller.h: `predict_device` here,
`GreenLightVecEnv.step_rule_based*` for the fused controller-in-the-loop step.
"""
import numpy as np

from .weather import co2_dens_to_ppm, sat_vp

DEFAULT_SETTINGS = dict(  # configs/agents/rule_based.yml
    lamps_on=0, lamps_off=18, lamps_day_start=-1, lamps_day_stop=366, lamps_off_sun=400, lamp_rad_sum_limit=10,
    temp_setpoint_day=19.5, temp_setpoint_night=16.5, heat_correction=0, heat_deadzone=5, co2_day=800, vent_heat_Pband=4,
    rh_max=85, mech_dehumid_Pband=2, vent_rh_Pband=5, t_vent_off=1, vent_cold_Pband=-1, thScrSpDay=5, thScrSpNight=10,
    thScrPband=-1, thScrDeadZone=4, thScrRh=-2, thScrRhPband=2, lampExtraHeat=2, blScrExtraRh=100, rhMax=85, tHeatBand=-1,
    co2Band=-100, useBlScr=1,
)
SETTING_NAMES = tuple(DEFAULT_SETTINGS)  # the 29 keys in rule_based.yml order: the columns of a settings vector


def proportional_control(process_var, set_pt, p_band, min_val, max_val):
    """Sigmoid proportional band (baseline.py:226-227)."""
    return min_val + (max_val - min_val) * (1 / (1 + np.exp(-2 / p_band * np.log(100) * (process_var - set_pt - p_band / 2))))


class RuleBasedController:
    def __init__(self, **settings):
        cfg = dict(DEFAULT_SETTINGS)
        cfg.update(settings)
        self.__dict__.update(cfg)

    @classmethod
    def from_vector(cls, v):
        """The controller of a settings vector: 29 numbers in the order of SETTING_NAMES (the inverse of settings_vector)."""
        v = np.asarray(v, dtype=np.float64).reshape(-1)
        if v.shape != (len(SETTING_NAMES),):
            raise ValueError(f"a settings vector has {len(SETTING_NAMES)} entries; got {v.shape[0]}")
        return cls(**{k: float(x) for k, x in zip(SETTING_NAMES, v)})

    def settings_vector(self):
        """float64[29] in the order of rule_based.yml -- what `glg_set_rule_controller` / `glg_rule_control_batch` take."""
        return np.array([float(getattr(self, k)) for k in DEFAULT_SETTINGS], dtype=np.float64)

    def predict_device(self, x, d, hour_of_day, day_of_year, device=0):
        """Same as `predict`, evaluated by the CUDA controller (glg_rule_control_batch); inputs/outputs are torch CUDA
        or numpy arrays [n,28], [n,10], [n], [n] -> [n,6] (torch, float64, on `device`)."""
        import torch
        from . import _lib
        dev = torch.device("cuda", device)
        t = lambda a, shape: torch.as_tensor(a, dtype=torch.float64, device=dev).reshape(shape).contiguous()
        x = t(x, (-1, 28))
        n = x.shape[0]
        d, hod, doy = t(d, (n, 10)), t(hour_of_day, (n,)), t(day_of_year, (n,))
        u = torch.empty((n, 6), dtype=torch.float64, device=dev)
        s = np.ascontiguousarray(self.settings_vector())
        _lib.check(_lib.load().glg_rule_control_batch(s.ctypes.data, x.data_ptr(), d.data_ptr(), hod.data_ptr(), doy.data_ptr(),
                                                      u.data_ptr(), n, device, torch.cuda.current_stream(dev).cuda_stream),
                   None, "glg_rule_control_batch")
        return u

    def _window(self, lo, hi, v):
        """1 inside the (possibly wrapping) interval (lo, hi), else 0 (baseline.py:76-86)."""
        inside = (lo < v) & (v < hi)
        wrap = (lo < v) | (v < hi)
        return np.where(lo <= hi, inside, wrap).astype(np.float64)

    def predict(self, x, d, hour_of_day, day_of_year):
        x, d = np.atleast_2d(np.asarray(x, dtype=np.float64)), np.atleast_2d(np.asarray(d, dtype=np.float64))
        hod = np.broadcast_to(np.asarray(hour_of_day, dtype=np.float64), x.shape[:1])
        doy = np.broadcast_to(np.asarray(day_of_year, dtype=np.float64), x.shape[:1])
        pc = proportional_control
        lamp_tod = self._window(self.lamps_on, self.lamps_off, hod)
        lamp_doy = self._window(self.lamps_day_start, self.lamps_day_stop, doy)
        lamp_no_cons = (d[:, 0] < self.lamps_off_sun) * (d[:, 7] < self.lamp_rad_sum_limit) * lamp_tod * lamp_doy
        sw_on = np.clip(hod - self.lamps_on + 1, 0, 1)
        sw_off = np.clip(self.lamps_off - hod + 1, 0, 1)
        both = (self.lamps_on != self.lamps_off) * (np.minimum(sw_on, sw_off) if self.lamps_on < self.lamps_off
                                                    else np.maximum(sw_on, sw_off))
        smooth_lamp = both * (d[:, 7] < self.lamp_rad_sum_limit) * lamp_doy
        is_day_inside = np.maximum(smooth_lamp, d[:, 8])
        heat_sp = is_day_inside * self.temp_setpoint_day + (1 - is_day_inside) * self.temp_setpoint_night \
            + self.heat_correction * lamp_no_cons
        heat_max = heat_sp + self.heat_deadzone
        co2_sp = is_day_inside * self.co2_day
        co2_ppm = co2_dens_to_ppm(x[:, 2], 1e-6 * x[:, 0])
        vent_heat = pc(x[:, 2], heat_max, self.vent_heat_Pband, 0, 1)
        rh_in = 100 * x[:, 15] / sat_vp(x[:, 2])
        vent_rh = pc(rh_in, self.rh_max + 0 * self.mech_dehumid_Pband, self.vent_rh_Pband, 0, 1)
        vent_cold = pc(x[:, 2], heat_sp - self.t_vent_off, self.vent_cold_Pband, 1, 0)
        th_sp = d[:, 8] * self.thScrSpDay + (1 - d[:, 8]) * self.thScrSpNight
        th_cold = pc(d[:, 1], th_sp, self.thScrPband, 0, 1)
        th_heat = pc(x[:, 2], heat_sp + self.thScrDeadZone, -self.thScrPband, 1, 0)
        th_rh = np.maximum(pc(rh_in, self.rhMax + self.thScrRh, self.thScrRhPband, 1, 0), 1 - vent_cold)
        lamp_on = lamp_no_cons * pc(x[:, 2], heat_max + self.lampExtraHeat, -0.5, 0, 1) * (d[:, 9] + (1 - d[:, 9])) * \
            np.maximum(pc(rh_in, self.rhMax + self.blScrExtraRh, -0.5, 0, 1), 1 - vent_cold)
        u = np.zeros((x.shape[0], 6))
        u[:, 0] = pc(x[:, 2], heat_sp, self.tHeatBand, 0, 1)
        with np.errstate(divide="ignore", over="ignore"):
            u[:, 1] = pc(co2_ppm, co2_sp, self.co2Band, 0, 1)
        u[:, 2] = np.minimum(th_cold, np.maximum(th_heat, th_rh))
        u[:, 3] = np.minimum(vent_cold, np.maximum(vent_heat, vent_rh))
        u[:, 4] = lamp_on
        u[:, 5] = self.useBlScr * (1 - d[:, 9]) * lamp_on
        return u
