"""glgym -- B200-native batched GreenLight env-step path (drop-in for GreenLight-Gym2's TomatoEnv step path)."""
from .params import init_default_params  # noqa: F401
from .weather import init_state, load_weather_data  # noqa: F401


def __getattr__(name):  # lazy: importing the package must not require torch/CUDA
    if name == "GreenLightVecEnv":
        from .vec_env import GreenLightVecEnv
        return GreenLightVecEnv
    if name == "TomatoEnv":
        from .tomato_env import TomatoEnv
        return TomatoEnv
    if name == "DeviceReplayBuffer":
        from .replay import DeviceReplayBuffer
        return DeviceReplayBuffer
    if name == "DevicePlanner":
        from .planning import DevicePlanner
        return DevicePlanner
    if name == "GreenLight":
        from .model import GreenLight
        return GreenLight
    raise AttributeError(name)
