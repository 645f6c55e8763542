"""wildfire_control_python_b200 -- B200-native batched forest-fire environment step.

Drop-in for the hot path of dashdeckers/Wildfire-Control-Python (Simulation/forest_fire.py +
Simulation/environment.py): ``BatchedForestFire`` steps thousands of environments per CUDA
launch; ``ForestFire`` is the single-env facade with the reference's attribute surface.
The compute lives in ``libwildfire_b200.so`` (csrc/, sm_100a) behind include/wildfire.h.
"""
from . import _lib
from ._lib import obs_bits_words
from .constants import METADATA, grass, layer, make_metadata, types

__all__ = ["BatchedForestFire", "ForestFire", "METADATA", "grass", "layer", "types", "make_metadata", "build",
           "DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH", "learn_population", "obs_bits_words", "unpack_obs", "pack_obs",
           "FinalStates"]


def build(force: bool = False, verbose: bool = False) -> str:
    return _lib.build(force=force, verbose=verbose)


def __getattr__(name):  # torch is imported lazily so that `import wildfire_control_python_b200` stays cheap
    if name == "BatchedForestFire":
        from .batched import BatchedForestFire
        return BatchedForestFire
    if name in ("unpack_obs", "pack_obs", "FinalStates"):
        from . import batched
        return getattr(batched, name)
    if name == "ForestFire":
        from .compat import ForestFire
        return ForestFire
    if name in ("DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH", "learn_population"):
        from . import agents
        return getattr(agents, name)
    raise AttributeError(name)
