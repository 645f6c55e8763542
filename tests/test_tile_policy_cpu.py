"""learn_batched on grids larger than 32x32 without a GPU: it is no longer refused for the grid, and it has no CPU fallback."""
import pytest
import torch

from wildfire_control_python_b200 import _lib
from wildfire_control_python_b200 import agents as A
from wildfire_control_python_b200.compat import get_name
from wildfire_control_python_b200.constants import make_metadata


class _World:
    DEPTH = 3
    agents = []

    def __init__(self, W, H):
        self.WIDTH, self.HEIGHT = W, H


class _Sim:
    def __init__(self, W, H, **kw):
        self.METADATA = make_metadata(width=W, height=H, **kw)
        self.n_actions, self.DEBUG, self.get_name = int(self.METADATA["n_actions"]), 1, get_name
        self.W = _World(W, H)


@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA"])
def test_learn_batched_on_a_tile_grid_has_no_cpu_fallback(name):
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the agent would live on it")
    ag = getattr(A, name)(_Sim(40, 40), verbose=False, device="cpu")
    with pytest.raises(_lib.WildfireError, match="no CPU fallback"):
        ag.learn_batched(10, n_envs=64)
