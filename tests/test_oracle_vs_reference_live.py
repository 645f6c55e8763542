"""Live differential test: the C oracle against the UNMODIFIED Python reference, step by step.

Runs only where the reference is reachable (oracle/ref_harness.py: the tree named by WF_REFERENCE_ROOT, or
the snapshot `make -C oracle ref REF=<tree>` leaves in oracle/_ref/); elsewhere the committed golden
trajectories of tests/golden/ stand in (tests/test_oracle_golden.py).  It is the pytest face of
`python -m oracle.validate_oracle` (69 000 steps over 23 scenarios, run by hand): a bounded
number of steps of every scenario, every plane / scalar / observation / reward / done compared, and
for the `walk_*` scenarios the reference's own `DQN.choose_randomwalk_action` against the oracle's
restatement, action by action.
"""
import pytest

from oracle import ref_harness

pytestmark = pytest.mark.skipif(not ref_harness.reference_available(),
                                reason="the original project is not reachable (WF_REFERENCE_ROOT or oracle/_ref)")


def _scenarios():
    try:
        from oracle.validate_oracle import SCENARIOS
        return SCENARIOS
    except Exception:  # the harness imports the reference at module import time
        return []


@pytest.mark.parametrize("sc", _scenarios(), ids=lambda s: s["name"])
def test_oracle_equals_python_reference(sc):
    from oracle.validate_oracle import run
    st = run(sc, 350)
    assert st["steps"] == 350 and st["maxerr"] <= 1e-12
    if sc.get("policy", "").startswith(("ring", "walk")):
        assert st["contained"] >= 1  # the scripted / heuristic walks do contain the fire


def _random_scenarios(n=12, seed=2026):
    try:
        import numpy as np

        from oracle.validate_oracle import random_scenario
        rng = np.random.default_rng(seed)
        return [random_scenario(rng, i) for i in range(n)]
    except Exception:
        return []


@pytest.mark.parametrize("sc", _random_scenarios(), ids=lambda s: s["name"])
def test_oracle_equals_python_reference_random_configs(sc):
    """Randomised configurations (size, wind, rivers, dig toggle, a_speed, extra ignitions, policy): the pytest face of
    `python -m oracle.validate_oracle --random N` (DESIGN.md section 4 records the last long run)."""
    from oracle.validate_oracle import run
    st = run(sc, 250)
    assert st["steps"] == 250 and st["maxerr"] <= 1e-12
