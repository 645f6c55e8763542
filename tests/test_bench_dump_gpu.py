"""bench.py's measured path on the GPU: exactly warm-up + --steps steps run, the outputs kept for --dump-outputs are those of
the last timed step, and two runs with the same arguments keep identical outputs (what lets two builds of the project be
compared output for output)."""
import numpy as np
import pytest

import bench


@pytest.mark.gpu
def test_c2_outputs_are_the_last_timed_step():
    from oracle import wf_oracle as wo
    D = bench.Dist(1)
    K, Wm = 20, 5
    res = bench.measure(D, "c2", K, Wm, 0, False, False, 16 << 20)
    N = res["N"]
    steps = res["warmup"] + K
    assert res["warmup"] == 256 and res["launches"] == 1 and res["stats"]["env_steps"] == N * steps
    out = res["outputs"]
    assert np.array_equal(out["obs_env_index"], np.arange(N)) and out["obs"].shape == (N, 14, 14, 3)
    for i in range(0, N, 512):  # the C oracle, stepped the same number of times from the same seed
        e = wo.OracleEnv(bench.oracle_cfg(bench.WORKLOADS["c2"]["meta"]), env_id=i)
        e.reset()
        for _ in range(steps):
            o, r, d, _ = e.step(e.random_action())
            if d:
                o = e.reset()
        assert out["reward"][i] == r and bool(out["done"][i]) == d and np.array_equal(out["obs"][i], o), i
    again = bench.measure(D, "c2", K, Wm, 0, False, False, 16 << 20)["outputs"]
    assert all(np.array_equal(out[k], again[k]) for k in out)


@pytest.mark.gpu
def test_c3_outputs_repeat():
    D = bench.Dist(1)
    one = bench.measure_policy(D, "c3", 20, 5, 4 << 20)["outputs"]
    two = bench.measure_policy(D, "c3", 20, 5, 4 << 20)["outputs"]
    assert len(one["obs_env_index"]) < 8192 and one["obs"].dtype == np.float32
    assert all(np.array_equal(one[k], two[k]) for k in one)
