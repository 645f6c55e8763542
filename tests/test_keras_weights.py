"""Next-row N2 (SURVEY.md 8(f)): the reference's trained networks (Keras HDF5 ``Models/<name>``) are read
without h5py, and -- the strongest end-to-end parity statement this repo has -- a policy the REFERENCE
trained on ITS environment earns, on OUR environment, the return the reference's own training log
records for it (Logs/<name>: last 2500 episodes, the quantity the thesis tabulates).  That pins the
dynamics, the reward, the start distribution and the observation layout (Keras ``Flatten`` order) at once.

Fixtures: tests/golden/keras/ (two weight files + kat.json), made by oracle/gen_keras_fixture.py.
"""
import glob
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import ref_harness
from wildfire_control_python_b200.keras_h5 import H5Error, canonical_dense_names, read_h5_datasets, read_keras_weights

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "keras")
KAT = json.load(open(os.path.join(HERE, "kat.json")))


@pytest.mark.parametrize("name", sorted(KAT))
def test_reader_returns_the_recorded_arrays(name):
    w = read_keras_weights(os.path.join(HERE, name))
    want = KAT[name]["arrays"]
    assert sorted(w) == sorted(want)
    for k, meta in want.items():
        assert list(w[k].shape) == meta["shape"] and str(w[k].dtype) == meta["dtype"]
        assert hashlib.sha256(np.ascontiguousarray(w[k]).tobytes()).hexdigest() == meta["sha256"], k
        assert float(w[k].ravel()[0]) == meta["first"]
    size = KAT[name]["size"]
    assert w["dense_1/kernel:0"].shape == (size * size * 3, 50)  # Flatten(W, H, 3) -> Dense(50), DQN.py:209-215


def test_reader_rejects_what_it_does_not_understand(tmp_path):
    p = tmp_path / "x"
    p.write_bytes(b"not hdf5 at all")
    with pytest.raises(H5Error):
        read_keras_weights(str(p))
    good = open(os.path.join(HERE, sorted(KAT)[0]), "rb").read()
    p.write_bytes(good[:8] + bytes([3]) + good[9:])  # superblock version 3: new-style file
    with pytest.raises(H5Error):
        read_keras_weights(str(p))


def test_layer_renumbering():
    w = {"dense_7/kernel:0": np.zeros((3, 2)), "dense_7/bias:0": np.zeros(2), "dense_9/kernel:0": np.zeros((2, 1)), "dense_9/bias:0": np.zeros(1)}
    assert sorted(canonical_dense_names(w)) == ["dense_1/bias:0", "dense_1/kernel:0", "dense_2/bias:0", "dense_2/kernel:0"]


@pytest.mark.skipif(not os.path.isdir(os.path.join(ref_harness.REF_ROOT, "Models")),
                    reason="the original project's Models/ tree is not reachable (WF_REFERENCE_ROOT)")
def test_every_model_of_the_reference_tree_parses():
    n = 0
    for f in sorted(glob.glob(os.path.join(ref_harness.REF_ROOT, "Models", "*", "*"))):
        if open(f, "rb").read(8) != b"\x89HDF\r\n\x1a\n":
            continue  # three stray non-HDF5 files ("... (1)") sit in Models/14-sized
        w = read_keras_weights(f)
        size = 10 if "/10-sized/" in f else 14
        assert w["dense_1/kernel:0"].shape == (size * size * 3, 50) and w["dense_2/kernel:0"].shape == (50, 4)
        assert len(w) in (4, 8) and all(np.isfinite(v).all() for v in w.values())
        n += 1
    assert n >= 230


def _numpy_policy(w):
    w = {k: v.astype(np.float64) for k, v in w.items()}

    def sig(z):
        return 1.0 / (1.0 + np.exp(-np.clip(z, -60, 60)))

    def q(obs):
        x = obs.reshape(-1).astype(np.float64)
        adv = sig(x @ w["dense_1/kernel:0"] + w["dense_1/bias:0"]) @ w["dense_2/kernel:0"] + w["dense_2/bias:0"]
        if "dense_3/kernel:0" in w:  # dueling head, DQN_DUEL.py:26-39
            val = sig(x @ w["dense_3/kernel:0"] + w["dense_3/bias:0"]) @ w["dense_4/kernel:0"] + w["dense_4/bias:0"]
            return val + adv - adv.mean()
        return adv
    return q


@pytest.mark.parametrize("name", sorted(KAT))
def test_reference_policy_earns_its_logged_return_on_the_oracle(name):
    """The C oracle (validated step by step against the Python reference) under the reference's trained policy."""
    from oracle import wf_oracle as wo
    meta, log = KAT[name], KAT[name]["log"]
    q = _numpy_policy(read_keras_weights(os.path.join(HERE, name)))
    env = wo.OracleEnv(dict(width=meta["size"], height=meta["size"], seed=11))
    rng = np.random.default_rng(0)
    rets, deaths, n = [], 0, 250
    for _ in range(n):
        o, done, tot = env.reset(), False, 0.0
        while not done:
            a = int(np.argmax(q(o))) if rng.random() > log["min_eps"] else int(rng.integers(4))
            o, r, done, _ = env.step(a)
            tot += r
        rets.append(tot)
        deaths += int(r == -1000)
    rets = np.array(rets)
    se = rets.std() / np.sqrt(n)
    assert abs(rets.mean() - log["mean_last_2500"]) < 4 * se + 25, (rets.mean(), se, log["mean_last_2500"])
    assert abs(deaths / n - log["death_rate_last_2500"]) < 0.05


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(KAT))
def test_reference_policy_earns_its_logged_return_on_the_cuda_env(name):
    """8192 CUDA environments, two episodes each, under the reference's trained network: the mean total
    reward and the death rate must agree with the reference's own log of that training run."""
    from wildfire_control_python_b200 import ForestFire
    from wildfire_control_python_b200 import agents as A
    meta, log = KAT[name], KAT[name]["log"]
    cls = A.DQN_BOTH if name.startswith("BOTH") else A.DQN_SARSA
    sim = ForestFire(width=meta["size"], height=meta["size"], seed=1)
    ag = cls(sim, verbose=False)
    ag.load_keras_weights(os.path.join(HERE, name))
    rets, died = ag.evaluate_batched(n_envs=8192, episodes_per_env=2, eps=log["min_eps"], seed=3)  # Q-network in the step kernel
    rets_t, died_t = ag.evaluate_batched(n_envs=4096, episodes_per_env=1, eps=log["min_eps"], seed=4, in_kernel=False)  # via torch
    se = rets.std() / np.sqrt(len(rets))
    assert len(rets) == 16384 and se < 6
    assert abs(rets_t.mean() - rets.mean()) < 5 * (se + rets_t.std() / np.sqrt(len(rets_t)))
    assert abs(died_t.mean() - died.mean()) < 0.015
    # the log's own figure is an average over 2500 episodes of a still-changing policy: +-25 covers its noise
    assert abs(rets.mean() - log["mean_last_2500"]) < 4 * se + 25, (rets.mean(), se, log["mean_last_2500"])
    assert abs(died.mean() - log["death_rate_last_2500"]) < 0.02, (died.mean(), log["death_rate_last_2500"])


@pytest.mark.gpu
@pytest.mark.parametrize("name,eps", [(sorted(KAT)[0], 0.05), (sorted(KAT)[1], 0.0), (sorted(KAT)[1], 0.3)])
def test_in_kernel_q_network_chooses_the_reference_networks_actions(name, eps):
    """WF_POLICY_MLP: the step kernel evaluates the Q-network itself (first layer kept incrementally as a sum of
    weight rows).  Every chosen action is checked against a float64 evaluation of the same weights on the
    observation the policy saw -- greedy steps must pick a maximiser of Q (up to float32 rounding), explored
    steps must follow the shared EXPLORE Philox stream -- and the trajectory against the oracle."""
    import torch
    from oracle import philox
    from oracle import wf_oracle as wo
    from tests.gpu_util import make_pair, to_np
    meta = KAT[name]
    size = meta["size"]
    cfg = dict(width=size, height=size, seed=77)
    w = {k: v.astype(np.float64) for k, v in read_keras_weights(os.path.join(HERE, name)).items()}
    N, K = 67, 300
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    gpu.set_policy_mlp(w["dense_1/kernel:0"], w["dense_1/bias:0"], w["dense_2/kernel:0"], w["dense_2/bias:0"], eps=eps)
    obs0 = to_np(gpu.reset())
    for e in orc:
        e.reset()
    obs, rew, done, acts = gpu.rollout(K, policy="mlp", return_actions=True)
    obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
    eps_u32 = 0xFFFFFFFF if eps >= 1.0 else int(eps * 4294967296.0)

    def qvals(o):
        x = o.reshape(-1).astype(np.float64)
        return (1.0 / (1.0 + np.exp(-np.clip(x @ w["dense_1/kernel:0"] + w["dense_1/bias:0"], -60, 60)))) @ w["dense_2/kernel:0"] \
            + w["dense_2/bias:0"]

    n_explored = n_greedy = n_ties = 0
    for i, e in enumerate(orc):
        episode, t = 0, 0
        for k in range(K):
            seen = obs0[i] if k == 0 else obs[k - 1, i]
            u0, u1 = philox.explore_draw(cfg["seed"], i, episode, t)
            a = int(acts[k, i])
            if u0 < eps_u32:
                assert a == u1 % 4, (i, k)
                n_explored += 1
            else:
                q = qvals(seen)
                assert q[a] >= q.max() - 1e-3 * max(1.0, abs(q.max())), (i, k, a, q)
                n_ties += int(a != int(np.argmax(q)))
                n_greedy += 1
            o, r, d, _ = e.step(a)
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k)
            t += 1
            if d:
                o = e.reset()
                episode, t = episode + 1, 0
            assert np.array_equal(obs[k, i], o), (i, k)
    assert n_greedy > 0.6 * N * K and n_ties < 0.002 * n_greedy
    assert (n_explored == 0) if eps == 0 else abs(n_explored / (N * K) - eps) < 0.02
