"""WF_POLICY_MLP on the tile family (grids larger than 32x32): every chosen action against a float64 evaluation of the
network and the EXPLORE stream, the trajectories against the oracle, and actions that do not depend on the geometry, on
how the steps are split into launches, on the observation format, on the refresh path or on sharding.  Then
evaluate_batched(in_kernel=True) and learn_batched on tile grids."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import philox
from tests.gpu_util import make_pair, to_np
from wildfire_control_python_b200 import agents as A
from wildfire_control_python_b200.batched import BatchedForestFire
from wildfire_control_python_b200.compat import get_name
from wildfire_control_python_b200.constants import make_metadata

pytestmark = pytest.mark.gpu


def _net(W, H, n_actions, hidden=50, seed=0):
    """Random weights whose greedy action follows the agent's position: a Glorot-sized first layer with the agent channel
    400 times heavier, and a second layer uniform in [-1, 1]."""
    rng = np.random.default_rng(seed)
    n_in = W * H * 3
    k1 = rng.uniform(-1, 1, (n_in, hidden)) * np.sqrt(6.0 / (n_in + hidden))
    k1[0::3] *= 400.0
    b1 = rng.uniform(-1, 1, hidden)
    k2 = rng.uniform(-1, 1, (hidden, n_actions))
    b2 = rng.uniform(-0.1, 0.1, n_actions)
    return [x.astype(np.float32) for x in (k1, b1, k2, b2)]


def _run(env, K, launches=1, **kw):
    """rollout(policy="mlp") of K steps in `launches` equal launches; (obs, reward, done, actions) on the host."""
    outs = [env.rollout(K // launches, policy="mlp", return_actions=True, **kw) for _ in range(launches)]
    return [None if outs[0][j] is None else torch.cat([o[j] for o in outs]).cpu() for j in range(4)]


def _same(a, b):
    for x, y in zip(a, b):
        assert (x is None) == (y is None)
        if x is not None:
            assert torch.equal(x, y)


CASES = [
    (dict(width=40, height=40, seed=11, extra_ignitions=2), 0.3),  # HW = 2
    (dict(width=40, height=40, seed=12, wind=[0.85, (0, 1)]), 0.0),
    (dict(width=40, height=40, seed=13), 1.0),
    (dict(width=100, height=70, seed=14, wind=[0.85, (1, 0)], extra_ignitions=6), 0.3),  # ragged H
    (dict(width=128, height=128, seed=15, extra_ignitions=3), 0.3),  # HW = 4: the VW = 4 path
    (dict(width=48, height=48, seed=16, fuel=40, allow_dig_toggle=True, n_actions=5, a_speed=2, make_rivers=True,
          wind="random", extra_ignitions=2), 0.3),  # FB = 8
]


def _check_against_float64_and_oracle(cfg, eps, N, K, auto_reset=True, launches=1):
    """A rollout(policy="mlp") of K steps in `launches` launches, step by step: explored steps follow the EXPLORE stream,
    greedy steps pick a maximiser of the float64 Q on the observation the policy saw (what the previous step emitted, or
    the new episode's first frame), and every reward, done flag and observation equals the oracle's driven with the chosen
    actions.  Without auto_reset a finished env is frozen: reward 0, done 1, its last observation, and no action is taken.
    Returns the number of episodes that ended."""
    W, H = cfg["width"], cfg["height"]
    gpu, orc = make_pair(N, cfg, auto_reset=auto_reset)
    n_act = gpu.n_actions
    k1, b1, k2, b2 = _net(W, H, n_act, seed=W + H)
    gpu.set_policy_mlp(k1, b1, k2, b2, eps=eps)
    w1, v1, w2, v2 = (x.astype(np.float64) for x in (k1, b1, k2, b2))
    obs0 = to_np(gpu.reset())
    for e in orc:
        e.reset()
    obs, rew, done, acts = (x.numpy() for x in _run(gpu, K, launches=launches))
    eps_u32 = 0xFFFFFFFF if eps >= 1.0 else int(eps * 4294967296.0)
    n_explored = n_greedy = n_ties = n_ended = n_acted = 0
    greedy_actions = set()
    for i, e in enumerate(orc):
        episode, t, frozen = 0, 0, None
        for k in range(K):
            if frozen is not None:
                assert rew[k, i] == 0.0 and done[k, i] and np.array_equal(obs[k, i], frozen), (i, k)
                continue
            seen = obs0[i] if k == 0 else obs[k - 1, i]
            u0, u1 = philox.explore_draw(cfg["seed"], i, episode, t)
            a = int(acts[k, i])
            n_acted += 1
            if u0 < eps_u32:
                assert a == u1 % n_act, (i, k)
                n_explored += 1
            else:
                x = seen.reshape(-1).astype(np.float64)
                q = (1.0 / (1.0 + np.exp(-np.clip(x @ w1 + v1, -60, 60)))) @ w2 + v2
                assert q[a] >= q.max() - 1e-3 * max(1.0, abs(q.max())), (i, k, a, q)
                n_ties += int(a != int(np.argmax(q)))
                n_greedy += 1
                greedy_actions.add(a)
            o, r, d, _ = e.step(a)
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k)
            t += 1
            if d:
                n_ended += 1
                if auto_reset:
                    o = e.reset()
                    episode, t = episode + 1, 0
                else:
                    frozen = o
            assert np.array_equal(obs[k, i], o), (i, k)
    if eps == 1.0:
        assert n_greedy == 0
    else:
        assert n_greedy > 0.5 * n_acted and n_ties <= 0.002 * n_greedy
        assert len(greedy_actions) > 1
    if eps == 0.0:
        assert n_explored == 0
    return n_ended


@pytest.mark.parametrize("cfg,eps", CASES)
def test_tile_policy_chooses_the_networks_actions(cfg, eps):
    """Every action against a float64 evaluation and the EXPLORE stream, every step against the oracle, auto-resets
    included (at least one episode ends in every case)."""
    W, H = cfg["width"], cfg["height"]
    assert _check_against_float64_and_oracle(cfg, eps, 4, 96 if W * H > 5000 else 160) > 0


@pytest.mark.parametrize("cfg", [dict(width=40, height=40, seed=13, extra_ignitions=2),
                                 dict(width=48, height=48, seed=16, fuel=40, allow_dig_toggle=True, n_actions=5, a_speed=2,
                                      make_rivers=True, wind="random", extra_ignitions=2)])
def test_tile_policy_freezes_finished_envs(cfg):
    """Without auto_reset: envs that finish are frozen (reward 0, done 1, unchanged observation; the policy pass is skipped
    for them, in the launch where they finish and in the later ones) while the others keep acting as checked above."""
    assert _check_against_float64_and_oracle(cfg, 0.3, 6, 240, auto_reset=False, launches=3) > 0


def test_tile_policy_refuses_weights_beyond_the_exact_sum():
    """On tile grids the first layer is an exact int64 fixed-point sum: wf_set_policy_mlp refuses a kernel1 entry that
    is not finite or reaches 2^31 / (2 W H + 1), before anything is packed."""
    from wildfire_control_python_b200 import _lib
    env = BatchedForestFire(2, auto_reset=True, width=40, height=40, seed=1)
    k1, b1, k2, b2 = _net(40, 40, 4)
    bound = 2.0 ** 31 / (2 * 40 * 40 + 1)
    for bad in (np.float32(bound * 1.001), np.float32(-bound * 1.001), np.float32(np.inf), np.float32(np.nan)):
        k = k1.copy()
        k[123, 7] = bad
        with pytest.raises(_lib.WildfireError):
            env.set_policy_mlp(k, b1, k2, b2, eps=0.1)
    k = k1.copy()
    k[123, 7] = np.float32(bound * 0.999)
    env.set_policy_mlp(k, b1, k2, b2, eps=0.1)  # within the bound
    env.close()


@pytest.mark.parametrize("cfg", [dict(width=100, height=70, seed=21, wind=[0.85, (1, 0)], extra_ignitions=6, a_speed=2),
                                 dict(width=128, height=128, seed=22, make_rivers=True, wind="random", extra_ignitions=3)])
def test_tile_policy_does_not_depend_on_the_geometry(monkeypatch, cfg):
    """The same actions, rewards, done flags and observations for every (threads, cluster size): the first layer is an
    exact integer sum whatever the slices."""
    W, H = cfg["width"], cfg["height"]
    net = _net(W, H, 4, seed=3)
    ref = None
    for T, CS in [(128, 1), (256, 1), (512, 1), (128, 2), (256, 4), (128, 8), (128, 16)]:
        monkeypatch.setenv("WF_TILE_T", str(T))
        monkeypatch.setenv("WF_TILE_CS", str(CS))
        env = BatchedForestFire(3, auto_reset=True, **cfg)
        assert env.tile_geometry == (T, CS)
        env.set_policy_mlp(*net, eps=0.2)
        env.reset()
        out = _run(env, 64, launches=2)
        env.close()
        if ref is None:
            ref = out
        else:
            _same(ref, out)


def test_tile_policy_does_not_depend_on_how_it_is_called():
    """One launch of 64 steps, 64 launches of 1 and 4 of 16 agree; so do uint8, bits and obs=None rollouts; and so do
    differently split launches after set_state and after set_fire_to between launches."""
    cfg = dict(width=64, height=48, seed=31, extra_ignitions=4, a_speed=2)
    net = _net(64, 48, 4, seed=5)

    def env_(obs_dtype=torch.uint8):
        e = BatchedForestFire(4, obs_dtype=obs_dtype, auto_reset=True, **cfg)
        e.set_policy_mlp(*net, eps=0.1)
        e.reset()
        return e

    ref = _run(env_(), 64, launches=1)
    _same(ref, _run(env_(), 64, launches=64))
    _same(ref, _run(env_(), 64, launches=4))
    bits = _run(env_("bits"), 64, launches=4)
    none = _run(env_(), 64, launches=2, obs=False)
    for out in (bits, none):
        for j in (1, 2, 3):
            assert torch.equal(ref[j], out[j])
    # the state changed from outside between launches: the policy sees it the same way whatever the split
    fire = torch.tensor([[5, 7], [60, 40], [-1, 0], [32, 24]], dtype=torch.int32, device="cuda")
    outs = []
    for split in (1, 8):
        e = env_()
        e.rollout(16, policy="mlp", obs=False)
        e.set_fire_to(fire)
        o1 = _run(e, 32, launches=split)
        e.set_state(**e.get_state())
        o2 = _run(e, 32, launches=split)
        outs.append(o1 + o2)
    _same(outs[0], outs[1])


def test_tile_policy_host_and_device_refresh_agree():
    """set_policy_mlp and set_policy_mlp_dev give byte-identical rollouts, including a device refresh queued behind a
    rollout on the same stream."""
    cfg = dict(width=48, height=40, seed=41, allow_dig_toggle=True, n_actions=5, extra_ignitions=2)
    nets = [_net(48, 40, 5, seed=s) for s in (7, 8)]
    outs = []
    for dev_path in (False, True):
        env = BatchedForestFire(6, auto_reset=True, **cfg)
        env.reset()
        res = []
        for k1, b1, k2, b2 in nets:
            if dev_path:
                env.set_policy_mlp_dev(*(torch.from_numpy(x).cuda() for x in (k1.T.copy(), b1, k2.T.copy(), b2)), eps=0.2)
            else:
                torch.cuda.synchronize()
                env.set_policy_mlp(k1, b1, k2, b2, eps=0.2)
            res.append(env.rollout(48, policy="mlp", return_actions=True))
        outs.append([[t.cpu() for t in r] for r in res])
        env.close()
    for r_host, r_dev in zip(*outs):
        _same(r_host, r_dev)


def test_tile_policy_sharded_batch_acts_as_the_whole():
    """A batch split over two handles by env_id_base acts exactly as the unsplit batch, over three launches."""
    cfg = dict(width=40, height=40, seed=51, extra_ignitions=3)
    net = _net(40, 40, 4, seed=9)
    envs = [BatchedForestFire(6, auto_reset=True, **cfg), BatchedForestFire(2, auto_reset=True, env_id_base=0, **cfg),
            BatchedForestFire(4, auto_reset=True, env_id_base=2, **cfg)]
    for e in envs:
        e.set_policy_mlp(*net, eps=0.3)
        e.reset()
    for _ in range(3):
        whole, a, b = (_run(e, 40) for e in envs)
        for j in range(4):
            assert torch.equal(whole[j][:, :2], a[j]) and torch.equal(whole[j][:, 2:], b[j]), j


# ---------------------------------------------------------------------------------------------------------------------
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


def _agent(name, W, H, seed=0, **kw):
    torch.manual_seed(seed)
    return getattr(A, name)(_Sim(W, H, **kw), verbose=False, device="cuda")


def _flat(ag):
    from torch.nn.utils import parameters_to_vector as p2v
    ps = list(ag.model.parameters())
    st = [ag.optimizer.state[p] for p in ps]
    return [p2v(x).detach().cpu().numpy() for x in (ps, list(ag.target.parameters()), [s["m"] for s in st], [s["v"] for s in st])]


def test_evaluate_batched_in_kernel_on_a_tile_grid():
    """evaluate_batched(in_kernel=True) on 48x48: returns and deaths equal those of one explicit rollout(policy="mlp")
    with the same seed and network."""
    from wildfire_control_python_b200.constants import DQN_DEFAULTS as _D
    ag = _agent("DQN", 48, 48, seed=4)
    N, eps, seed = 64, 0.1, 5
    rets, died = ag.evaluate_batched(n_envs=N, eps=eps, seed=seed, in_kernel=True)
    keys = {k: v for k, v in ag.METADATA.items() if k not in _D and k not in ("debug", "a_speed_iter", "seed", "auto_reset")}
    env = BatchedForestFire(N, auto_reset=True, seed=seed, **keys)
    w = ag.get_weights()
    env.set_policy_mlp(w["dense_1/kernel:0"], w["dense_1/bias:0"], w["dense_2/kernel:0"], w["dense_2/bias:0"], eps=eps)
    env.reset()
    _, rew, done = env.rollout(4096, policy="mlp", obs=False)
    rew, done = to_np(rew), to_np(done)
    assert done.any(axis=0).all()
    first = done.argmax(axis=0)
    want = np.cumsum(rew, axis=0)[first, np.arange(N)]
    want_died = rew[first, np.arange(N)] == float(ag.METADATA["death_penalty"])
    # (evaluate_batched sums 64-step chunks: only the float64 summation order differs)
    assert np.allclose(rets, want, rtol=1e-12, atol=1e-9) and np.array_equal(died, want_died)


@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"])
def test_learn_batched_end_to_end_on_a_tile_grid(name, tmp_path):
    """Demonstrations, then learn_batched on 40x40 (replays as fit_batch calls): the logs in the reference's format, eps
    on its schedule, the same weights from two runs with one seed, and replay() / evaluate_batched afterwards."""
    def run():
        ag = _agent(name, 40, 40, seed=1)
        ag.out_dir = str(tmp_path)
        ag.collect_memories_batched(8, n_envs=64, k_steps=64, seed=2)
        init = len(ag.memory)
        steps = ag.learn_batched(120, n_envs=128, k_steps=16, replays_per_launch=4, seed=3)
        return ag, init, steps

    ag, init, steps = run()
    ag2, _, _ = run()
    for x, y in zip(_flat(ag), _flat(ag2)):
        assert x.tobytes() == y.tobytes()
    assert steps > 0 and init > 0
    logs = sorted(os.listdir(tmp_path / "Logs"))
    with open(tmp_path / "Logs" / logs[0]) as f:
        log = json.load(f)
    assert log["n_episodes"] == 120 and len(log["total_rewards"]) == 120 and len(log["agent_deaths"]) == 120
    assert log["init_memories"] == init and log["total_time"] >= 0
    assert set(log) >= {"best_reward", "total_rewards", "agent_pos", "agent_deaths", "maps", "init_memories", "total_time",
                        "n_episodes", "metadata"}
    eps, ended = np.array(ag.eps_per_launch), np.array(ag.episodes_before_launch)
    assert ended[0] == 0 and eps[0] == ag.max_eps and (np.diff(ended) >= 0).all() and ended[-1] < 120
    assert np.allclose(eps, ag.min_eps + (ag.max_eps - ag.min_eps) * np.exp(-ag.eps_decay_rate * ended), rtol=0, atol=1e-12)
    ag.replay()
    rets, died = ag.evaluate_batched(n_envs=64, seed=9, in_kernel=True)
    assert len(rets) == 64 and len(died) == 64


def test_learn_batched_on_a_tile_grid_refreshes_the_target_on_schedule():
    """target_update = 3 with 4 replays per launch: the refresh phase carries across launches, so after n replays the
    target equals the model exactly when n is a multiple of 3, and the next refresh is 3 - n % 3 replays away."""
    ag = _agent("DQN", 40, 40, seed=6, target_update=3)
    ag.collect_memories_batched(4, n_envs=64, k_steps=64, seed=2)
    assert len(ag.memory) > ag.METADATA["batch_size"]  # so every launch replays
    for n_eps in (10, 25, 40):
        ag.learn_batched(n_eps, n_envs=32, k_steps=8, replays_per_launch=4, seed=n_eps)
        n = 4 * len(ag.eps_per_launch)
        model, target = (torch.nn.utils.parameters_to_vector(m.parameters()) for m in (ag.model, ag.target))
        assert torch.equal(model, target) == (n % 3 == 0), n
        assert ag._until_sync == 3 - n % 3
