"""Batched learning on the GPU: wf_replay_fit (DQN.fit_batches_fused) against the N1 golden fixture and against the torch
fit_batch loop, its determinism and out-of-range rules; wf_set_policy_mlp_dev against wf_set_policy_mlp; learn_batched
end to end."""
import copy
import json
import os

import numpy as np
import pytest
import torch

from tests.test_agents import FakeSim, _load_n1
from wildfire_control_python_b200 import agents as A
from wildfire_control_python_b200 import pack_obs, unpack_obs
from wildfire_control_python_b200.batched import BatchedForestFire
from wildfire_control_python_b200.compat import get_name
from wildfire_control_python_b200.constants import make_metadata

pytestmark = pytest.mark.gpu

# Rise in mean evaluate_batched return that test_learn_batched_improves_the_policy demands.  Measured on a B200 with that
# test's configuration for seeds 0, 1 and 2 (untrained returns -265 ... -427): DQN +1442 / +1491 / +1479, DQN_SARSA
# +1833 / +1399 / -95, DQN_DUEL +466 / +689 / +2034, DQN_BOTH +1675 / +1285 / +1769.  11 of the 12 runs gain more than
# 450; one SARSA run at this short budget had not yet left the untrained level.  The test uses seed 0, and the run is
# deterministic for a given seed.
MARGIN = 300.0


class _World:
    DEPTH = 3
    agents = []

    def __init__(self, W, H):
        self.WIDTH, self.HEIGHT = W, H


class _Sim:
    """The surface DQN.__init__ / write_data read, for any grid."""

    def __init__(self, W, H, **kw):
        self.METADATA = make_metadata(width=W, height=H, **kw)
        self.n_actions, self.DEBUG, self.get_name = int(self.METADATA["n_actions"]), 1, get_name
        self.W = _World(W, H)


def _agent(name, W=10, H=10, seed=0, **kw):
    torch.manual_seed(seed)
    return getattr(A, name)(_Sim(W, H, **kw), verbose=False, device="cuda")


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"])
def test_fused_replay_reproduces_the_n1_fixture(name):
    """The golden fixture of agents' N1 test (two consecutive updates, float64 restatement of Keras): loss and every
    updated weight with the tolerances test_agents._check_n1 uses.  The targets are internal to the kernel; the loss,
    computed from them, pins them."""
    fx = _load_n1(name)
    ag = getattr(A, name)(FakeSim(), verbose=False, device="cuda")
    keys = sorted(k[3:] for k in fx if k.startswith("w0/"))
    ag.set_weights({k: fx["w0/" + k] for k in keys})
    with torch.no_grad():
        for lname, m in ag.target.named_children():
            m.weight.copy_(torch.as_tensor(fx[f"target/{lname}/kernel:0"]).t())
            m.bias.copy_(torch.as_tensor(fx[f"target/{lname}/bias:0"]))
    for t in (1, 2):
        b = {k: fx[f"t{t}/batch_{k}"] for k in ("s", "a", "r", "sp", "ap", "d")}
        B = len(b["a"])
        obs = torch.as_tensor(np.concatenate([b["s"], b["sp"]]).reshape(-1, 10, 10, 3), device="cuda")
        frames = pack_obs(obs)
        rows = torch.arange(2 * B, device="cuda")
        loss = ag.fit_batches_fused(frames, rows[:B], rows[B:], b["a"], b["ap"], b["r"], b["d"], 1)
        assert float(loss[0]) == pytest.approx(float(fx[f"t{t}/loss"]), rel=1e-4)
        got = ag.get_weights()
        for k in keys:
            want = fx[f"t{t}/w/{k}"]
            have = got[k][::16] if got[k].shape[0] == 300 else got[k]
            assert np.allclose(have, want, rtol=0, atol=2e-6), (name, t, k, np.abs(have - want).max())
        assert ag.optimizer.state[ag.model.dense_1.weight]["t"] == t


def _random_replays(ag, n_frames, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    W, H = ag.obs_shape[0], ag.obs_shape[1]
    obs = (torch.rand((n_frames, W, H, 3), device="cuda", generator=g) < 0.35).to(torch.uint8)
    frames = pack_obs(obs)
    s_row = torch.randint(0, n_frames, (n,), device="cuda", generator=g)
    sp_row = torch.randint(0, n_frames, (n,), device="cuda", generator=g)
    a = torch.randint(0, ag.action_size, (n,), device="cuda", generator=g)
    ap = torch.randint(0, ag.action_size, (n,), device="cuda", generator=g)
    r = torch.randn((n,), device="cuda", generator=g) * 3
    d = torch.rand((n,), device="cuda", generator=g) < 0.1
    return frames, s_row, sp_row, a, ap, r, d


def _warm(ag, frames, n_frames, seed):
    """A few torch updates so that Adam starts at t > 0 and the target differs from the model."""
    fr, s, sp, a, ap, r, d = _random_replays(ag, n_frames, 3 * 32, seed + 1)
    W, H = ag.obs_shape[0], ag.obs_shape[1]
    for i in range(3):
        sl = slice(32 * i, 32 * i + 32)
        ag.fit_batch((unpack_obs(fr, W, H, s[sl], torch.uint8), a[sl], r[sl], unpack_obs(fr, W, H, sp[sl], torch.uint8),
                      ap[sl], d[sl]))


def _flat(ag):
    from torch.nn.utils import parameters_to_vector as p2v
    ps = list(ag.model.parameters())
    st = [ag.optimizer.state[p] for p in ps]
    return [p2v(x).detach().cpu().numpy() for x in (ps, list(ag.target.parameters()), [s["m"] for s in st], [s["v"] for s in st])]


@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"])
@pytest.mark.parametrize("W,B", [(10, 32), (10, 256), (32, 32), (32, 256)])
def test_fused_replays_match_the_torch_loop(name, W, B):
    """64 replays in one launch against 64 fit_batch calls from the same weights, target and Adam state (t = 3), with the
    same rows and a target refresh inside the run (target_update = 20, phase 7: refreshes after replays 7, 27 and 47).

    Tolerance: the kernel sums in a different order than cuBLAS, so every update differs in the last float32 bits, and
    these differences accumulate over 64 updates.  Measured on a B200, the largest difference over all 16 cases and
    every element (biases included) was 3.9e-7 for weights and target, 7.7e-8 for m and 7.5e-9 for v; the bounds are
    about 25 times that.  Adam divides m by sqrt(v) + 1e-7, so an element whose gradient were pure rounding noise
    could take a step of the other sign (a difference of about lr = 5e-3): these inputs have no such element, and such
    a step would fail the test rather than pass unnoticed."""
    R = 64
    ag = _agent(name, W, W, seed=W + B)
    n_frames = 4 * B
    frames, s, sp, a, ap, r, d = _random_replays(ag, n_frames, R * B, seed=W * B)
    _warm(ag, frames, n_frames, W * B)
    ref = copy.deepcopy(ag)
    until, te = 7, ref.target_update_freq
    ref_loss = []
    for i in range(R):
        sl = slice(B * i, B * i + B)
        ref_loss.append(ref.fit_batch((unpack_obs(frames, W, W, s[sl], torch.uint8), a[sl], r[sl],
                                       unpack_obs(frames, W, W, sp[sl], torch.uint8), ap[sl], d[sl])))
        until -= 1
        if until == 0:
            until = te
            ref.target.load_state_dict(ref.model.state_dict())
    loss = ag.fit_batches_fused(frames, s, sp, a, ap, r, d, R, phase=7).cpu().numpy()
    assert ag._until_sync == until
    assert np.allclose(loss, ref_loss, rtol=1e-3, atol=1e-5), np.abs(loss - ref_loss).max()
    for what, x, y in zip(("params", "target", "m", "v"), _flat(ag), _flat(ref)):
        bound = {"params": 1e-5, "target": 1e-5, "m": 2e-6, "v": 2e-7}[what]
        diff = np.abs(x - y)
        assert diff.max() <= bound, (what, diff.max(), int(diff.argmax()))
    assert ag.optimizer.state[ag.model.dense_1.weight]["t"] == 3 + R


@pytest.mark.parametrize("name", ["DQN_SARSA", "DQN_BOTH"])
def test_fused_replay_is_deterministic(name):
    ag = _agent(name, 14, 14, seed=3)
    frames, s, sp, a, ap, r, d = _random_replays(ag, 512, 64 * 128, seed=4)
    _warm(ag, frames, 512, 4)
    ag2 = copy.deepcopy(ag)
    l1 = ag.fit_batches_fused(frames, s, sp, a, ap, r, d, 64).cpu().numpy()
    l2 = ag2.fit_batches_fused(frames, s, sp, a, ap, r, d, 64).cpu().numpy()
    assert l1.tobytes() == l2.tobytes()
    for x, y in zip(_flat(ag), _flat(ag2)):
        assert x.tobytes() == y.tobytes()


def test_out_of_range_rows_and_actions():
    """Rows outside the frames are all-zero observations; a next action outside [0, A) bootstraps nothing (as if done);
    an action outside [0, A) replaces no target entry (the torch update with that sample's target = Q_target(s))."""
    B, W = 32, 10
    ag = _agent("DQN_SARSA", W, W, seed=5)
    frames, s, sp, a, ap, r, d = _random_replays(ag, 64, B, seed=6)
    _warm(ag, frames, 64, 6)
    zero_frames = torch.cat([frames, torch.zeros_like(frames[:1])])
    bad = torch.arange(B, device="cuda") % 4 == 0
    # rows: -5 / 10**9 against an explicit all-zero row
    x, y = copy.deepcopy(ag), copy.deepcopy(ag)
    x.fit_batches_fused(frames, torch.where(bad, -5, s), torch.where(bad, 10**9, sp), a, ap, r, d, 1)
    y.fit_batches_fused(zero_frames, torch.where(bad, 64, s), torch.where(bad, 64, sp), a, ap, r, d, 1)
    for p, q in zip(_flat(x), _flat(y)):
        assert p.tobytes() == q.tobytes()
    # next actions: out of range == terminal
    x, y = copy.deepcopy(ag), copy.deepcopy(ag)
    x.fit_batches_fused(frames, s, sp, a, torch.where(bad, 99, ap), r, d, 1)
    y.fit_batches_fused(frames, s, sp, a, ap, r, d | bad, 1)
    for p, q in zip(_flat(x), _flat(y)):
        assert p.tobytes() == q.tobytes()
    # actions: out of range replaces nothing
    x, ref = copy.deepcopy(ag), copy.deepcopy(ag)
    a_bad = torch.where(bad, -1, a)
    lx = float(x.fit_batches_fused(frames, s, sp, a_bad, ap, r, d, 1)[0])
    su, spu = unpack_obs(frames, W, W, s, torch.float32), unpack_obs(frames, W, W, sp, torch.float32)
    tgt = ref.replay_targets((su, a, r, spu, ap, d))
    with torch.no_grad():
        tgt[bad] = ref.target(su[bad])
    loss = torch.nn.functional.mse_loss(ref.model(su), tgt)
    ref.optimizer.zero_grad(set_to_none=True)
    loss.backward()
    ref.optimizer.step()
    assert lx == pytest.approx(float(loss), rel=1e-4)
    for p, q in zip(_flat(x)[:1], _flat(ref)[:1]):
        assert np.abs(p - q).max() < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,hidden,dig", [(14, 50, False), (14, 64, True), (32, 50, True), (20, 64, False)])
def test_device_policy_refresh_matches_the_host_path(W, hidden, dig):
    """set_policy_mlp_dev and set_policy_mlp give the same 256-step mlp rollouts (actions, rewards, dones, observations),
    on 16- and 32-lane grids, with A = 4 and 5; and a device refresh queued behind a rollout on the same stream is ordered
    without a synchronisation."""
    N, K, eps = 512, 256, 0.1
    cfg = dict(width=W, height=W, seed=11, allow_dig_toggle=dig, n_actions=5 if dig else 4)
    g = torch.Generator(device="cuda").manual_seed(W + hidden)
    A_ = cfg["n_actions"]
    nets = [[torch.randn(shape, device="cuda", generator=g) * sc for shape, sc in
             (((hidden, W * W * 3), 0.3), ((hidden,), 1.0), ((A_, hidden), 1.0), ((A_,), 1.0))] for _ in range(2)]
    outs = []
    for dev_path in (False, True):
        env = BatchedForestFire(N, auto_reset=True, **cfg)
        env.reset()
        res = []
        for w1, b1, w2, b2 in nets:
            if dev_path:
                env.set_policy_mlp_dev(w1, b1, w2, b2, eps=eps)  # the second one is queued behind the first rollout
            else:
                torch.cuda.synchronize()
                env.set_policy_mlp(w1.t().cpu(), b1.cpu(), w2.t().cpu(), b2.cpu(), eps=eps)
            res.append(env.rollout(K, policy="mlp", return_actions=True))
        outs.append([[t.cpu() for t in r] for r in res])
        env.close()
    for r_host, r_dev in zip(*outs):
        for x, y in zip(r_host, r_dev):
            assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"])
def test_learn_batched_end_to_end(name, tmp_path):
    """Demonstrations, then learn_batched on 10x10: the logs in the reference's format, eps on its schedule, the same
    weights from two runs with one seed, and replay() / evaluate_batched afterwards."""
    def run():
        ag = _agent(name, 10, 10, seed=1)
        ag.out_dir = str(tmp_path)
        ag.collect_memories_batched(20, n_envs=256, k_steps=64, seed=2)
        init = len(ag.memory)
        steps = ag.learn_batched(300, n_envs=256, k_steps=16, seed=3)
        return ag, init, steps

    ag, init, steps = run()
    ag2, _, _ = run()
    for x, y in zip(_flat(ag), _flat(ag2)):
        assert x.tobytes() == y.tobytes()
    assert steps > 0 and init > 0
    logs = sorted(os.listdir(tmp_path / "Logs"))
    with open(tmp_path / "Logs" / logs[0]) as f:
        log = json.load(f)
    assert log["n_episodes"] == 300 and len(log["total_rewards"]) == 300 and len(log["agent_deaths"]) == 300
    assert log["init_memories"] == init and log["total_time"] >= 0
    assert set(log) >= {"best_reward", "total_rewards", "agent_pos", "agent_deaths", "maps", "init_memories", "total_time",
                        "n_episodes", "metadata"}
    # eps before every launch: min + (max - min) * exp(-rate * episodes completed before it) (decay_epsilon)
    eps, ended = np.array(ag.eps_per_launch), np.array(ag.episodes_before_launch)
    assert ended[0] == 0 and eps[0] == ag.max_eps and (np.diff(ended) >= 0).all() and ended[-1] < 300
    assert np.allclose(eps, ag.min_eps + (ag.max_eps - ag.min_eps) * np.exp(-ag.eps_decay_rate * ended), rtol=0, atol=1e-12)
    assert eps[-1] < eps[0]
    ag.replay()
    rets, died = ag.evaluate_batched(n_envs=512, seed=9)
    assert len(rets) == 512 and len(died) == 512


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA"])
def test_replay_ring_of_one_group_holds_the_rollouts_transitions(name):
    """learn_batched's ring (_PackedReplayRing with one group, i.e. one demonstration memory) over 6 launches of the mlp
    policy with auto-resets, wrapping twice: after every launch each sampleable (s, a, r, s', a', done) equals the one of
    a uint8 rollout of the same seed re-driven with the recorded actions (s = the frame before step t, the reset frame for
    t = 0; a' = the action of step t + 1), the window holds at least memory_size transitions, and the demonstrations
    come back unchanged."""
    from wildfire_control_python_b200.constants import DQN_DEFAULTS
    N, K, W, launches = 64, 16, 10, 6
    ag = _agent(name, W, W, seed=7)
    ag.collect_memories_batched(3, n_envs=64, k_steps=64, seed=1)
    D = len(ag.memory)
    keys = {k: v for k, v in ag.METADATA.items() if k not in DQN_DEFAULTS and k not in ("debug", "a_speed_iter", "seed",
                                                                                      "auto_reset")}
    env = BatchedForestFire(N, obs_dtype="bits", auto_reset=True, seed=5, **keys)
    ref = BatchedForestFire(N, auto_reset=True, seed=5, **keys)
    memory_size = K * N
    ring = A._PackedReplayRing(env, K, memory_size, [ag.memory], ag._SARSA)
    assert ring.T == 2 * K  # wraps after two launches
    obs = [ref.reset().clone()]  # obs[t + 1] = the frame of step t
    acts, rews, dones = [], [], []
    net = ag.model
    for launch in range(launches):
        env.set_policy_mlp_dev(net.dense_1.weight, net.dense_1.bias, net.dense_2.weight, net.dense_2.bias, eps=0.3)
        ring.launch()
        sl = slice((launch * K) % ring.T, (launch * K) % ring.T + K)
        a_k = ring.acts[sl].clone()
        o, r, d = ref.rollout(K, actions=a_k)
        obs += list(o.clone())
        acts += list(a_k)
        rews += list(r)
        dones += list(d)
        steps = (launch + 1) * K
        lo, hi = max(0, steps - ring.T + 1), steps - (1 if ag._SARSA else 0)
        assert ring.sampleable(0) == (hi - lo) * N + D
        if launch >= 2:
            assert (hi - lo) * N >= memory_size
        s_row, sp_row, a, ap, r, d = ring.gather(torch.arange(ring.sampleable(0), device="cuda"))
        s_u8 = unpack_obs(ring.frames, W, W, s_row, torch.uint8)
        sp_u8 = unpack_obs(ring.frames, W, W, sp_row, torch.uint8)
        ts = range(lo, hi)
        assert torch.equal(s_u8[:(hi - lo) * N], torch.cat([obs[t] for t in ts]))
        assert torch.equal(sp_u8[:(hi - lo) * N], torch.cat([obs[t + 1] for t in ts]))
        assert torch.equal(a[:(hi - lo) * N], torch.cat([acts[t] for t in ts]))
        assert torch.equal(r[:(hi - lo) * N], torch.cat([rews[t] for t in ts]).float())
        assert torch.equal(d[:(hi - lo) * N].bool(), torch.cat([dones[t] for t in ts]))
        if ag._SARSA:
            assert torch.equal(ap[:(hi - lo) * N], torch.cat([acts[t + 1] for t in ts]))
        m = ag.memory
        assert torch.equal(s_u8[(hi - lo) * N:], m._s[:D]) and torch.equal(sp_u8[(hi - lo) * N:], m._sp[:D])
        assert torch.equal(a[(hi - lo) * N:].long(), m._a[:D]) and torch.equal(r[(hi - lo) * N:], m._r[:D])
        assert torch.equal(d[(hi - lo) * N:].bool(), m._d[:D])
        if ag._SARSA:
            assert torch.equal(ap[(hi - lo) * N:].long(), m._ap[:D])
    assert int(torch.stack(dones).sum()) > 0  # episodes ended: auto-reset frames are among the checked transitions
    env.close()
    ref.close()


@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"])
def test_learn_batched_improves_the_policy(name, tmp_path):
    """50 demonstration episodes, then 4000 training episodes of learn_batched (64 envs, 16 steps and 256 replays per
    launch) on 10x10: the mean return of evaluate_batched (2048 episodes, eps = min_eps) must rise by at least MARGIN
    over the untrained network's."""
    ag = _agent(name, 10, 10, seed=0)
    ag.out_dir = str(tmp_path)
    before, _ = ag.evaluate_batched(n_envs=2048, seed=100)
    ag.collect_memories_batched(50, n_envs=256, k_steps=64, seed=0)
    ag.learn_batched(4000, n_envs=64, k_steps=16, replays_per_launch=256, seed=0)
    after, _ = ag.evaluate_batched(n_envs=2048, seed=100)
    print(f"{name}: untrained {before.mean():.1f}, trained {after.mean():.1f}")
    assert after.mean() - before.mean() >= MARGIN, (before.mean(), after.mean())
