"""Populations on the GPU: wf_replay_fit_many against one wf_replay_fit call per learner (bit for bit, several waves of
clusters), the in-kernel policy with one network per env group against separate handles, and learn_population against
each agent trained alone by learn_batched."""
import copy
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from wildfire_control_python_b200 import _lib, pack_obs
from wildfire_control_python_b200 import agents as A
from wildfire_control_python_b200.batched import BatchedForestFire
from wildfire_control_python_b200.compat import get_name
from wildfire_control_python_b200.constants import make_metadata

pytestmark = pytest.mark.gpu


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dueling,sarsa,B", [(0, 0, 32), (0, 1, 256), (1, 0, 256), (1, 1, 32)])
def test_replay_fit_many_equals_one_call_per_learner(dueling, sarsa, B):
    """20 learners (more clusters of 16 CTAs than a B200 holds at once) with their own parameters, moments, lr, gamma,
    target_every, phase and Adam step, and out-of-range rows and actions among their transitions: params, target, m, v
    and loss of every learner are bit-identical to a wf_replay_fit call on that learner alone."""
    L = _lib.lib()
    M, R, W, H, hid, A_ = 20, 6, 14, 14, 50, 4
    n_frames = 3000
    g = torch.Generator(device="cuda").manual_seed(17 + B + 2 * dueling + sarsa)
    P = _lib.mlp_param_count(W, H, hid, A_, dueling)
    frames = pack_obs((torch.rand((n_frames, W, H, 3), device="cuda", generator=g) < 0.35).to(torch.uint8))
    sh = _lib.WfMlpShape(width=W, height=H, hidden=hid, n_actions=A_, dueling=dueling, batch=B)
    n = R * B
    state0, data, hps = [], [], []
    rng = np.random.default_rng(B + dueling)
    for j in range(M):
        params = torch.randn(P, device="cuda", generator=g) * 0.05
        m = torch.randn(P, device="cuda", generator=g) * 1e-3
        v = torch.rand(P, device="cuda", generator=g) * 1e-4
        state0.append((params, params + torch.randn(P, device="cuda", generator=g) * 0.01, m, v))
        rows = lambda: torch.randint(-20, n_frames + 20, (n,), device="cuda", generator=g)  # noqa: E731
        acts = lambda: torch.randint(-1, A_ + 1, (n,), device="cuda", generator=g, dtype=torch.int32)  # noqa: E731
        data.append((rows(), rows(), acts(), acts() if sarsa else None, torch.randn(n, device="cuda", generator=g) * 5,
                     (torch.rand(n, device="cuda", generator=g) < 0.1).to(torch.uint8)))
        te = int(rng.integers(1, 9))
        hps.append(_lib.WfFitParams(gamma=float(rng.uniform(0.8, 0.999)), lr=float(rng.uniform(1e-4, 1e-2)), beta_1=0.9,
                                    beta_2=0.999, epsilon=1e-7, clipvalue=1.0, adam_t=int(rng.integers(0, 500)),
                                    target_every=te, phase=int(rng.integers(1, te + 1))))
    many = [[t.clone() for t in s] + [torch.full((R,), -1.0, device="cuda")] for s in state0]
    desc = (_lib.WfFitLearner * M)(*[
        _lib.WfFitLearner(*[_p(t) for t in many[j][:4]], *[_p(t) for t in data[j]], _p(many[j][4]), hps[j]) for j in range(M)])
    _lib.check(L.wf_replay_fit_many(C.byref(sh), M, desc, R, _p(frames), n_frames, _stream()))
    for j in range(M):
        one = [t.clone() for t in state0[j]] + [torch.full((R,), -1.0, device="cuda")]
        s, sp, a, ap, r, d = data[j]
        _lib.check(L.wf_replay_fit(C.byref(sh), C.byref(hps[j]), R, *[_p(t) for t in one[:4]], _p(frames), n_frames, _p(s),
                                   _p(sp), _p(a), _p(ap), _p(r), _p(d), _p(one[4]), _stream()))
        for x, y, what in zip(many[j], one, ("params", "target", "m", "v", "loss")):
            assert torch.equal(x, y), (j, what)
        assert not torch.equal(many[j][0], state0[j][0])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,dig,dueling", [(14, False, 0), (14, True, 1), (24, False, 1), (24, True, 0)])
def test_group_networks_act_as_separate_handles(W, dig, dueling):
    """One handle of M x G envs with M networks (eps 0, 0.3, 1 across groups) against M handles of G envs with
    env_id_base = j * G, each with its network through set_policy_mlp_dev: the same actions, bit observations, rewards and
    done flags over 2 x 16 steps with auto-resets, the second refresh queued behind the first rollout."""
    M, G, K, hid = 4, 16, 16, 50
    A_ = 5 if dig else 4
    eps = [0.0, 0.3, 1.0, 0.3]
    cfg = dict(width=W, height=W, seed=23, allow_dig_toggle=dig, n_actions=A_)
    P = _lib.mlp_param_count(W, W, hid, A_, dueling)
    n_in = W * W * 3
    g = torch.Generator(device="cuda").manual_seed(W + 2 * dig + dueling)
    rounds = [torch.randn((M, P), device="cuda", generator=g) * 0.3 for _ in range(2)]

    def split(flat):  # dense_1 / dense_2 of the flat layout, nn.Linear orientation
        w1 = flat[:hid * n_in].view(hid, n_in)
        b1 = flat[hid * n_in:hid * n_in + hid]
        w2 = flat[hid * n_in + hid:hid * n_in + hid + A_ * hid].view(A_, hid)
        b2 = flat[hid * n_in + hid + A_ * hid:hid * n_in + hid + A_ * hid + A_]
        return w1, b1, w2, b2

    pop = BatchedForestFire(M * G, obs_dtype="bits", auto_reset=True, **cfg)
    pop.reset()
    got = []
    for params in rounds:
        pop.set_policy_mlp_flat_dev(params, hid, dueling, eps)
        got.append([t.clone() for t in pop.rollout(K, policy="mlp", return_actions=True)])
    for j in range(M):
        env = BatchedForestFire(G, obs_dtype="bits", auto_reset=True, env_id_base=j * G, **cfg)
        env.reset()
        for params, (o, r, d, a) in zip(rounds, got):
            env.set_policy_mlp_dev(*split(params[j]), eps=eps[j])
            o1, r1, d1, a1 = env.rollout(K, policy="mlp", return_actions=True)
            cols = slice(j * G, (j + 1) * G)
            assert torch.equal(a[:, cols], a1), j
            assert torch.equal(o[:, cols], o1), j
            assert torch.equal(r[:, cols], r1), j
            assert torch.equal(d[:, cols], d1), j
        env.close()
    assert bool(torch.cat([d for _, _, d, _ in got]).any())  # auto-resets happened
    pop.close()


def test_group_networks_refuse_uneven_groups():
    cfg = dict(width=14, height=14, seed=1)
    P = _lib.mlp_param_count(14, 14, 50, 4, False)
    env = BatchedForestFire(48, obs_dtype="bits", auto_reset=True, **cfg)
    for M in (5, 3, 65):  # 48 % 5 != 0; 48 / 3 = 16 is fine; 65 networks are too many
        params = torch.zeros((M, P), device="cuda")
        if M == 3:
            env.set_policy_mlp_flat_dev(params, 50, False, [0.1] * M)
            continue
        with pytest.raises(_lib.WildfireError):
            env.set_policy_mlp_flat_dev(params, 50, False, [0.1] * M)
    with pytest.raises(_lib.WildfireError, match="multiple of 8"):
        env.set_policy_mlp_flat_dev(torch.zeros((12, P), device="cuda"), 50, False, [0.1] * 12)  # groups of 4
    with pytest.raises(ValueError):
        env.set_policy_mlp_flat_dev(torch.zeros((3, P + 1), device="cuda"), 50, False, [0.1] * 3)
    env.close()


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


def _state(ag):
    opt = [ag.optimizer.state[p] for p in ag.model.parameters()]
    return ([p.detach().cpu().numpy().tobytes() for p in ag.model.parameters()],
            [p.detach().cpu().numpy().tobytes() for p in ag.target.parameters()],
            [st["m"].cpu().numpy().tobytes() for st in opt], [st["v"].cpu().numpy().tobytes() for st in opt],
            [st["t"] for st in opt])


@pytest.mark.parametrize("name", ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"])
def test_learn_population_equals_each_agent_alone(name, tmp_path):
    """Three agents with different initial weights, demonstrations (one with none), alpha and target_update, trained
    together by learn_population, against each trained alone by learn_batched(seed, replay_seed=seed + j) on the envs
    j * 64 ... of the same Philox stream: byte-identical weights, target, Adam m, v and t, logs, eps schedule and step
    counts; each Logs/ file in the reference's format."""
    W, G, K, R, n_ep, seed = 10, 64, 16, 64, 300, 5
    settings = [dict(alpha=0.005, target_update=20), dict(alpha=0.002, target_update=7), dict(alpha=0.01, target_update=50)]
    demos = []
    for j, n_demo in enumerate((4, 0, 2)):
        torch.manual_seed(1000 + j)
        ag = getattr(A, name)(_Sim(W, W), verbose=False, device="cuda")
        ag.collect_memories_batched(n_demo, n_envs=256, k_steps=64, seed=j)
        demos.append((copy.deepcopy(ag.memory), ag.logs["init_memories"]))
    assert demos[0][1] > 0 and demos[1][1] == 0 and demos[2][1] > 0

    def make(j, out, **kw):
        torch.manual_seed(j)
        ag = getattr(A, name)(_Sim(W, W, **settings[j], **kw), verbose=False, device="cuda")
        ag.memory, ag.logs["init_memories"] = copy.deepcopy(demos[j][0]), demos[j][1]
        ag.out_dir = str(out)
        return ag

    pop = [make(j, tmp_path / "pop") for j in range(3)]
    steps = A.learn_population(pop, n_ep, envs_per_learner=G, k_steps=K, replays_per_launch=R, seed=seed)
    logs = sorted(os.listdir(tmp_path / "pop" / "Logs"))
    assert len(logs) == 3
    for f in logs:
        with open(tmp_path / "pop" / "Logs" / f) as fh:
            log = json.load(fh)
        assert set(log) >= {"best_reward", "total_rewards", "agent_pos", "agent_deaths", "maps", "init_memories",
                            "total_time", "n_episodes", "metadata"}
        assert log["n_episodes"] == n_ep and len(log["total_rewards"]) == n_ep and len(log["agent_deaths"]) == n_ep
    for j in range(3):
        solo = make(j, tmp_path / f"solo{j}", env_id_base=j * G)
        s = solo.learn_batched(n_ep, n_envs=G, k_steps=K, replays_per_launch=R, seed=seed, replay_seed=seed + j)
        assert steps[j] == s, j
        assert _state(pop[j]) == _state(solo), j
        for key in ("total_rewards", "agent_deaths", "init_memories", "n_episodes"):
            assert pop[j].logs[key] == solo.logs[key], (j, key)
        assert pop[j].eps_per_launch == solo.eps_per_launch and pop[j].episodes_before_launch == solo.episodes_before_launch
        assert pop[j]._until_sync == solo._until_sync
    assert len({tuple(a.logs["total_rewards"]) for a in pop}) == 3
