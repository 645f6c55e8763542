"""Resumed training runs on the GPU: learn_batched and learn_population stopped after every launch (time_limit=0) and
resumed from freshly built agents, each call from its checkpoint file, against one uninterrupted call -- byte for byte:
weights, target, Adam m, v and t, _until_sync, the logged returns, deaths, init_memories and n_episodes, the eps schedule
and the returned step counts.  And a resume whose replay generator is not restored diverges, so the comparison sees it."""
import copy

import pytest
import torch

from tests.test_learn_gpu import _agent
from tests.test_population_gpu import _state
from wildfire_control_python_b200 import agents as A

pytestmark = pytest.mark.gpu

NAMES = ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"]
LOGGED = ("total_rewards", "agent_deaths", "init_memories", "n_episodes")


def _result(ag, steps):
    return dict(state=_state(ag), until_sync=ag._until_sync, logs={k: ag.logs[k] for k in LOGGED},
                eps_per_launch=list(ag.eps_per_launch), episodes_before_launch=list(ag.episodes_before_launch), steps=steps)


def _demos(name, W, n_demo, seed=2):
    ag = _agent(name, W, W, seed=1)
    ag.collect_memories_batched(n_demo, n_envs=64 if W > 32 else 256, k_steps=64, seed=seed)
    return copy.deepcopy(ag.memory), ag.logs["init_memories"]


def _resume_until_done(make, train, path):
    """Call ``train(make(i))`` with fresh agents until a call completes; returns (agents, result, number of stops)."""
    stops = 0
    while True:
        ag = make(stops)
        out = train(ag)
        if out is not None:
            return ag, out, stops
        assert path.exists()
        stops += 1


def _learn_batched_resumed_equals_whole(name, W, n_ep, kw, tmp_path):
    memory, init = _demos(name, W, 20 if W <= 32 else 4)

    def make(i, out):
        ag = _agent(name, W, W, seed=1 if i == 0 else 100 + i)  # later segments start from other weights: all overwritten
        ag.memory, ag.logs["init_memories"], ag.out_dir = copy.deepcopy(memory), init, str(out)
        return ag

    whole = make(0, tmp_path / "whole")
    want = _result(whole, whole.learn_batched(n_ep, **kw))
    path = tmp_path / "run.ckpt"
    ag, steps, stops = _resume_until_done(lambda i: make(i, tmp_path / "resumed"),
                                          lambda a: a.learn_batched(n_ep, checkpoint=path, time_limit=0, **kw), path)
    assert stops == len(whole.eps_per_launch) - 1  # time_limit=0: one launch per call
    assert not path.exists() and len(list((tmp_path / "resumed" / "Logs").iterdir())) == 1
    assert _result(ag, steps) == want
    return whole, stops


@pytest.mark.parametrize("name", NAMES)
def test_learn_batched_resumed_after_every_launch(name, tmp_path):
    """10x10 with demonstrations, 256 envs: stopped after every launch, each segment a fresh agent."""
    whole, stops = _learn_batched_resumed_equals_whole(name, 10, 300, dict(n_envs=256, k_steps=16, seed=3), tmp_path)
    assert stops >= 3


@pytest.mark.parametrize("name", ["DQN", "DQN_BOTH"])
def test_learn_batched_on_a_tile_grid_resumed_after_every_launch(name, tmp_path):
    """40x40 (tile kernel, wf_replay_fit_large): at least three stops, and episodes ended (auto-resets) inside launches
    that were followed by a stop."""
    whole, stops = _learn_batched_resumed_equals_whole(name, 40, 40, dict(n_envs=64, k_steps=8, replays_per_launch=4, seed=3),
                                                       tmp_path)
    assert stops >= 3 and whole.episodes_before_launch[stops] > 0


@pytest.mark.parametrize("name", NAMES)
def test_learn_population_resumed_after_every_launch(name, tmp_path):
    """Three agents of different alpha, target_update and demonstration counts (as in
    test_population_gpu.test_learn_population_equals_each_agent_alone), stopped after every launch, among them stops
    after some learners have finished and before the others have."""
    W, G, K, R, n_ep, seed = 10, 64, 16, 64, 300, 5
    settings = [dict(alpha=0.005, target_update=20), dict(alpha=0.002, target_update=7), dict(alpha=0.01, target_update=50)]
    demos = []
    for j, n_demo in enumerate((4, 0, 2)):
        ag = _agent(name, W, W, seed=1000 + j)
        ag.collect_memories_batched(n_demo, n_envs=256, k_steps=64, seed=j)
        demos.append((copy.deepcopy(ag.memory), ag.logs["init_memories"]))

    def make(i, out):
        pop = []
        for j in range(3):
            pop.append(_agent(name, W, W, seed=j if i == 0 else 100 * i + j, **settings[j]))
            pop[-1].memory, pop[-1].logs["init_memories"] = copy.deepcopy(demos[j][0]), demos[j][1]
            pop[-1].out_dir = str(out)
        return pop

    kw = dict(envs_per_learner=G, k_steps=K, replays_per_launch=R, seed=seed)
    whole = make(0, tmp_path / "whole")
    steps = A.learn_population(whole, n_ep, **kw)
    want = [_result(a, s) for a, s in zip(whole, steps)]
    path = tmp_path / "run.ckpt"
    finished = []

    def train(pop):
        out = A.learn_population(pop, n_ep, checkpoint=path, time_limit=0, **kw)
        if out is None:
            finished.append(torch.load(path, weights_only=True)["state"]["finished"])
        return out

    pop, got, stops = _resume_until_done(lambda i: make(i, tmp_path / "resumed"), train, path)
    assert stops == max(len(a.eps_per_launch) for a in whole) - 1
    assert any(0 < sum(f) < 3 for f in finished), finished
    assert not path.exists() and len(list((tmp_path / "resumed" / "Logs").iterdir())) == 3
    for j in range(3):
        assert _result(pop[j], got[j]) == want[j], j


def test_a_resume_with_a_freshly_seeded_replay_generator_diverges(tmp_path):
    """The same stop and resume with the checkpoint's replay generator (learner 0's of the stacked layout) replaced by a
    freshly seeded one: the replays draw other minibatches, and the weights and logs come out different."""
    memory, init = _demos("DQN", 10, 20)

    def make(out):
        ag = _agent("DQN", 10, 10, seed=1)
        ag.memory, ag.logs["init_memories"], ag.out_dir = copy.deepcopy(memory), init, str(out)
        return ag

    kw = dict(n_envs=256, k_steps=16, seed=3)
    whole = make(tmp_path / "whole")
    want = _result(whole, whole.learn_batched(300, **kw))
    for restore in (True, False):
        path = tmp_path / f"run_{restore}.ckpt"
        assert make(tmp_path / "resumed").learn_batched(300, checkpoint=path, time_limit=0, **kw) is None
        if not restore:
            ck = torch.load(path, weights_only=True)
            assert ck["state"]["adam_t"][0] > 0  # the first launch replayed: the generator has moved
            ck["state"]["replay_generators"][0] = torch.Generator(device="cuda").manual_seed(3).get_state()
            torch.save(ck, path)
        ag = make(tmp_path / "resumed")
        got = _result(ag, ag.learn_batched(300, checkpoint=path, **kw))
        if restore:
            assert got == want
        else:
            assert got["state"][0] != want["state"][0] and got["logs"]["total_rewards"] != want["logs"]["total_rewards"]
