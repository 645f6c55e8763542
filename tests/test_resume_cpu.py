"""Checkpoints of learn_batched and learn_population without a GPU: the time_limit / checkpoint pairing, the refusal of a
checkpoint written by another run (one case per fingerprint field, through both entry points), the atomic write, and the
no-CPU-fallback error with the new arguments."""
import os
import re

import pytest
import torch
from torch import nn

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


def _agent(cls="DQN", demos=0, **kw):
    ag = getattr(A, cls)(_Sim(10, 10, **kw), verbose=False, device="cpu")
    if demos:
        ag.memory = ag._new_memory(None)
        zero = torch.zeros(ag.obs_shape, dtype=torch.uint8)
        for _ in range(demos):
            ag.memory.append(zero, 0, -1.0, zero, False)
    return ag


def _widen(ag):
    """The same METADATA, a network with 64 hidden units instead of 50."""
    ag.model.dense_1, ag.model.dense_2 = nn.Linear(300, 64), nn.Linear(64, 4)


BATCHED = dict(n_episodes=50, n_envs=64, k_steps=16, replays_per_launch=16, batch_size=32, seed=3, replay_seed=3)
POPULATION = dict(n_episodes=50, envs_per_learner=64, k_steps=16, replays_per_launch=16, batch_size=32, seed=3)


def _write(path, entry, agents, args):
    A._RunCheckpoint(path, A._run_fingerprint(entry, agents, **args)).save({"marker": 1})


def _refused(where, call):
    with pytest.raises(ValueError, match=re.escape(f"another run: {where} is")):
        call()


@pytest.mark.parametrize("field", ["entry", "agent_class", "network", "METADATA", "demonstrations", "n_episodes", "n_envs",
                                   "k_steps", "replays_per_launch", "batch_size", "seed", "replay_seed"])
def test_learn_batched_refuses_a_checkpoint_of_another_run(tmp_path, field):
    path = tmp_path / "run.ckpt"
    _write(path, "learn_population" if field == "entry" else "learn_batched", [_agent(demos=3)], BATCHED)
    before = path.read_bytes()
    ag, kw, where = _agent(demos=3), dict(BATCHED), field
    if field == "agent_class":
        ag = _agent("DQN_SARSA", demos=3)
    elif field == "network":
        _widen(ag)
        where = "network[0][0]"  # dense_1.weight: [50, 300] there, [64, 300] here
    elif field == "METADATA":
        ag, where = _agent(demos=3, alpha=0.001), "METADATA[0]['alpha']"
    elif field == "demonstrations":
        ag, where = _agent(demos=4), "demonstrations[0]"
    elif field in kw:
        kw[field] += 1
    n = kw.pop("n_episodes")
    _refused(where, lambda: ag.learn_batched(n, checkpoint=path, **kw))
    _refused(where, lambda: ag.learn_batched(n, checkpoint=path, time_limit=10.0, **kw))
    assert path.read_bytes() == before  # a refused checkpoint is left as it was


def test_learn_batched_refuses_a_checkpoint_of_the_per_agent_layout(tmp_path):
    """A checkpoint in the layout learn_batched wrote before it shared learn_population's (one agent's modules under
    ``agent``, one ``replay_generator``), whose fingerprint has no ``layout``: refused with ValueError naming that field
    before anything is restored, and left as it was."""
    path = tmp_path / "run.ckpt"
    ag = _agent(demos=3)
    fp = A._run_fingerprint("learn_batched", [ag], **BATCHED)
    del fp["layout"]
    cpu = lambda m: {k: v.cpu() for k, v in m.state_dict().items()}  # noqa: E731
    A._RunCheckpoint(path, fp).save(dict(
        env={"scalars": torch.zeros((64, 8), dtype=torch.int32)}, ring={"steps": 16},
        replay_generator=torch.Generator().manual_seed(3).get_state(),
        agent=dict(model=cpu(ag.model), target=cpu(ag.target), adam_t=0, adam_m=[], adam_v=[], until_sync=20,
                   logs="{}", eps=1.0, eps_per_launch=[1.0], episodes_before_launch=[0]),
        carry=torch.zeros(64, dtype=torch.float64), done_eps=0, rewards=[], deaths=[], elapsed=0.5))
    before = path.read_bytes()
    kw = dict(BATCHED)
    n = kw.pop("n_episodes")
    _refused("layout", lambda: _agent(demos=3).learn_batched(n, checkpoint=path, **kw))
    assert path.read_bytes() == before


def _population(n=3, **kw):
    settings = [dict(alpha=0.005, target_update=20), dict(alpha=0.002, target_update=7), dict(alpha=0.01, target_update=50)]
    return [_agent(demos=d, **settings[j], **kw) for j, d in zip(range(n), (4, 0, 2))]


@pytest.mark.parametrize("field", ["entry", "agent_class", "network", "agents", "METADATA", "demonstrations", "n_episodes",
                                   "envs_per_learner", "k_steps", "replays_per_launch", "batch_size", "seed"])
def test_learn_population_refuses_a_checkpoint_of_another_run(tmp_path, field):
    path = tmp_path / "run.ckpt"
    _write(path, "learn_batched" if field == "entry" else "learn_population", _population(), POPULATION)
    ags, kw, where = _population(), dict(POPULATION), field
    if field == "agent_class":
        ags = [_agent("DQN_DUEL", alpha=a.alpha, target_update=a.target_update_freq) for a in ags]
    elif field == "network":
        for a in ags:
            _widen(a)
        where = "network[0][0]"
    elif field == "agents":
        ags = ags[:2]
    elif field == "METADATA":
        ags[1] = _agent(alpha=0.003, target_update=7)
        where = "METADATA[1]['alpha']"
    elif field == "demonstrations":
        ags[1] = _agent(demos=5, alpha=0.002, target_update=7)
        where = "demonstrations[1]"
    elif field == "envs_per_learner":
        kw[field] += 8
    elif field in kw:
        kw[field] += 1
    n = kw.pop("n_episodes")
    _refused(where, lambda: A.learn_population(ags, n, checkpoint=path, **kw))
    assert os.path.exists(path)


def test_time_limit_needs_a_checkpoint(tmp_path):
    with pytest.raises(ValueError, match="time_limit needs a checkpoint"):
        _agent().learn_batched(10, time_limit=60)
    with pytest.raises(ValueError, match="time_limit needs a checkpoint"):
        A.learn_population(_population(2), 10, time_limit=0)
    assert os.listdir(tmp_path) == []


def test_a_checkpoint_of_the_same_run_loads(tmp_path):
    """The fingerprint survives the file (METADATA holds tuples, e.g. the wind): the same run's checkpoint is accepted, its
    state comes back, and a missing file means a fresh start."""
    path = tmp_path / "run.ckpt"
    ags = _population()
    fp = lambda: A._run_fingerprint("learn_population", ags, **POPULATION)  # noqa: E731
    assert A._RunCheckpoint(path, fp()).load() is None
    A._RunCheckpoint(path, fp()).save({"w": torch.arange(4.0), "rewards": [[1.5, -3.0]], "finished": [True, False]})
    got = A._RunCheckpoint(path, fp()).load()
    assert torch.equal(got["w"], torch.arange(4.0)) and got["rewards"] == [[1.5, -3.0]] and got["finished"] == [True, False]
    assert torch.load(path, weights_only=True)["state"]["rewards"] == [[1.5, -3.0]]
    A._RunCheckpoint(path, fp()).remove()
    assert not path.exists()


def test_checkpoint_write_is_atomic(tmp_path, monkeypatch):
    """A write that fails midway leaves the previous checkpoint intact and no temporary file; a write that succeeds is
    flushed to disk (fsync) before it replaces the old file."""
    path = tmp_path / "run.ckpt"
    ck = A._RunCheckpoint(path, {"entry": "learn_batched"})
    ck.save({"launch": 1, "w": torch.arange(5)})
    before = path.read_bytes()

    def torn_write(obj, f, *args, **kwargs):
        f.write(before[: len(before) // 2])
        raise OSError(28, "No space left on device")

    with monkeypatch.context() as m:
        m.setattr(torch, "save", torn_write)
        with pytest.raises(OSError, match="No space"):
            ck.save({"launch": 2, "w": torch.arange(6)})
    assert path.read_bytes() == before
    assert os.listdir(tmp_path) == ["run.ckpt"]
    assert ck.load()["launch"] == 1

    calls = []
    real_fsync, real_replace = os.fsync, os.replace
    monkeypatch.setattr(os, "fsync", lambda fd: (calls.append("fsync"), real_fsync(fd))[1])
    monkeypatch.setattr(os, "replace", lambda a, b: (calls.append("replace"), real_replace(a, b))[1])
    ck.save({"launch": 3, "w": torch.arange(7)})
    assert calls[:2] == ["fsync", "replace"]
    assert ck.load()["launch"] == 3 and os.listdir(tmp_path) == ["run.ckpt"]


def test_no_cpu_fallback_with_a_checkpoint(tmp_path):
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the agents would live on it")
    path = tmp_path / "run.ckpt"
    with pytest.raises(_lib.WildfireError, match="no CPU fallback"):
        _agent().learn_batched(10, n_envs=64, checkpoint=path, time_limit=0)
    with pytest.raises(_lib.WildfireError, match="no CPU fallback"):
        A.learn_population(_population(), 10, checkpoint=path, time_limit=0)
    _write(path, "learn_batched", [_agent(demos=3)], BATCHED)  # a matching checkpoint is accepted, then the device is needed
    kw = dict(BATCHED)
    with pytest.raises(_lib.WildfireError, match="no CPU fallback"):
        _agent(demos=3).learn_batched(kw.pop("n_episodes"), checkpoint=path, **kw)
    assert os.listdir(tmp_path) == ["run.ckpt"]
