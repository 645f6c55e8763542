"""Populations without a GPU: argument checks of wf_replay_fit_many and wf_set_policy_mlp_nets_dev (no CPU fallback), the
ctypes wf_fit_learner against include/wildfire.h, and learn_population's validation of its agents."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from wildfire_control_python_b200 import _lib
from wildfire_control_python_b200 import agents as A
from wildfire_control_python_b200.compat import get_name
from wildfire_control_python_b200.constants import make_metadata

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


def fake(i):  # never dereferenced: every call below is refused before any device access
    return 0x10000 + 0x1000 * i


def shape(**kw):
    d = dict(width=14, height=14, hidden=50, n_actions=4, dueling=0, batch=32)
    d.update(kw)
    return _lib.WfMlpShape(**d)


def params(**kw):
    d = dict(gamma=0.99, lr=0.005, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipvalue=1.0, adam_t=0, target_every=20, phase=20)
    d.update(kw)
    return _lib.WfFitParams(**d)


def learner(j, hp=None, **ptrs):
    d = {name: fake(16 * j + i) for i, name in enumerate(("params", "target", "adam_m", "adam_v", "s_row", "sp_row", "action",
                                                         "next_action", "reward", "done", "loss"))}
    d.update(ptrs)
    return _lib.WfFitLearner(**d, hp=hp or params())


def fit_many(lib, learners, sh=None, n_replays=1, frames=fake(999), n_frames=100, n=None):
    arr = (_lib.WfFitLearner * max(1, len(learners)))(*learners)
    return lib.wf_replay_fit_many(None if sh is False else C.byref(sh or shape()), len(learners) if n is None else n,
                                  None if learners is None else arr, n_replays, frames, n_frames, None)


def test_fit_learner_layout_matches_the_header(tmp_path):
    """sizeof and every offsetof of wf_fit_learner (and wf_fit_params inside it) as a C compiler sees include/wildfire.h."""
    fields = [f for f, _ in _lib.WfFitLearner._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "wildfire.h"\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(wf_fit_learner));\n'
                   + "".join(f'  printf("%zu\\n", offsetof(wf_fit_learner, {f}));\n' for f in fields)
                   + '  printf("%zu\\n", sizeof(wf_fit_params));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(_lib.WfFitLearner)] + [getattr(_lib.WfFitLearner, f).offset for f in fields] + [C.sizeof(_lib.WfFitParams)]
    assert got == want
    assert C.sizeof(_lib.WfFitLearner) == 11 * 8 + 6 * 8 + 8 + 2 * 4 and _lib.WfFitLearner.hp.offset == 88


def test_replay_fit_many_refuses_learner_counts_and_null_arguments(lib):
    ok = [learner(j, next_action=None) for j in range(3)]
    for n in (0, 65, -1):
        assert fit_many(lib, ok, n=n) == _lib.WF_ERR_INVALID
    assert fit_many(lib, [learner(j) for j in range(65)]) == _lib.WF_ERR_INVALID
    assert fit_many(lib, ok, sh=False) == _lib.WF_ERR_INVALID
    assert fit_many(lib, ok, frames=None) == _lib.WF_ERR_INVALID
    assert lib.wf_replay_fit_many(C.byref(shape()), 1, None, 1, fake(999), 100, None) == _lib.WF_ERR_INVALID
    assert fit_many(lib, ok, n_replays=0) == _lib.WF_ERR_INVALID
    assert fit_many(lib, ok, n_frames=-1) == _lib.WF_ERR_INVALID
    for name in ("params", "target", "adam_m", "adam_v", "s_row", "sp_row", "action", "reward", "done"):
        bad = list(ok)
        bad[2] = learner(2, **{name: None})
        assert fit_many(lib, bad) == _lib.WF_ERR_INVALID, name
        assert b"learner 2" in lib.wf_last_error()


def test_replay_fit_many_refuses_misaligned_pointers(lib):
    ok = [learner(j) for j in range(2)]
    assert fit_many(lib, ok, frames=fake(999) + 2) == _lib.WF_ERR_INVALID
    for name in ("params", "target", "adam_m", "adam_v", "action", "next_action", "reward", "loss"):
        assert fit_many(lib, [ok[0], learner(1, **{name: fake(40) + 2})]) == _lib.WF_ERR_INVALID, name
        assert b"learner 1" in lib.wf_last_error()
    for name in ("s_row", "sp_row"):
        assert fit_many(lib, [learner(0, **{name: fake(40) + 4}), ok[1]]) == _lib.WF_ERR_INVALID, name


@pytest.mark.parametrize("bad", [
    dict(hidden=0), dict(hidden=65), dict(n_actions=0), dict(n_actions=9), dict(batch=0), dict(batch=257),
    dict(width=9, height=9), dict(width=33, height=14), dict(width=14, height=20), dict(dueling=2)])
def test_replay_fit_many_refuses_bad_shapes(lib, bad):
    assert fit_many(lib, [learner(j) for j in range(4)], sh=shape(**bad)) == _lib.WF_ERR_INVALID


@pytest.mark.parametrize("bad", [dict(target_every=0), dict(phase=0), dict(phase=21), dict(adam_t=-1), dict(clipvalue=0.0),
                                 dict(beta_1=1.0), dict(beta_2=-0.1), dict(epsilon=-1.0), dict(lr=float("nan")),
                                 dict(gamma=float("inf"))])
def test_replay_fit_many_refuses_bad_hyper_parameters_of_any_learner(lib, bad):
    for j in (0, 3):
        ls = [learner(i, hp=params(**bad) if i == j else None) for i in range(4)]
        assert fit_many(lib, ls) == _lib.WF_ERR_INVALID
        assert f"learner {j}".encode() in lib.wf_last_error()


def test_replay_fit_many_has_no_cpu_fallback(lib):
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the no-device error cannot be provoked")
    ls = [learner(j, next_action=None if j % 2 else fake(16 * j + 7)) for j in range(64)]
    assert fit_many(lib, ls) == _lib.WF_ERR_CUDA and b"no CPU fallback" in lib.wf_last_error()


def nets(lib, env=fake(900), sh=None, n_nets=2, p=fake(901), eps=(0.1, 0.2)):
    e = None if eps is None else (C.c_double * max(1, len(eps)))(*eps)
    return lib.wf_set_policy_mlp_nets_dev(env, None if sh is False else C.byref(sh or shape()), n_nets, p, e, None)


def test_set_policy_mlp_nets_dev_refuses_bad_arguments(lib):
    """Everything that can be refused without a handle (group sizes need one: tests/test_population_gpu.py)."""
    assert nets(lib, env=None) == _lib.WF_ERR_INVALID
    assert nets(lib, sh=False) == _lib.WF_ERR_INVALID
    assert nets(lib, p=None) == _lib.WF_ERR_INVALID
    assert nets(lib, eps=None) == _lib.WF_ERR_INVALID
    for n in (0, 65, -3):
        assert nets(lib, n_nets=n, eps=[0.1] * 65) == _lib.WF_ERR_INVALID
    assert b"n_nets" in lib.wf_last_error()
    for bad in (dict(hidden=0), dict(hidden=65), dict(n_actions=0), dict(n_actions=9), dict(dueling=2),
                dict(width=9, height=9), dict(width=33, height=33), dict(width=14, height=20)):
        assert nets(lib, sh=shape(**bad)) == _lib.WF_ERR_INVALID, bad
    for eps in ((0.1, -0.01), (1.5, 0.1), (0.1, float("nan"))):
        assert nets(lib, eps=eps) == _lib.WF_ERR_INVALID, eps
    assert nets(lib, p=fake(901) + 2) == _lib.WF_ERR_INVALID


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


def _agent(cls="DQN", W=10, H=10, **kw):
    return getattr(A, cls)(_Sim(W, H, **kw), verbose=False, device="cpu")


@pytest.mark.parametrize("case", ["classes", "metadata", "memory_size", "batch_size", "shape", "count", "none", "grid",
                                  "group"])
def test_learn_population_validates_its_agents(case):
    ags = [_agent(), _agent(alpha=0.001, gamma=0.9, target_update=5, max_eps=0.5, min_eps=0.1, eps_decay_rate=0.01)]
    kw = {}
    if case == "classes":
        ags.append(_agent("DQN_SARSA"))
    elif case == "metadata":
        ags.append(_agent(a_speed=2))
    elif case == "memory_size":
        ags.append(_agent(memory_size=1000))
    elif case == "batch_size":
        ags.append(_agent(batch_size=64))
    elif case == "shape":
        ags.append(_agent(n_actions=5, allow_dig_toggle=True))
        ags[-1].METADATA.update({k: v for k, v in ags[0].METADATA.items() if k in ("n_actions", "allow_dig_toggle")})
    elif case == "count":
        ags = [_agent() for _ in range(65)]
    elif case == "none":
        ags = []
    elif case == "grid":
        ags = [_agent(W=40, H=40) for _ in range(2)]
    elif case == "group":
        kw = dict(envs_per_learner=12)
    with pytest.raises(ValueError):
        A.learn_population(ags, 10, **kw)


def test_learn_population_has_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the agents would live on it")
    ags = [_agent(), _agent(alpha=0.01)]
    with pytest.raises(_lib.WildfireError, match="no CPU fallback"):
        A.learn_population(ags, 10)
