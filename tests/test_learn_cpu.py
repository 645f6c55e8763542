"""Batched learning without a GPU: argument checks of wf_replay_fit and wf_set_policy_mlp_dev (no CPU fallback), pack_obs
against the NumPy reference of the WF_OBS_BITS layout, and wf_replay_fit's flat parameter layout against
torch.nn.utils.parameters_to_vector."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from wildfire_control_python_b200 import _lib, pack_obs
from wildfire_control_python_b200.agents import _DuelNet, _QNet

from tests.test_obs_bits_cpu import np_pack


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


FAKE = [C.c_void_p(0x10000 + 0x1000 * i) for i in range(12)]  # never dereferenced: every call below is refused


def shape(**kw):
    d = dict(width=14, height=14, hidden=50, n_actions=4, dueling=0, batch=32)
    d.update(kw)
    return _lib.WfMlpShape(**d)


def params(**kw):
    d = dict(gamma=0.99, lr=0.005, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipvalue=1.0, adam_t=0, target_every=20, phase=20)
    d.update(kw)
    return _lib.WfFitParams(**d)


def fit(lib, sh=None, hp=None, n_replays=1, ptrs=None, n_frames=100):
    p = list(FAKE) if ptrs is None else ptrs
    return lib.wf_replay_fit(None if sh is False else C.byref(sh or shape()), None if hp is False else C.byref(hp or params()),
                             n_replays, p[0], p[1], p[2], p[3], p[4], n_frames, p[5], p[6], p[7], p[8], p[9], p[10], p[11],
                             None)


@pytest.mark.parametrize("bad", [
    dict(hidden=0), dict(hidden=65), dict(n_actions=0), dict(n_actions=9), dict(batch=0), dict(batch=257),
    dict(width=9, height=9), dict(width=33, height=14), dict(width=14, height=20), dict(dueling=2)])
def test_replay_fit_refuses_bad_shapes(lib, bad):
    assert fit(lib, sh=shape(**bad)) == _lib.WF_ERR_INVALID


@pytest.mark.parametrize("bad", [dict(target_every=0), dict(phase=0), dict(phase=21), dict(adam_t=-1), dict(clipvalue=0.0),
                                 dict(beta_1=1.0), dict(beta_2=-0.1), dict(epsilon=-1.0), dict(lr=math.nan)])
def test_replay_fit_refuses_bad_hyper_parameters(lib, bad):
    assert fit(lib, hp=params(**bad)) == _lib.WF_ERR_INVALID


def test_replay_fit_refuses_null_pointers_and_counts(lib):
    assert fit(lib, sh=False) == _lib.WF_ERR_INVALID
    assert fit(lib, hp=False) == _lib.WF_ERR_INVALID
    for i in range(11):
        if i == 8:  # next_action may be NULL (off-policy learners)
            continue
        p = list(FAKE)
        p[i] = None
        assert fit(lib, ptrs=p) == _lib.WF_ERR_INVALID, i
    assert fit(lib, n_replays=0) == _lib.WF_ERR_INVALID
    assert fit(lib, n_frames=-1) == _lib.WF_ERR_INVALID
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the no-device error cannot be provoked")
    p = list(FAKE)
    p[8] = None  # the off-policy form passes every check up to the device
    assert fit(lib, ptrs=p) == _lib.WF_ERR_CUDA and b"no CPU fallback" in lib.wf_last_error()


def test_set_policy_mlp_dev_refuses_null_arguments(lib):
    f = lib.wf_set_policy_mlp_dev
    assert f(None, FAKE[0], FAKE[1], FAKE[2], FAKE[3], 50, 0.1, None) == _lib.WF_ERR_INVALID
    assert f(FAKE[4], None, FAKE[1], FAKE[2], FAKE[3], 50, 0.1, None) == _lib.WF_ERR_INVALID
    assert f(FAKE[4], FAKE[0], FAKE[1], FAKE[2], None, 50, 0.1, None) == _lib.WF_ERR_INVALID


@pytest.mark.parametrize("W,H", [(10, 10), (11, 10), (14, 14), (17, 16), (32, 32), (100, 70)])
def test_pack_obs_matches_the_numpy_reference(W, H):
    rng = np.random.default_rng(W * 100 + H)
    obs = rng.integers(0, 2, size=(2, 3, W, H, 3), dtype=np.uint8)
    got = pack_obs(torch.as_tensor(obs))
    assert got.dtype == torch.int32 and tuple(got.shape) == (2, 3, _lib.obs_bits_words(W, H))
    assert np.array_equal(got.numpy().view(np.uint32), np_pack(obs))
    assert np.array_equal(pack_obs(torch.as_tensor(obs[0, 0]).float()).numpy().view(np.uint32), np_pack(obs[0, 0]))


@pytest.mark.parametrize("net,dueling", [(_QNet, 0), (_DuelNet, 1)])
@pytest.mark.parametrize("W,H,A", [(10, 10, 4), (14, 14, 5), (32, 20, 6)])
def test_flat_layout_is_parameters_to_vector(net, dueling, W, H, A):
    """include/wildfire.h's layout: dense_1.weight [hidden][n_in] | dense_1.bias | dense_2.weight [A][hidden] |
    dense_2.bias, then (dueling) dense_3.* and dense_4.* -- exactly parameters_to_vector(model.parameters())."""
    n_in, hid = W * H * 3, 50
    m = net(n_in, A)
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn_like(p))
    flat = torch.nn.utils.parameters_to_vector(m.parameters())
    assert flat.numel() == _lib.mlp_param_count(W, H, hid, A, dueling)
    off = 0
    names = ["dense_1", "dense_2"] + (["dense_3", "dense_4"] if dueling else [])
    for name in names:
        layer = getattr(m, name)
        for t in (layer.weight, layer.bias):
            assert torch.equal(flat[off:off + t.numel()].view_as(t), t.detach())
            off += t.numel()
    assert off == flat.numel()
