"""wf_replay_fit_large without a GPU: its argument checks (the shape limits of wf_replay_fit without the 32x32 bound, the
2^31 - 1-float bound of the flat buffer, pointers and hyper-parameters) and the no-CPU-fallback error."""
import ctypes as C
import math

import pytest
import torch

from wildfire_control_python_b200 import _lib

FAKE = [C.c_void_p(0x10000 + 0x1000 * i) for i in range(12)]  # never dereferenced: every call below is refused


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


def shape(**kw):
    d = dict(width=40, height=40, hidden=50, n_actions=4, dueling=0, batch=32)
    d.update(kw)
    return _lib.WfMlpShape(**d)


def params(**kw):
    d = dict(gamma=0.99, lr=0.005, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipvalue=1.0, adam_t=0, target_every=20, phase=20)
    d.update(kw)
    return _lib.WfFitParams(**d)


def fit(lib, sh=None, hp=None, n_replays=1, ptrs=None, n_frames=100):
    p = list(FAKE) if ptrs is None else ptrs
    return lib.wf_replay_fit_large(None if sh is False else C.byref(sh or shape()),
                                   None if hp is False else C.byref(hp or params()),
                                   n_replays, p[0], p[1], p[2], p[3], p[4], n_frames, p[5], p[6], p[7], p[8], p[9], p[10],
                                   p[11], None)


def no_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the no-device error cannot be provoked with fake pointers")


@pytest.mark.parametrize("bad", [
    dict(hidden=0), dict(hidden=65), dict(n_actions=0), dict(n_actions=9), dict(batch=0), dict(batch=257), dict(dueling=2),
    dict(width=9, height=9), dict(width=40, height=9), dict(width=40, height=50), dict(width=14, height=20)])
def test_replay_fit_large_refuses_bad_shapes(lib, bad):
    assert fit(lib, sh=shape(**bad)) == _lib.WF_ERR_INVALID


@pytest.mark.parametrize("sh,ok", [
    # hidden * (n_in + 1 + A) + A floats: 2^31 - 1 is the largest flat buffer
    (dict(width=4096, height=4096, hidden=14, n_actions=4), True),     # 14 * (50331648 + 5) + 4 = 704643146
    (dict(width=4096, height=4096, hidden=43, n_actions=4), False),    # 43 * (50331648 + 5) + 4 = 2164261083
    (dict(width=4096, height=4096, hidden=22, n_actions=4, dueling=1), False),  # 2 * 22 * 50331648 + ... > 2^31
    (dict(width=100000, height=100000, hidden=1, n_actions=1), False),  # n_in = 3e10 alone overflows 32 bits
])
def test_replay_fit_large_bounds_the_flat_buffer(lib, sh, ok):
    if ok:
        no_cuda()
        assert fit(lib, sh=shape(**sh)) == _lib.WF_ERR_CUDA
    else:
        assert fit(lib, sh=shape(**sh)) == _lib.WF_ERR_INVALID
        assert b"2^31 - 1" in lib.wf_last_error()


def test_flat_buffer_bound_matches_mlp_param_count():
    assert _lib.mlp_param_count(4096, 4096, 14, 4, False) <= 2**31 - 1
    assert _lib.mlp_param_count(4096, 4096, 43, 4, False) > 2**31 - 1
    assert _lib.mlp_param_count(4096, 4096, 22, 4, True) > 2**31 - 1


@pytest.mark.parametrize("bad", [dict(target_every=0), dict(phase=0), dict(phase=21), dict(adam_t=-1), dict(clipvalue=0.0),
                                 dict(beta_1=1.0), dict(beta_2=-0.1), dict(epsilon=-1.0), dict(lr=math.nan),
                                 dict(gamma=math.inf)])
def test_replay_fit_large_refuses_bad_hyper_parameters(lib, bad):
    assert fit(lib, hp=params(**bad)) == _lib.WF_ERR_INVALID


def test_replay_fit_large_refuses_null_and_misaligned_pointers(lib):
    assert fit(lib, sh=False) == _lib.WF_ERR_INVALID
    assert fit(lib, hp=False) == _lib.WF_ERR_INVALID
    for i in range(12):
        if i in (8, 11):  # next_action and loss may be NULL
            continue
        p = list(FAKE)
        p[i] = None
        assert fit(lib, ptrs=p) == _lib.WF_ERR_INVALID, i
    for i in range(12):
        p = list(FAKE)
        p[i] = C.c_void_p(FAKE[i].value + (4 if i in (5, 6) else 2))  # rows: 8-byte aligned, the rest 4-byte
        if i == 10:  # done (uint8) needs no alignment
            continue
        assert fit(lib, ptrs=p) == _lib.WF_ERR_INVALID, i
    assert fit(lib, n_replays=0) == _lib.WF_ERR_INVALID
    assert fit(lib, n_frames=-1) == _lib.WF_ERR_INVALID


@pytest.mark.parametrize("W,H", [(40, 40), (100, 70), (256, 256), (14, 14), (32, 32)])
def test_replay_fit_large_accepts_any_grid_up_to_the_device(lib, W, H):
    """Grids past 32x32 (and the small ones, for comparisons with wf_replay_fit) pass every check; without a device the
    call then fails with the no-CPU-fallback error, never with WF_ERR_INVALID."""
    no_cuda()
    p = list(FAKE)
    p[8] = None  # the off-policy form
    assert fit(lib, sh=shape(width=W, height=H), ptrs=p) == _lib.WF_ERR_CUDA
    assert b"no CPU fallback" in lib.wf_last_error()
    assert fit(lib, sh=shape(width=W, height=H, dueling=1, hidden=64, n_actions=8, batch=256)) == _lib.WF_ERR_CUDA
