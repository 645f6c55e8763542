"""WF_OBS_BITS without a GPU: the header and the binding agree on the format's constants, obs_bits_words, the NumPy
reference the GPU tests unpack with, and the argument checks of wf_unpack_obs_bits (which has no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from wildfire_control_python_b200 import _lib, obs_bits_words

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


def np_pack(obs_u8):
    """[..., W, H, 3] 0/1 uint8 -> [..., words] uint32 in the WF_OBS_BITS layout (include/wildfire.h)."""
    lead, (W, H) = obs_u8.shape[:-3], obs_u8.shape[-3:-1]
    flat = obs_u8.reshape(*lead, W * H * 3)
    pad = obs_bits_words(W, H) * 32 - W * H * 3
    flat = np.concatenate([flat, np.zeros((*lead, pad), np.uint8)], axis=-1)
    return np.packbits(flat, axis=-1, bitorder="little").view(np.uint32)


def np_unpack(bits, W, H):
    """The header's reference: np.unpackbits(a.view(np.uint8), axis=-1, bitorder="little")[..., :W*H*3]."""
    u = np.unpackbits(np.ascontiguousarray(bits).view(np.uint8), axis=-1, bitorder="little")
    return u[..., : W * H * 3].reshape(*bits.shape[:-1], W, H, 3), u[..., W * H * 3:]


def test_header_constant_and_symbol_match_the_binding():
    text = open(os.path.join(ROOT, "include", "wildfire.h")).read()
    m = re.search(r"WF_OBS_BITS\s*=\s*(\d+)", text)
    assert m and int(m.group(1)) == _lib.WF_OBS_BITS == 3
    assert re.search(r"\bint\s+wf_unpack_obs_bits\s*\(", text)
    assert "wf_unpack_obs_bits" in _lib.EXPORTED_SYMBOLS


@pytest.mark.parametrize("W,H,words", [(10, 10, 10), (14, 14, 19), (32, 32, 96), (100, 70, 657), (256, 256, 6144),
                                       (1024, 1024, 98304)])
def test_obs_bits_words(W, H, words):
    assert obs_bits_words(W, H) == words == -(-W * H * 3 // 32)


@pytest.mark.parametrize("W,H", [(10, 10), (14, 14), (17, 16), (32, 32), (100, 70)])
def test_numpy_reference_round_trips_with_zero_padding(W, H):
    rng = np.random.default_rng(W * 1000 + H)
    obs = rng.integers(0, 2, size=(5, W, H, 3), dtype=np.uint8)
    bits = np_pack(obs)
    assert bits.dtype == np.uint32 and bits.shape == (5, obs_bits_words(W, H))
    # element k = (x*H + y)*3 + c is bit k % 32 of word k // 32
    for n, x, y, c in [(0, 0, 0, 0), (1, W - 1, H - 1, 2), (4, W // 2, H // 3, 1)]:
        k = (x * H + y) * 3 + c
        assert (int(bits[n, k // 32]) >> (k % 32)) & 1 == obs[n, x, y, c]
    back, pad = np_unpack(bits, W, H)
    assert np.array_equal(back, obs)
    assert not pad.any()
    # random words with the padding cleared survive the trip the other way too
    words = rng.integers(0, 2**32, size=(3, obs_bits_words(W, H)), dtype=np.uint64).astype(np.uint32)
    tail = (W * H * 3) % 32
    if tail:
        words[:, -1] &= np.uint32((1 << tail) - 1)
    assert np.array_equal(np_pack(np_unpack(words, W, H)[0]), words)


def test_unpack_validates_arguments_and_has_no_cpu_fallback(lib):
    f = lib.wf_unpack_obs_bits
    fake_bits, fake_out = C.c_void_p(0x10000), C.c_void_p(0x20000)  # never dereferenced: every call below is refused
    assert f(fake_bits, 4, None, 4, 10, 10, fake_out, 7, None) == _lib.WF_ERR_INVALID
    assert f(fake_bits, 4, None, 4, 10, 10, fake_out, _lib.WF_OBS_BITS, None) == _lib.WF_ERR_INVALID
    assert f(fake_bits, 4, None, 4, 0, 10, fake_out, _lib.WF_OBS_U8, None) == _lib.WF_ERR_INVALID
    assert f(fake_bits, 4, None, 4, 10, 0, fake_out, _lib.WF_OBS_U8, None) == _lib.WF_ERR_INVALID
    assert f(fake_bits, 4, None, -1, 10, 10, fake_out, _lib.WF_OBS_U8, None) == _lib.WF_ERR_INVALID
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the no-device error cannot be provoked")
    rc = f(fake_bits, 4, None, 4, 10, 10, fake_out, _lib.WF_OBS_F32, None)
    assert rc == _lib.WF_ERR_CUDA and b"no CPU fallback" in lib.wf_last_error()
