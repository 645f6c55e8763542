"""Final-state records without a GPU: the C ABI prototype and the record layout constants against the Python binding, and
FinalStates' parsing, types() and render() against a NumPy statement of the layout (include/wildfire.h)."""
import os
import re

import numpy as np
import pytest
import torch

from wildfire_control_python_b200 import _lib
from wildfire_control_python_b200.batched import FinalStates
from wildfire_control_python_b200.constants import ascii_of_type

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "wildfire.h")).read(), flags=re.S)


def _enum_values(text):
    vals = {}
    for body in re.findall(r"enum\s*\{(.*?)\}", text, flags=re.S):
        nxt = 0
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, expr = (x.strip() for x in item.split("=", 1))
                nxt = eval(expr, {}, dict(vals))
            else:
                name = item
            vals[name] = nxt
            nxt += 1
    return vals


def test_prototype_matches_the_binding():
    text = " ".join(_header().split())
    assert "int wf_set_final_capture(wf_env* env, uint32_t* records_dev, int64_t capacity, uint32_t* count_dev);" in text
    assert "int64_t wf_final_record_words(int32_t width, int32_t height);" in text
    assert {"wf_set_final_capture", "wf_final_record_words"} <= set(_lib.EXPORTED_SYMBOLS)


def test_layout_constants_match_the_binding():
    v = _enum_values(_header())
    names = ["K", "ENV", "EPISODE", "T", "AX", "AY", "FLAGS", "NEXT_AX", "NEXT_AY"]
    assert [v["WF_F_" + n] for n in names] == [getattr(_lib, "F_" + n) for n in names]
    assert v["WF_FINAL_HEADER_WORDS"] == _lib.FINAL_HEADER_WORDS and v["WF_FINAL_OBS"] == _lib.FINAL_OBS
    for n in ("ALIVE", "VISIBLE", "DEAD", "DIGGING"):
        assert v["WF_FINAL_" + n] == getattr(_lib, "FINAL_" + n)
    for n in ("FIRE", "BURNT", "DIRT", "WATER"):
        assert v["WF_FINAL_PLANE_" + n] == getattr(_lib, "FINAL_PLANE_" + n)
    assert v["WF_F_NEXT_AY"] < v["WF_FINAL_HEADER_WORDS"]


def test_record_words_match_the_library():
    _lib.build()
    L = _lib.lib()
    for W, H in [(10, 10), (14, 14), (12, 10), (32, 32), (40, 20), (48, 48), (100, 70), (256, 256), (1024, 1024)]:
        n = _lib.final_record_words(W, H)
        assert L.wf_final_record_words(W, H) == n and n % 4 == 0
        assert _lib.final_plane_offset(W, H) >= _lib.FINAL_OBS + _lib.obs_bits_words(W, H)
        assert n >= _lib.final_plane_offset(W, H) + 4 * _lib.final_plane_words(W, H)


def _pack_bits(flat):
    """0/1 vector -> uint32 words, element i = bit i % 32 of word i // 32."""
    words = (len(flat) + 31) // 32
    padded = np.zeros(words * 32, np.uint64)
    padded[:len(flat)] = flat
    return (padded.reshape(words, 32) << np.arange(32, dtype=np.uint64)).sum(1).astype(np.uint32)


def _record(W, H, typ, k, env, ax, ay, flags, nxt, episode=3, t=17):
    rec = np.zeros(_lib.final_record_words(W, H), np.uint32)
    rec[:9] = np.array([k, env, episode, t, ax, ay, flags, nxt[0], nxt[1]], np.int64).astype(np.uint32)
    obs = np.zeros((W, H, 3), np.uint8)
    if flags & _lib.FINAL_VISIBLE:
        obs[ax, ay, 0] = 1
    obs[..., 1] = typ == 1
    obs[..., 2] = (typ != 3) & (typ != 4)  # fire_mobility != inf: everything but dirt and water
    ow = _lib.obs_bits_words(W, H)
    rec[_lib.FINAL_OBS:_lib.FINAL_OBS + ow] = _pack_bits(obs.reshape(-1))
    po, pw = _lib.final_plane_offset(W, H), _lib.final_plane_words(W, H)
    for p, code in enumerate((1, 2, 3, 4)):
        rec[po + p * pw:po + (p + 1) * pw] = _pack_bits((typ == code).reshape(-1).astype(np.uint8))
    return rec, obs


def _np_render(typ, alive, ax, ay):
    W, H = typ.shape
    rows = ["".join("A" if alive and (x, y) == (ax, ay) else ascii_of_type[int(typ[x, y])] for x in range(W)) for y in range(H)]
    return "\n" + "\n".join(rows) + "\n"


@pytest.mark.parametrize("W,H", [(10, 10), (14, 14), (12, 10), (40, 20), (33, 33)])
def test_parsing_types_and_render_against_numpy(W, H):
    rng = np.random.default_rng(W * 100 + H)
    cases = [(2, 5, 1), (0, 7, 0), (2, 1, 2), (1, 0, 3)]  # (k, env, flag set); deliberately out of (k, env) order
    flag_sets = [_lib.FINAL_ALIVE | _lib.FINAL_VISIBLE | _lib.FINAL_DIGGING, _lib.FINAL_DEAD, _lib.FINAL_ALIVE, 0]
    recs, expect = [], []
    for k, env, f in cases:
        typ = rng.integers(0, 5, (W, H)).astype(np.uint8)
        ax, ay = int(rng.integers(0, W)), int(rng.integers(0, H))
        nxt = (-1, -1) if f == 3 else (int(rng.integers(0, W)), int(rng.integers(0, H)))
        rec, obs = _record(W, H, typ, k, env, ax, ay, flag_sets[f], nxt)
        recs.append(rec)
        expect.append(dict(k=k, env=env, typ=typ, ax=ax, ay=ay, flags=flag_sets[f], nxt=nxt, obs=obs, rec=rec))
    fs = FinalStates(torch.from_numpy(np.stack(recs).view(np.int32)), W, H, "bits", n_envs=8)
    expect.sort(key=lambda e: (e["k"], e["env"]))
    assert len(fs) == 4
    assert fs.k.tolist() == [e["k"] for e in expect] and fs.env.tolist() == [e["env"] for e in expect]
    for i, e in enumerate(expect):
        assert np.array_equal(fs.records[i].numpy().view(np.uint32), e["rec"])
        assert np.array_equal(fs.types()[i].numpy(), e["typ"])
        assert fs.agent[i].tolist() == [e["ax"], e["ay"]] and fs.next_start[i].tolist() == list(e["nxt"])
        assert bool(fs.alive[i]) == bool(e["flags"] & _lib.FINAL_ALIVE)
        assert bool(fs.visible[i]) == bool(e["flags"] & _lib.FINAL_VISIBLE)
        assert bool(fs.dead[i]) == bool(e["flags"] & _lib.FINAL_DEAD)
        assert bool(fs.digging[i]) == bool(e["flags"] & _lib.FINAL_DIGGING)
        assert int(fs.episode[i]) == 3 and int(fs.t[i]) == 17
        bits = fs.obs[i].numpy().view(np.uint32)
        got = np.unpackbits(bits.view(np.uint8), bitorder="little")[:W * H * 3].reshape(W, H, 3)
        assert np.array_equal(got, e["obs"])
        assert fs.render(i) == _np_render(e["typ"], bool(e["flags"] & _lib.FINAL_ALIVE), e["ax"], e["ay"])


def test_empty_finals():
    fs = FinalStates(torch.zeros((0, _lib.final_record_words(14, 14)), dtype=torch.int32), 14, 14, "bits")
    assert len(fs) == 0 and tuple(fs.types().shape) == (0, 14, 14)


def _reference_rule(returns, best=-10000):
    """DQN.py:120-148 as the reference writes it: the maps log and the best return after a run of episodes."""
    maps = []
    for episode, total_reward in enumerate(returns):
        if total_reward >= 0.9 * best or total_reward > 300:
            map_string = f"map{episode}"
            if total_reward > best:
                best = total_reward
            maps.append([episode, map_string])
    return maps, best


@pytest.mark.parametrize("seed", range(4))
def test_map_rule_matches_end_of_episode(seed):
    """The learners' map rule (agents._map_rule, used by _end_of_episode and by record_maps) against the reference's
    statement, and _end_of_episode itself (called on a stand-in agent) against both, on synthetic returns."""
    import types as pytypes

    from wildfire_control_python_b200 import agents as A
    rng = np.random.default_rng(seed)
    returns = list(rng.choice([-1000.0, -120.0, -35.0, 0.0, 150.0, 320.0, 640.0, 999.5], size=200)
                   + rng.normal(0, 20, size=200).round(2))
    want_maps, want_best = _reference_rule(returns)
    maps, best = [], -10000
    for i, r in enumerate(returns):
        best = A._map_rule(maps, best, i, r, lambda i=i: f"map{i}")
    assert maps == want_maps and best == want_best
    rendered = []
    fake = pytypes.SimpleNamespace(
        sim=pytypes.SimpleNamespace(W=pytypes.SimpleNamespace(agents=[1])), DEBUG=1, verbose=False, eps=1.0,
        logs={"best_reward": -10000, "maps": [], "agent_deaths": [], "total_rewards": []},
        decay_epsilon=lambda episode: None)
    fake._render_string = lambda: (rendered.append(1), f"map{len(fake.logs['total_rewards'])}")[1]
    for i, r in enumerate(returns):
        A.DQN._end_of_episode(fake, i, r, 0.0)
    assert fake.logs["maps"] == want_maps and fake.logs["best_reward"] == want_best
    assert len(rendered) == len(want_maps)
