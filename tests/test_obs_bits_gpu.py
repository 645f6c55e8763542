"""WF_OBS_BITS on the GPU: a handle with obs_dtype="bits" and a uint8 handle with the same seed and config step alike, and
every packed observation, unpacked with NumPy, equals the uint8 one element for element (padding bits zero); reward and
done are identical.  Covers both kernel families (the tile family on production, cluster and ragged geometries under
its three step structures), the host-buffer paths and wf_unpack_obs_bits."""
import time

import numpy as np
import pytest
import torch

from tests.test_obs_bits_cpu import np_unpack
from wildfire_control_python_b200 import _lib, obs_bits_words, unpack_obs
from wildfire_control_python_b200.batched import BatchedForestFire

pytestmark = pytest.mark.gpu

RICH = dict(make_rivers=True, wind="random", a_speed=2)  # rivers, random wind, a fire tick every other step


def np_(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)


def assert_bits_equal(bits, obs_u8, W, H, tag=""):
    b = np_(bits)
    assert b.shape[-1] == obs_bits_words(W, H), tag
    back, pad = np_unpack(b, W, H)
    assert not pad.any(), f"{tag}: padding bits set"
    o = np_(obs_u8)
    if not np.array_equal(back, o):
        idx = np.argwhere(back != o)[:5]
        raise AssertionError(f"{tag}: {int((back != o).sum())} elements differ, first at {idx.tolist()}")


def pair(n, **cfg):
    return BatchedForestFire(n, **cfg), BatchedForestFire(n, obs_dtype="bits", **cfg)


def step_both(a, b, acts, W, H, tag):
    oa, ra, da, _ = a.step(acts)
    ob, rb, db, _ = b.step(acts)
    assert ob.dtype == torch.int32 and tuple(ob.shape) == (a.n_envs, obs_bits_words(W, H))
    assert torch.equal(ra, rb) and torch.equal(da, db), tag
    assert_bits_equal(ob, oa, W, H, tag)
    return da


def rollout_both(a, b, K, W, H, tag, **kw):
    oa, ra, da = a.rollout(K, **kw)
    ob, rb, db = b.rollout(K, **kw)
    assert tuple(ob.shape) == (K, a.n_envs, obs_bits_words(W, H))
    assert torch.equal(ra, rb) and torch.equal(da, db), tag
    assert_bits_equal(ob, oa, W, H, tag)
    return da


# ---------------------------------------------------------------------------------------------
# warp family (W, H <= 32): 16- and 32-lane envs, two envs per record with a half-full last warp
@pytest.mark.parametrize("cfg", [dict(), RICH], ids=["plain", "rivers_randwind_aspeed2"])
@pytest.mark.parametrize("W,H,N", [(10, 10, 37), (14, 14, 67), (17, 16, 37), (32, 32, 67)])
def test_warp_family_bits_equal_uint8(W, H, N, cfg):
    a, b = pair(N, width=W, height=H, seed=7, auto_reset=True, extra_ignitions=2, **cfg)
    assert a.kernel_family == "warp"
    assert_bits_equal(b.reset(), a.reset(), W, H, "reset")
    g = torch.Generator("cuda").manual_seed(W * 100 + N)
    done_seen = 0
    for s in range(24):
        acts = torch.randint(0, 5, (N,), dtype=torch.int32, device="cuda", generator=g)
        done_seen += int(step_both(a, b, acts, W, H, f"step {s}").sum())
    for pol in ("stream", "walk"):
        done_seen += int(rollout_both(a, b, 40, W, H, f"rollout {pol}", policy=pol).sum())
    acts = torch.randint(0, 4, (8, N), dtype=torch.int32, device="cuda", generator=g)
    rollout_both(a, b, 8, W, H, "rollout with actions", actions=acts)
    rng = np.random.default_rng(W)
    k1, b1 = rng.normal(size=(W * H * 3, 16)).astype(np.float32), rng.normal(size=16).astype(np.float32)
    k2, b2 = rng.normal(size=(16, 4)).astype(np.float32), rng.normal(size=4).astype(np.float32)
    for env in (a, b):
        env.set_policy_mlp(k1, b1, k2, b2, eps=0.2)
    rollout_both(a, b, 16, W, H, "rollout mlp", policy="mlp")
    mask = torch.tensor(rng.integers(0, 2, N), dtype=torch.uint8, device="cuda")
    assert_bits_equal(b.reset(mask=mask), a.reset(mask=mask), W, H, "masked reset")
    step_both(a, b, torch.zeros(N, dtype=torch.int32, device="cuda"), W, H, "after masked reset")
    assert_bits_equal(b.observe(), a.observe(), W, H, "observe")
    assert done_seen > 0  # auto-reset emitted observations of fresh episodes


# ---------------------------------------------------------------------------------------------
# tile family
def _tile_run(monkeypatch, W, H, N, T, CS, steps, chunk, want_done, **cfg):
    monkeypatch.setenv("WF_TILE_T", str(T))
    monkeypatch.setenv("WF_TILE_CS", str(CS))
    a, b = pair(N, width=W, height=H, seed=5, auto_reset=True, **cfg)
    assert a.kernel_family == "tile" and a.tile_geometry == b.tile_geometry
    assert_bits_equal(b.reset(), a.reset(), W, H, "reset")
    done = 0
    g = torch.Generator("cuda").manual_seed(W + H)
    step_both(a, b, torch.randint(0, 4, (N,), dtype=torch.int32, device="cuda", generator=g), W, H, "step")
    for s in range(0, steps, chunk):
        done += int(rollout_both(a, b, chunk, W, H, f"rollout from step {s}").sum())
    assert_bits_equal(b.observe(), a.observe(), W, H, "observe")
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[0] = 1
    assert_bits_equal(b.reset(mask=mask), a.reset(mask=mask), W, H, "masked reset")
    if want_done:
        assert done > 0  # the second emission of a step's observation under auto-reset was checked
    return a.tile_geometry


def test_tile_c4_production_geometry(monkeypatch):
    geom = _tile_run(monkeypatch, 256, 256, 4, 256, 1, 96, 16, False, wind=[0.85, (1, 0)], extra_ignitions=32)
    assert geom == (256, 1)


@pytest.mark.parametrize("T,CS", [(256, 8), (128, 16)])
def test_tile_1024_clusters(monkeypatch, T, CS):
    geom = _tile_run(monkeypatch, 1024, 1024, 2, T, CS, 32, 16, False, extra_ignitions=64)
    assert geom[1] > 1


@pytest.mark.parametrize("W,H,T,CS", [(100, 70, 128, 4), (48, 33, 128, 2), (40, 40, 128, 2)])
def test_tile_ragged_sizes_straddle_cta_slices(monkeypatch, W, H, T, CS):
    geom = _tile_run(monkeypatch, W, H, 5, T, CS, 320, 32, True, wind=[0.85, (1, 0)], extra_ignitions=3)
    assert geom[1] == CS


# ---------------------------------------------------------------------------------------------
# host-buffer API
def _host_step(env, acts, obs, code, pageable):
    """wf_step_host with the handle's pinned arrays (pageable=False: BatchedForestFire.step_host) or with pageable numpy."""
    if not pageable:
        o, r, d, _ = env.step_host(acts)
        return o.copy(), r.copy(), d.copy()
    a = np.ascontiguousarray(acts, dtype=np.int32)
    r = np.empty(env.n_envs, np.float64)
    d = np.empty(env.n_envs, np.uint8)
    _lib.check(_lib.lib().wf_step_host(env._h, a.ctypes.data, obs.ctypes.data, code, r.ctypes.data, d.ctypes.data))
    return obs.copy(), r, d.view(np.bool_)


@pytest.mark.parametrize("pageable", [False, True], ids=["pinned", "pageable"])
@pytest.mark.parametrize("session", [0, 1, 2])
@pytest.mark.parametrize("W,H,N", [(14, 14, 67), (32, 32, 37), (40, 40, 5)])
def test_host_paths_bits(W, H, N, session, pageable):
    cfg = dict(width=W, height=H, seed=9, auto_reset=True, extra_ignitions=1)
    a = BatchedForestFire(N, **cfg)                     # uint8, host path
    b = BatchedForestFire(N, obs_dtype="bits", **cfg)   # bits, host path
    c = BatchedForestFire(N, obs_dtype="bits", **cfg)   # bits, device path
    words = obs_bits_words(W, H)
    if session:
        ok_a = a.host_session(True, persistent_obs=session == 2)
        ok_b = b.host_session(True, persistent_obs=session == 2)
        assert ok_a == ok_b == (a.kernel_family == "warp")
    oa_buf = np.empty((N, W, H, 3), np.uint8)
    ob_buf = np.empty((N, words), np.uint32)
    # wf_reset_host with bits
    L = _lib.lib()
    _lib.check(L.wf_reset_host(a._h, None, None, oa_buf.ctypes.data, _lib.WF_OBS_U8))
    _lib.check(L.wf_reset_host(b._h, None, None, ob_buf.ctypes.data, _lib.WF_OBS_BITS))
    oc = c.reset()
    assert np.array_equal(ob_buf, np_(oc).view(np.uint32))
    assert_bits_equal(ob_buf, oa_buf, W, H, "reset_host")
    rng = np.random.default_rng(N)
    for s in range(30):
        acts = rng.integers(0, 4, N).astype(np.int32)
        if s == 12:  # the session's kernel parks itself after WF_SESSION_IDLE_US (2 ms) without a step
            time.sleep(0.02)
        if s == 20:  # an interleaved device step parks the session; the next host step starts it again
            t = torch.as_tensor(acts, device="cuda")
            a.step(t)
            b.step(t)
            c.step(t)
            torch.cuda.synchronize()
            continue
        o_a, r_a, d_a = _host_step(a, acts, oa_buf, _lib.WF_OBS_U8, pageable)
        o_b, r_b, d_b = _host_step(b, acts, ob_buf, _lib.WF_OBS_BITS, pageable)
        o_c, r_c, d_c, _ = c.step(torch.as_tensor(acts, device="cuda"))
        assert o_b.dtype == np.uint32 and o_b.shape == (N, words)
        assert np.array_equal(o_b, np_(o_c).view(np.uint32)), f"step {s}: host bits != device bits"
        assert_bits_equal(o_b, o_a, W, H, f"step {s}")
        assert np.array_equal(r_b, r_a) and np.array_equal(r_b, np_(r_c)), s
        assert np.array_equal(d_b, d_a) and np.array_equal(d_b, np_(d_c)), s
    if session:
        for env in (a, b):
            env.host_session(False)


def test_session_alternating_dtypes_mode2():
    """Mode 2 with uint8 and bits calls on one handle, each dtype with its own persistent array: a call whose dtype
    differs from the previous one's gets every record in full, so both arrays stay complete."""
    W, H, N = 14, 14, 67
    cfg = dict(width=W, height=H, seed=4, auto_reset=True)
    s = BatchedForestFire(N, **cfg)
    c = BatchedForestFire(N, **cfg)
    assert s.host_session(True, persistent_obs=True)
    s.reset()
    c.reset()
    ou8 = np.empty((N, W, H, 3), np.uint8)
    obits = np.empty((N, obs_bits_words(W, H)), np.uint32)
    rng = np.random.default_rng(1)
    for k in range(16):
        acts = rng.integers(0, 4, N).astype(np.int32)
        bits = k % 3 == 2
        _host_step(s, acts, obits if bits else ou8, _lib.WF_OBS_BITS if bits else _lib.WF_OBS_U8, True)
        o_c, _, _, _ = c.step(torch.as_tensor(acts, device="cuda"))
        if bits:
            assert_bits_equal(obits, o_c, W, H, f"step {k}")
        else:
            assert np.array_equal(ou8, np_(o_c)), k
    s.host_session(False)


# ---------------------------------------------------------------------------------------------
# wf_unpack_obs_bits
@pytest.mark.parametrize("W,H,N", [(14, 14, 67), (32, 32, 37), (100, 70, 3)])
def test_unpack_obs(W, H, N):
    a, b = pair(N, width=W, height=H, seed=2, auto_reset=True, extra_ignitions=2)
    a.reset()
    b.reset()
    K = 6
    oa, _, _ = a.rollout(K)
    ob, _, _ = b.rollout(K)
    words = obs_bits_words(W, H)
    flat_bits, flat_u8 = ob.view(-1, words), oa.view(-1, W, H, 3)
    rows = K * N
    idx = torch.cat([torch.arange(rows - 1, -1, -1), torch.tensor([3, 3, 0, rows - 1, 3])]).cuda()
    bad = torch.tensor([-1, rows, rows + 7, -(2**40)], device="cuda")
    for dt in (torch.uint8, torch.float32, torch.bfloat16):
        u = unpack_obs(flat_bits, W, H, dtype=dt)
        assert u.dtype == dt and tuple(u.shape) == (rows, W, H, 3)
        assert torch.equal(u, flat_u8.to(dt))
        assert np.array_equal(np_(u.to(torch.uint8)), np_unpack(np_(flat_bits).view(np.uint32), W, H)[0])
        g = unpack_obs(flat_bits, W, H, index=idx, dtype=dt)
        assert torch.equal(g, flat_u8[idx].to(dt))
        z = unpack_obs(flat_bits, W, H, index=torch.cat([bad, idx[:2]]), dtype=dt)
        assert not z[: len(bad)].any() and torch.equal(z[len(bad):], flat_u8[idx[:2]].to(dt))
    assert unpack_obs(flat_bits, W, H, index=torch.empty(0, dtype=torch.int64)).shape == (0, W, H, 3)
    # one step's rows feed the reference's Flatten order unchanged
    assert torch.equal(unpack_obs(b.observe(), W, H).flatten(1), a.observe().float().flatten(1))


def test_sharded_forest_fire_passes_bits_through():
    from wildfire_control_python_b200.sharding import ShardedForestFire
    s = ShardedForestFire(10, width=14, height=14, seed=1, obs_dtype="bits")
    a = BatchedForestFire(10, width=14, height=14, seed=1)
    assert tuple(s.reset().shape) == (10, obs_bits_words(14, 14))
    assert_bits_equal(s.observe(), a.reset(), 14, 14, "sharded")
