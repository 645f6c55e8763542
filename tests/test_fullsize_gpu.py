"""Parity at BASELINE.json's full sizes.

C2 (4096 envs of 14x14) is small enough for the C oracle to replay every env.  For the large-grid
configs (C4: 256x256, C5: 1024x1024) the oracle replays a handful of envs for a bounded number of
steps, and the whole batch is checked through size-independent properties: determinism, independence
of the batch composition (sharding), fused rollout == repeated steps, mirror symmetry of a free burn
without wind, and conservation (every cell is exactly one type; burning cells have fuel).
"""
import numpy as np
import pytest
import torch

from oracle import wf_oracle as wo
from tests.gpu_util import compare_states, make_pair, to_np

pytestmark = pytest.mark.gpu


def test_c2_full_batch_every_env_matches_oracle():
    cfg = dict(width=14, height=14, seed=0)
    N, K = 4096, 120
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    gpu.reset()
    for e in orc:
        e.reset()
    _, rew, done = gpu.rollout(K, obs=False)
    rew, done = to_np(rew), to_np(done)
    for i, e in enumerate(orc):
        for k in range(K):
            _, r, d, _ = e.step(e.random_action())
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k)
            if d:
                e.reset()
    compare_states("c2 full batch", gpu, orc, envs=range(0, N, 97))
    obs = gpu.observe()
    for i in range(0, N, 211):
        assert np.array_equal(to_np(obs[i]), orc[i].obs())


@pytest.mark.parametrize("size,n_envs,steps,ign,wind", [(256, 6, 120, 32, [0.85, (1, 0)]), (1024, 2, 40, 256, [0.54, (0, 0)])],
                         ids=["c4_256", "c5_1024"])
def test_large_grid_envs_match_oracle(size, n_envs, steps, ign, wind):
    cfg = dict(width=size, height=size, seed=5, wind=wind, extra_ignitions=ign)
    gpu, orc = make_pair(n_envs, cfg)
    obs = gpu.reset()
    for e in orc:
        e.reset()
    compare_states("reset", gpu, orc, obs=obs)
    for s in range(steps):
        acts = [e.random_action() for e in orc]
        live = [bool(e.planes()["running"]) for e in orc]
        obs, rew, done, _ = gpu.step(torch.tensor(acts, dtype=torch.int32, device="cuda"))
        rew, done = to_np(rew), to_np(done)
        for i, e in enumerate(orc):
            if not live[i]:
                continue
            _, r, d, _ = e.step(acts[i])
            assert rew[i] == r and bool(done[i]) == d, (s, i)
        if s % 20 == 19 or s == steps - 1:
            compare_states(f"step {s}", gpu, orc, obs=obs)


def _conservation(st):
    typ, burning, fuel = st["type"], st["burning"], st["fuel"]
    assert int(typ.max()) <= 4
    assert bool(((burning == 1) <= ((typ == 1) | (typ == 3))).all())  # burning cells are fire (or dug while burning)
    assert bool((fuel[burning == 1] >= 1).all())
    assert bool((fuel[typ == 2] == 0).all())


def test_c4_full_batch_properties():
    from wildfire_control_python_b200.batched import BatchedForestFire
    cfg = dict(width=256, height=256, seed=11, wind=[0.85, (1, 0)], extra_ignitions=32, auto_reset=True)
    N, K = 1024, 48
    a = BatchedForestFire(N, **cfg)
    b = BatchedForestFire(N // 2, env_id_base=N // 2, **cfg)  # the upper half of the same global batch
    a.reset(); b.reset()
    acts = torch.randint(0, 4, (K, N), dtype=torch.int32, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    ra, da = [], []
    for k in range(K):
        o, r, d, _ = a.step(acts[k])
        ra.append(r.clone()); da.append(d.clone())
        ob, rb, db, _ = b.step(acts[k, N // 2:])
        assert torch.equal(r[N // 2:], rb) and torch.equal(d[N // 2:], db), k
        if k % 16 == 15:
            assert torch.equal(o[N // 2:], ob), k
    st = a.get_state()
    _conservation(st)
    # fused rollout from a fresh handle reproduces the stepped trajectory exactly (determinism)
    c = BatchedForestFire(N, **cfg)
    c.reset()
    _, rc, dc = c.rollout(K, actions=acts, obs=False)
    assert torch.equal(rc, torch.stack(ra)) and torch.equal(dc, torch.stack(da))
    sc = c.get_state()
    for k in ("type", "burning", "fm_inf", "fuel", "hits", "scalars"):
        assert torch.equal(st[k], sc[k]), k


def test_free_burn_without_wind_is_mirror_symmetric_256():
    """No wind: the quanta are direction-independent, so a free burn from the centre of an odd..even grid
    stays symmetric under (x, y) -> (y, x) (the transpose), whatever the size."""
    from wildfire_control_python_b200.batched import BatchedForestFire
    S = 256
    env = BatchedForestFire(2, width=S, height=S, seed=1)
    env.reset(starts=torch.tensor([[S // 2 + 3, S // 2 + 3]] * 2, dtype=torch.int32))  # agent parked on the diagonal
    noop = torch.full((2,), 7, dtype=torch.int32, device="cuda")
    for _ in range(400):
        env.step(noop)
    st = env.get_state()
    typ, fuel, hits = st["type"][0], st["fuel"][0], st["hits"][0]
    assert int((typ == 1).sum()) > 50  # a real front exists
    assert torch.equal(typ, typ.T) and torch.equal(fuel, fuel.T)
    total = hits.int().sum(-1)
    assert torch.equal(total, total.T)


# ---------------------------------------------------------------------------------------------
# The tile geometries bench.py really runs.  choose_geometry (wf_tile.cu) picks threads-per-CTA x CTAs-per-cluster from
# the number of envs: C4's 1024 envs of 256x256 get (256, 1), C5's 64 envs of 1024x1024 get (128, 16).  A handful of envs
# would get a different geometry, so the production one is forced (WF_TILE_T / WF_TILE_CS, read by wf_create) and the
# test asserts that it is the one the full batch gets.
def _production_geometry(monkeypatch, size, full_batch):
    from wildfire_control_python_b200.batched import BatchedForestFire
    monkeypatch.delenv("WF_TILE_T", raising=False)
    monkeypatch.delenv("WF_TILE_CS", raising=False)
    probe = BatchedForestFire(full_batch, width=size, height=size)  # no reset: only asks which geometry the batch gets
    geom = probe.tile_geometry
    probe.close()
    monkeypatch.setenv("WF_TILE_T", str(geom[0]))
    monkeypatch.setenv("WF_TILE_CS", str(geom[1]))
    return geom


def _rollout_against_oracle(gpu, orc, steps, chunk, policy, check_state_every):
    """`steps` steps in launches of `chunk` (what bench.py times), every action / reward / done / observation of every
    env against the oracle, auto-reset included; full state every `check_state_every` steps."""
    events = dict(contained=0, done=0, deaths=0)
    s = 0
    while s < steps:
        c = min(chunk, steps - s)
        obs, rew, done, acts = gpu.rollout(c, policy=policy, return_actions=True)
        obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
        for i, e in enumerate(orc):
            for k in range(c):
                a = e.walk_action() if policy == "walk" else e.random_action()
                assert acts[k, i] == a, (s + k, i)
                o, r, d, _ = e.step(a)
                if r == 1000.0:
                    events["contained"] += 1
                if d:
                    events["done"] += 1
                    events["deaths"] += int(r == -1000.0)
                    o = e.reset()
                assert rew[k, i] == r and bool(done[k, i]) == d, (s + k, i, rew[k, i], r)
                assert np.array_equal(obs[k, i], o), (s + k, i)
        s += c
        if s % check_state_every == 0 or s == steps:
            compare_states(f"step {s}", gpu, orc)
    return events


def test_c4_production_geometry_matches_oracle(monkeypatch):
    """C4 (256x256, wind [0.85,(1,0)], 32 extra ignitions) on the geometry its 1024-env batch runs with: 256 threads,
    cluster of 1.  300 ticks in 16-step launches: several ignition generations, burn-outs, deaths and auto-resets."""
    geom = _production_geometry(monkeypatch, 256, 1024)
    assert geom == (256, 1)
    cfg = dict(width=256, height=256, seed=6, wind=[0.85, (1, 0)], extra_ignitions=32)
    gpu, orc = make_pair(6, cfg, auto_reset=True)
    assert gpu.tile_geometry == geom
    obs = gpu.reset()
    for e in orc:
        e.reset()
    compare_states("reset", gpu, orc, obs=obs)
    ev = _rollout_against_oracle(gpu, orc, 304, 16, "stream", 64)
    assert ev["done"] >= 1  # at least one in-kernel reset happened


def test_c5_production_geometry_matches_oracle(monkeypatch):
    """C5 (1024x1024, no wind, 256 extra ignitions) on the geometry its 64-env batch runs with: 16 CTAs of 128 threads
    per env (8 of 256 where the device cannot hold a cluster of 16).  272 ticks in 16-step launches (14 ignition generations of the 19-tick delay; the first fires burn out at tick 20)."""
    geom = _production_geometry(monkeypatch, 1024, 64)
    assert geom in ((128, 16), (256, 8))
    cfg = dict(width=1024, height=1024, seed=6, extra_ignitions=256)  # envs 0 and 2 start with no fire on the border
    gpu, orc = make_pair(3, cfg, auto_reset=True)
    assert gpu.tile_geometry == geom
    obs = gpu.reset()
    for e in orc:
        e.reset()
    compare_states("reset", gpu, orc, obs=obs)
    _rollout_against_oracle(gpu, orc, 272, 16, "stream", 136)


def test_c5_geometry_walk_policy_contains_burns_out_and_resets(monkeypatch):
    """1024x1024 on the C5 geometry with the reference's heuristic walk policy (DQN.py:353-389): the bulldozer rings
    the fire (containment bonus, environment.py:342-377 -- the reach plane is cut by the closing dig and re-flooded by
    the whole cluster), the ring burns out (burn-out reward), the env resets inside the kernel and does it again."""
    geom = _production_geometry(monkeypatch, 1024, 64)
    cfg = dict(width=1024, height=1024, seed=6)
    gpu, orc = make_pair(2, cfg, auto_reset=True)
    assert gpu.tile_geometry == geom and geom in ((128, 16), (256, 8))
    gpu.reset()
    for e in orc:
        e.reset()
    ev = _rollout_against_oracle(gpu, orc, 256, 16, "walk", 128)
    assert ev["contained"] >= 2 and ev["done"] >= 2 and ev["deaths"] == 0
