"""GPU parity: the CUDA path (through the C ABI) against the golden fixtures recorded from the
Python reference and against the C oracle on the same seeded inputs.  Bit-exact on type /
burning / fm_inf / fuel / agent / fire_at_border / obs / reward / done; temp within 1e-9 on grass.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import wf_oracle as wo
from tests.golden_util import env_cfg, expected_obs, golden_names, load_golden
from tests.gpu_util import TEMP_TOL, compare_states, make_pair, to_np

pytestmark = pytest.mark.gpu


def _lib():
    from wildfire_control_python_b200 import _lib as L
    return L


KATS = [
    ((0, 0, 0, 0, 0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 6, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


@pytest.mark.parametrize("ctr_key,want", KATS)
def test_device_philox_kat(ctr_key, want):
    L = _lib()
    inp = (C.c_uint32 * 6)(*ctr_key)
    out = (C.c_uint32 * 4)()
    L.check(L.lib().wf_philox_kat(0, inp, out))
    assert tuple(out) == want


@pytest.mark.parametrize("name", golden_names())
def test_gpu_reproduces_reference_golden(name):
    """Env 0 of a 3-env batch must follow the trajectory the Python reference produced."""
    g = load_golden(name)
    cfg = env_cfg(g)
    from wildfire_control_python_b200.batched import BatchedForestFire
    L = _lib()
    gpu = BatchedForestFire(3, **cfg)
    F = len(g["kind"])
    mask = torch.tensor([1, 0, 0], dtype=torch.uint8, device="cuda")
    for f in range(F):
        tag = f"{name} frame {f}"
        if g["kind"][f] == 0:
            obs = gpu.reset() if f == 0 else gpu.reset(mask=mask)
        else:
            a = int(g["action"][f])
            obs, rew, done, _ = gpu.step(torch.tensor([a, a, a], dtype=torch.int32, device="cuda"))
            assert float(rew[0]) == float(g["reward"][f]), f"{tag}: reward {float(rew[0])} != {g['reward'][f]}"
            assert bool(done[0]) == bool(g["done"][f]), f"{tag}: done"
        st = {k: to_np(v)[0] for k, v in gpu.get_state().items()}
        for k in ("type", "burning", "fm_inf", "fuel", "apos"):
            assert np.array_equal(st[k], g[k][f]), f"{tag}: plane {k}\ngpu=\n{st[k].T}\nref=\n{g[k][f].T}"
        sc = st["scalars"]
        assert sc[L.S_ALIVE] == g["alive"][f], tag
        if g["alive"][f]:
            assert (sc[L.S_AX], sc[L.S_AY]) == (g["ax"][f], g["ay"][f]), tag
        assert sc[L.S_FIRE_AT_BORDER] == g["fire_at_border"][f], tag
        assert sc[L.S_RUNNING] == g["running"][f], tag
        assert (sc[L.S_WIND_X], sc[L.S_WIND_Y]) == (g["wind_x"][f], g["wind_y"][f]), tag
        assert gpu.wind_speed_table[sc[L.S_WIND_ID]] == g["wind_speed"][f], tag
        grass = g["type"][f] == 0
        assert np.abs(st["temp"] - g["temp"][f])[grass].max(initial=0.0) <= TEMP_TOL, f"{tag}: temp"
        assert np.array_equal(to_np(obs)[0], expected_obs(g, f)), f"{tag}: obs"


SCENARIOS = [
    dict(width=14, height=14, seed=101),
    dict(width=10, height=10, seed=102, allow_dig_toggle=True, n_actions=6),
    dict(width=20, height=20, seed=103, wind="random", make_rivers=True),
    dict(width=16, height=16, seed=104, a_speed=2, wind=[0.85, (1, 0)], extra_ignitions=2),
    dict(width=32, height=32, seed=105, wind=[0.85, (-1, 1)], extra_ignitions=5),
    dict(width=17, height=13, seed=106, wind=[0.7, (0, 1)]),
    dict(width=11, height=11, seed=107, fuel=40, threshold=5.0, heat=0.35),
    # tile family (W or H > 32): several words per row, ragged last word, rivers, wind, ignitions
    dict(width=40, height=40, seed=108, extra_ignitions=3),
    dict(width=64, height=64, seed=109, wind="random", make_rivers=True, extra_ignitions=6),
    dict(width=100, height=70, seed=110, wind=[0.85, (1, 0)], extra_ignitions=10, a_speed=2),
    dict(width=48, height=33, seed=111, allow_dig_toggle=True, n_actions=6, wind=[0.85, (0, -1)], extra_ignitions=2),
    dict(width=33, height=20, seed=112, fuel=50, threshold=4.0),
    # 4 words per row (128-bit path) with a ragged last word: H = 100
    dict(width=120, height=100, seed=113, wind=[0.85, (0, 1)], extra_ignitions=5),
]


@pytest.mark.parametrize("cfg", SCENARIOS, ids=lambda c: f"{c['width']}x{c['height']}_s{c['seed']}")
def test_step_matches_oracle_batch(cfg):
    """37 envs (ragged vs the 2-or-1 envs-per-warp packing), stream actions, explicit masked resets."""
    N, STEPS = 37, 220
    gpu, orc = make_pair(N, cfg)
    obs = gpu.reset()
    for e in orc:
        e.reset()
    compare_states("reset", gpu, orc, obs=obs)
    a_speed = cfg.get("a_speed", 1)
    a_iter = a_speed  # METADATA['a_speed_iter']: one counter per process in the reference, per handle here
    for s in range(STEPS):
        acts = [e.random_action() for e in orc]
        frozen = [not e.planes()["running"] for e in orc]
        for e in orc:
            e.set_a_speed_iter(a_iter)
        a_iter = a_speed if a_iter == 1 else a_iter - 1
        obs, rew, done, _ = gpu.step(torch.tensor(acts, dtype=torch.int32, device="cuda"))
        rew, done = to_np(rew), to_np(done)
        for i, e in enumerate(orc):
            if frozen[i]:
                assert rew[i] == 0.0 and done[i]
                continue
            _, r, d, _ = e.step(acts[i])
            assert rew[i] == r, f"step {s} env {i}: reward {rew[i]} != {r}"
            assert bool(done[i]) == d, f"step {s} env {i}: done"
        if s % 7 == 0 or s == STEPS - 1:
            compare_states(f"step {s}", gpu, orc, obs=obs)
        if s % 25 == 24:  # reset the finished envs, like a caller of the reference would
            m = np.array([not e.planes()["running"] for e in orc], np.uint8)
            if m.any():
                obs = gpu.reset(mask=torch.from_numpy(m).cuda())
                for i in np.nonzero(m)[0]:
                    orc[i].reset()
                compare_states(f"masked reset after step {s}", gpu, orc, obs=obs)


@pytest.mark.parametrize("cfg", [dict(width=14, height=14, seed=201),
                                 dict(width=12, height=12, seed=202, wind="random", make_rivers=True, a_speed=2),
                                 dict(width=40, height=36, seed=203, wind="random", extra_ignitions=2)],
                         ids=["c2", "rivers_wind_aspeed2", "tile_40x36"])
def test_fused_rollout_matches_oracle(cfg):
    """wf_rollout: K steps in one launch, actions from the ACTION stream, auto-reset on done."""
    N, K = 67, 300
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    gpu.reset()
    for e in orc:
        e.reset()
    obs, rew, done = gpu.rollout(K)
    obs, rew, done = to_np(obs), to_np(rew), to_np(done)
    n_done = 0
    for i, e in enumerate(orc):
        for k in range(K):
            o, r, d, _ = e.step(e.random_action())
            assert rew[k, i] == r, f"env {i} step {k}: reward {rew[k, i]} != {r}"
            assert bool(done[k, i]) == d, f"env {i} step {k}: done"
            if d:
                o = e.reset()
                n_done += 1
            assert np.array_equal(obs[k, i], o), f"env {i} step {k}: obs"
    assert n_done > N  # several episodes per env on average
    compare_states("after rollout", gpu, orc)
    st = gpu.stats()
    assert st["episodes"] == n_done and st["env_steps"] == N * K


@pytest.mark.parametrize("cfg", [dict(width=14, height=14, seed=601), dict(width=20, height=20, seed=602, make_rivers=True),
                                 dict(width=40, height=40, seed=603), dict(width=72, height=64, seed=604, a_speed=2),
                                 dict(width=64, height=64, seed=605, make_rivers=True, wind="random")],
                         ids=lambda c: f"{c['width']}x{c['height']}_s{c['seed']}")
def test_scripted_containment_matches_oracle(cfg):
    """Every env walks a ring of its own radius round the fire (containment bonus, latch, burn-out
    reward), then takes stream actions; resets are applied as soon as an env finishes."""
    from oracle.policies import ring_actions
    N, STEPS = 12, 260
    gpu, orc = make_pair(N, cfg)
    gpu.reset()
    for e in orc:
        e.reset()
    W, H = cfg["width"], cfg["height"]

    def plan_for(i):
        p = orc[i].planes()
        return ring_actions(p["ax"], p["ay"], W // 2, H // 2, 2 + i % 4)

    plans = [plan_for(i) for i in range(N)]
    tcount = [0] * N
    a_speed = cfg.get("a_speed", 1)
    a_iter = a_speed
    n_contained = 0
    for s in range(STEPS):
        acts = []
        for i, e in enumerate(orc):
            a = e.random_action()
            if tcount[i] < len(plans[i]):
                a = plans[i][tcount[i]]
            acts.append(a)
            e.set_a_speed_iter(a_iter)
        a_iter = a_speed if a_iter == 1 else a_iter - 1
        obs, rew, done, _ = gpu.step(torch.tensor(acts, dtype=torch.int32, device="cuda"))
        rew, done = to_np(rew), to_np(done)
        m = np.zeros(N, np.uint8)
        for i, e in enumerate(orc):
            _, r, d, _ = e.step(acts[i])
            tcount[i] += 1
            assert rew[i] == r, f"step {s} env {i}: reward {rew[i]} != {r}"
            assert bool(done[i]) == d, f"step {s} env {i}: done"
            n_contained += int(r == 1000)
            m[i] = d
        compare_states(f"step {s}", gpu, orc, obs=obs)
        if m.any():
            obs = gpu.reset(mask=torch.from_numpy(m).cuda())
            for i in np.nonzero(m)[0]:
                orc[i].reset()
                plans[i] = plan_for(i)
                tcount[i] = 0
            compare_states(f"reset after step {s}", gpu, orc, obs=obs)
    assert n_contained >= N // 2


def test_rollout_equals_repeated_step():
    cfg = dict(width=14, height=14, seed=301)
    N, K = 33, 64
    a, _ = make_pair(N, cfg, auto_reset=True)
    b, _ = make_pair(N, cfg, auto_reset=True)
    a.reset(); b.reset()
    acts = torch.randint(0, 4, (K, N), dtype=torch.int32, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    obs_a, rew_a, done_a = a.rollout(K, actions=acts)
    for k in range(K):
        o, r, d, _ = b.step(acts[k])
        assert torch.equal(o, obs_a[k]) and torch.equal(r, rew_a[k]) and torch.equal(d, done_a[k]), k


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("cfg,n_envs", [(dict(width=14, height=14, seed=401), 9), (dict(width=13, height=11, seed=402), 7),
                                        (dict(width=32, height=32, seed=403), 3), (dict(width=40, height=36, seed=404), 5),
                                        (dict(width=64, height=64, seed=405), 4), (dict(width=128, height=128, seed=406), 3),
                                        (dict(width=130, height=128, seed=407, extra_ignitions=8), 2)],
                         ids=["14", "13x11_odd", "32", "tile_40x36", "tile_64", "tile_128_wide", "tile_130x128_wide_tail"])
def test_float_observation_equals_u8(cfg, n_envs, dtype):
    """WF_OBS_F32 / WF_OBS_BF16 (SURVEY 8(b): obs delivered as f32 / bf16 directly for the learner) hold exactly the
    0 / 1 values of the uint8 observation, through reset, step, rollout, observe and step_host."""
    a, _ = make_pair(n_envs, cfg, auto_reset=True)
    b, _ = make_pair(n_envs, cfg, auto_reset=True, obs_dtype=dtype)
    oa, ob = a.reset(), b.reset()
    assert ob.dtype == dtype and torch.equal(oa.to(dtype), ob)
    gen = torch.Generator("cuda").manual_seed(cfg["seed"])
    for _ in range(30):
        acts = torch.randint(0, 4, (n_envs,), dtype=torch.int32, device="cuda", generator=gen)
        oa, ra, da, _ = a.step(acts)
        ob, rb, db, _ = b.step(acts)
        assert ob.dtype == dtype and torch.equal(oa.to(dtype), ob) and torch.equal(ra, rb) and torch.equal(da, db)
    assert torch.equal(a.observe().to(dtype), b.observe())
    acts = torch.randint(0, 4, (8, n_envs), dtype=torch.int32, device="cuda", generator=gen)
    (oa, ra, da), (ob, rb, db) = a.rollout(8, actions=acts), b.rollout(8, actions=acts)
    assert ob.dtype == dtype and torch.equal(oa.to(dtype), ob) and torch.equal(ra, rb) and torch.equal(da, db)
    for _ in range(5):
        h = torch.randint(0, 4, (n_envs,), dtype=torch.int32, generator=torch.Generator().manual_seed(5)).numpy()
        oa, ra, da, _ = a.step_host(h)
        ob, rb, db, _ = b.step_host(h)
        assert torch.equal(torch.as_tensor(oa).to(dtype), torch.as_tensor(ob)) and (ra == rb).all() and (da == db).all()


@pytest.mark.parametrize("cfg,n_envs,packed", [(dict(width=14, height=14, seed=501), 16, "1"), (dict(width=14, height=14, seed=502), 33, "1"),
                                               (dict(width=10, height=10, seed=503), 7, "1"), (dict(width=32, height=32, seed=504), 5, "1"),
                                               (dict(width=17, height=13, seed=505, wind="random"), 9, "1"),
                                               (dict(width=14, height=14, seed=506), 16, "0"), (dict(width=40, height=36, seed=507), 6, "1"),
                                               (dict(width=14, height=14, seed=508), 601, "1"), (dict(width=20, height=20, seed=509), 530, "1"),
                                               (dict(width=14, height=14, seed=510), 77, "1+graph"), (dict(width=32, height=30, seed=511), 9, "1+graph"),
                                               (dict(width=14, height=14, seed=512), 40, "direct")],
                         ids=["14_even", "14_odd", "10", "32", "17x13", "14_unpacked", "tile_40x36", "14_n601", "20_n530",
                              "14_graph", "32x30_graph", "14_direct"])
def test_step_host_roundtrip(monkeypatch, cfg, n_envs, packed):
    """wf_step_host with page-locked host buffers: the packed path (observation bit stream into mapped host
    memory + host-thread expansion, grids up to 32x32; "+graph": kernel + copy as one CUDA graph, WF_HOST_GRAPH=1;
    "direct": the kernel stores the stream straight into mapped host memory), the plain uint8 path (WF_HOST_PACKED=0)
    and the tile family."""
    if packed.endswith("+graph"):
        packed = packed[:-6]
        monkeypatch.setenv("WF_HOST_GRAPH", "1")
    monkeypatch.setenv("WF_HOST_PACKED", packed)
    monkeypatch.setenv("WF_HOST_THREADS", "3")
    gpu, orc = make_pair(n_envs, cfg)
    gpu.reset()
    for e in orc:
        e.reset()
    for s in range(40):
        acts = np.array([e.random_action() for e in orc], np.int32)
        obs, rew, done, _ = gpu.step_host(acts)
        for i, e in enumerate(orc):
            if not e.planes()["running"]:
                continue
            o, r, d, _ = e.step(int(acts[i]))
            assert rew[i] == r and bool(done[i]) == d and np.array_equal(obs[i], o), (s, i)
    want_threads = 3 if (packed != "0" and max(cfg["width"], cfg["height"]) <= 32) else 0
    assert gpu.host_threads == want_threads


def test_set_state_free_burn_known_answer():
    """SURVEY.md Appendix C: 14x14 free burn, agent parked at (7, 10): done at tick 185, nothing left."""
    from wildfire_control_python_b200.batched import BatchedForestFire
    gpu = BatchedForestFire(2, width=14, height=14, seed=0)
    gpu.reset(starts=torch.tensor([[7, 10], [7, 10]], dtype=torch.int32))
    noop = torch.full((2,), 5, dtype=torch.int32, device="cuda")
    t = 0
    while True:
        _, rew, done, _ = gpu.step(noop)
        t += 1
        if bool(done[0]):
            break
        assert float(rew[0]) == -1.0
    assert t == 185
    st = gpu.get_state()
    assert int((st["type"][0] == 0).sum()) == 0
    assert float(rew[0]) == 0.0


def test_errors_are_reported_not_thrown():
    from wildfire_control_python_b200.batched import BatchedForestFire
    L = _lib()
    with pytest.raises(L.WildfireError, match="radius"):
        BatchedForestFire(1, width=10, height=10, radius=2)
    with pytest.raises(L.WildfireError, match=">= 10"):
        BatchedForestFire(1, width=8, height=8)
    with pytest.raises(L.WildfireError, match="HEIGHT-1"):
        BatchedForestFire(1, width=10, height=12)


def test_trajectories_do_not_depend_on_sharding():
    """Two handles with env_id_base 0 / 16 (16 envs each) == one handle with 32 envs."""
    from wildfire_control_python_b200.batched import BatchedForestFire
    cfg = dict(width=14, height=14, seed=901, wind="random", auto_reset=True)
    whole = BatchedForestFire(32, **cfg)
    lo = BatchedForestFire(16, env_id_base=0, **cfg)
    hi = BatchedForestFire(16, env_id_base=16, **cfg)
    o = whole.reset()
    assert torch.equal(o[:16], lo.reset()) and torch.equal(o[16:], hi.reset())
    ow, rw, dw = whole.rollout(200)
    ol, rl, dl = lo.rollout(200)
    oh, rh, dh = hi.rollout(200)
    assert torch.equal(ow[:, :16], ol) and torch.equal(ow[:, 16:], oh)
    assert torch.equal(rw[:, :16], rl) and torch.equal(rw[:, 16:], rh)
    assert torch.equal(dw[:, :16], dl) and torch.equal(dw[:, 16:], dh)
    a, b, c = whole.stats(), lo.stats(), hi.stats()
    assert all(a[k] == b[k] + c[k] for k in a)


@pytest.mark.parametrize("policy", ["mlp", "walk"])
def test_device_policies_do_not_depend_on_sharding(policy):
    """BASELINE configs[2] shards 65 536 envs over 8 GPUs with the policy evaluated inside the step kernel: every env's
    trajectory (actions, rewards, dones, observations) must be the same whichever shard -- and whichever GPU, when the
    box has more than one -- it lands on.  Uneven shards, so that the warp packing (two envs per warp) differs too."""
    from wildfire_control_python_b200.batched import BatchedForestFire
    cfg = dict(width=14, height=14, seed=905, auto_reset=True)
    n_dev = torch.cuda.device_count()
    cuts = [0, 21, 42, 64]
    whole = BatchedForestFire(64, device="cuda:0", **cfg)
    shards = [BatchedForestFire(cuts[i + 1] - cuts[i], env_id_base=cuts[i], device=f"cuda:{i % n_dev}", **cfg) for i in range(3)]
    envs = [whole] + shards
    if policy == "mlp":
        g = torch.Generator().manual_seed(5)
        w1, b1 = torch.randn(588, 50, generator=g) * 0.3, torch.randn(50, generator=g) * 0.1
        w2, b2 = torch.randn(50, 4, generator=g) * 0.5, torch.randn(4, generator=g) * 0.1
        for e in envs:
            e.set_policy_mlp(w1, b1, w2, b2, eps=0.1)
    obs0 = [e.reset() for e in envs]
    for i, sh in enumerate(shards):
        assert torch.equal(obs0[0][cuts[i]:cuts[i + 1]].cpu(), obs0[1 + i].cpu())
    for _ in range(3):  # three launches: the policy's state (episode, step, hidden pre-activations) carries over
        outs = [e.rollout(70, policy=policy, return_actions=True) for e in envs]
        for i, sh in enumerate(shards):
            for j in range(4):  # obs, reward, done, actions
                assert torch.equal(outs[0][j][:, cuts[i]:cuts[i + 1]].cpu(), outs[1 + i][j].cpu()), (policy, i, j)
    assert int(outs[0][2].sum()) > 0  # episodes ended and were reset inside the kernel
    tot = whole.stats()
    parts = [sh.stats() for sh in shards]
    assert all(tot[k] == sum(p[k] for p in parts) for k in tot)


def _tile_geometry_case(monkeypatch, T, CS, cfg):
    monkeypatch.setenv("WF_TILE_T", str(T))
    monkeypatch.setenv("WF_TILE_CS", str(CS))
    N, K = 5, 150
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    obs0 = gpu.reset()
    for e in orc:
        e.reset()
    compare_states("reset", gpu, orc, obs=obs0)
    for policy in ("walk", "stream"):
        obs, rew, done, acts = gpu.rollout(K, policy=policy, return_actions=True)
        obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
        for i, e in enumerate(orc):
            for k in range(K):
                a = e.walk_action() if policy == "walk" else e.random_action()
                assert acts[k, i] == a, f"{policy} env {i} step {k}: action"
                o, r, d, _ = e.step(a)
                assert rew[k, i] == r and bool(done[k, i]) == d, f"{policy} env {i} step {k}: reward/done {rew[k, i]} {r}"
                if d:
                    o = e.reset()
                assert np.array_equal(obs[k, i], o), f"{policy} env {i} step {k}: obs"
        compare_states(f"after {policy} rollout", gpu, orc)


@pytest.mark.parametrize("T,CS", [(128, 1), (128, 2), (256, 4), (128, 8), (512, 2)])
@pytest.mark.parametrize("cfg", [dict(width=64, height=64, seed=701, make_rivers=True, wind="random", extra_ignitions=3),
                                 dict(width=100, height=70, seed=702, wind=[0.85, (1, 0)], extra_ignitions=6, a_speed=2),
                                 dict(width=128, height=128, seed=703, allow_dig_toggle=True, n_actions=6, extra_ignitions=4)],
                         ids=["64_rivers", "100x70_aspeed2", "128_toggle"])
def test_tile_cluster_geometries_match_oracle(monkeypatch, T, CS, cfg):
    """The tile family splits one env over a thread-block cluster of CS CTAs x T threads (chosen from
    the batch size in production): every split must give the oracle's trajectory -- walk-policy
    rollout with auto-reset (containments, re-floods of the reach plane, in-kernel resets)."""
    _tile_geometry_case(monkeypatch, T, CS, cfg)


@pytest.mark.parametrize("T,CS", [(128, 1), (128, 2), (256, 4), (256, 1)])
@pytest.mark.parametrize("cfg", [dict(width=128, height=128, seed=711, allow_dig_toggle=True, n_actions=6, extra_ignitions=4),
                                 dict(width=128, height=128, seed=712, make_rivers=True, wind="random", a_speed=2, extra_ignitions=3),
                                 dict(width=256, height=128, seed=713, wind=[0.85, (1, 0)], extra_ignitions=9, fuel=40)],
                         ids=["128_toggle", "128_rivers_aspeed2", "256x128_wide_fuel40"])
def test_tile_whole_group_slices_match_oracle(monkeypatch, T, CS, cfg):
    """Grids whose CTA slices are whole 128-word groups, so the observation runs on the wide path alone: dig toggle,
    rivers with a_speed 2, and a W > H map with 8 fuel bit-slices.  Same check as the geometry sweep above."""
    _tile_geometry_case(monkeypatch, T, CS, cfg)


def test_burning_border_point_is_not_its_own_goal():
    """W > H: the reference's literal border points [HEIGHT-1, y] (environment.py:222) form a column INSIDE the
    map, and for 24x13 the fire origin (12, 6) sits on it.  pyastar.astar_path returns an empty path when
    start == goal (pyastar.py:53-62), so the walk policy's ring round the origin pays the containment bonus
    although the burning cell is a border point itself (found by tools/soak.py; the Python reference agrees
    with the oracle on this trajectory)."""
    cfg = dict(width=24, height=13, seed=387835340, wind=[0.54, (1, 1)], allow_dig_toggle=True, n_actions=6, a_speed=2,
               fuel=40, threshold=4.5)
    N, K = 21, 71
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    gpu.reset()
    for e in orc:
        e.reset()
    obs, rew, done, acts = gpu.rollout(K, policy="walk", return_actions=True)
    obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
    n_bonus = 0
    for i, e in enumerate(orc):
        for k in range(K):
            assert acts[k, i] == e.walk_action(), (i, k)
            o, r, d, _ = e.step(int(acts[k, i]))
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k, rew[k, i], r)
            n_bonus += int(r == 1000)
            if d:
                o = e.reset()
            assert np.array_equal(obs[k, i], o), (i, k)
    assert n_bonus >= 1
    compare_states("end", gpu, orc)


def test_burning_border_point_is_a_goal_for_other_burning_cells():
    """Second W > H case from tools/soak.py (17x10, rivers): the fire reaches the interior border-point column
    x = 9, the agent seals the pocket, and the burning cell on that column is still reachable from the other
    burning cells through burnt cells -> no containment bonus."""
    cfg = dict(width=17, height=10, seed=1034441046, wind=[0.7, (0, 0)], make_rivers=True, allow_dig_toggle=True, n_actions=6)
    N, K = 27, 173
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    gpu.reset()
    for e in orc:
        e.reset()
    obs, rew, done, acts = gpu.rollout(K, policy="walk", return_actions=True)
    obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
    for i, e in enumerate(orc):
        for k in range(K):
            assert acts[k, i] == e.walk_action(), (i, k)
            o, r, d, _ = e.step(int(acts[k, i]))
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k, rew[k, i], r)
            if d:
                o = e.reset()
            assert np.array_equal(obs[k, i], o), (i, k)
    compare_states("end", gpu, orc)


@pytest.mark.parametrize("T,CS", [(0, 0), (128, 16), (256, 2)])
def test_tile_burning_border_point_sealed_in_a_pocket(monkeypatch, T, CS):
    """Third W > H case from tools/soak.py (70x33, wind blowing the fire onto the interior border-point column
    x = 32 inside the agent's ring): the only border point of the pocket is the burning cell itself, so the
    reference pays the containment bonus.  Tile family: needs the scratch flood from the cold border points."""
    monkeypatch.setenv("WF_TILE_T", str(T))
    monkeypatch.setenv("WF_TILE_CS", str(CS))
    cfg = dict(width=70, height=33, seed=359706589, wind="random")
    N, K = 3, 87
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    gpu.reset()
    for e in orc:
        e.reset()
    obs, rew, done, acts = gpu.rollout(K, policy="walk", return_actions=True)
    obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
    n_bonus = 0
    for i, e in enumerate(orc):
        for k in range(K):
            assert acts[k, i] == e.walk_action(), (i, k)
            o, r, d, _ = e.step(int(acts[k, i]))
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k, rew[k, i], r)
            n_bonus += int(r == 1000)
            if d:
                o = e.reset()
            assert np.array_equal(obs[k, i], o), (i, k)
    assert n_bonus >= 1
    compare_states("end", gpu, orc)


@pytest.mark.parametrize("T,CS", [(256, 2), (128, 1), (512, 2)])
def test_tile_slices_with_a_tail_emit_clean_observations(monkeypatch, T, CS):
    """130x128 over a cluster of 2: each CTA's slice is a few 128-word groups plus a tail that takes the narrow
    observation path; the two paths stage in shared memory at the same time (race found by tools/soak.py)."""
    monkeypatch.setenv("WF_TILE_T", str(T))
    monkeypatch.setenv("WF_TILE_CS", str(CS))
    cfg = dict(width=130, height=128, seed=667898885, make_rivers=True)
    N = 5
    gpu, orc = make_pair(N, cfg, auto_reset=True)
    for rep in range(4):
        obs = to_np(gpu.reset())
        for i, e in enumerate(orc):
            assert np.array_equal(obs[i], e.reset()), (rep, i)
    obs, rew, done, acts = gpu.rollout(40, policy="walk", return_actions=True)
    obs, rew, done, acts = to_np(obs), to_np(rew), to_np(done), to_np(acts)
    for i, e in enumerate(orc):
        for k in range(40):
            o, r, d, _ = e.step(int(acts[k, i]))
            assert rew[k, i] == r and bool(done[k, i]) == d, (i, k)
            if d:
                o = e.reset()
            assert np.array_equal(obs[k, i], o), (i, k)
