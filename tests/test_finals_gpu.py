"""Final-state capture (wf_set_final_capture, ``rollout(finals=True)``): every record written by the step kernels of both
families against the C oracle stepped through the same episodes with the recorded actions -- type planes, agent, flags,
terminal observation, the next episode's start cell and the rendered map -- plus records without auto-reset, the overflow
error, and the check that capture changes nothing else a launch returns."""
import numpy as np
import pytest
import torch

from oracle import wf_oracle as wo
from tests.gpu_util import to_np
from wildfire_control_python_b200 import _lib
from wildfire_control_python_b200.batched import BatchedForestFire, unpack_obs
from wildfire_control_python_b200.constants import ascii_of_type

pytestmark = pytest.mark.gpu


def _oracle_render(p):
    """ForestFire.render(print_map=False) of an oracle state (forest_fire.py:57-82)."""
    W, H = p["type"].shape
    rows = ["".join("A" if p["alive"] and (x, y) == (p["ax"], p["ay"]) else ascii_of_type[int(p["type"][x, y])]
                    for x in range(W)) for y in range(H)]
    return "\n" + "\n".join(rows) + "\n"


def _net(W, H, n_actions, hidden=32, seed=0):
    rng = np.random.default_rng(seed)
    n_in = W * H * 3
    k1 = rng.uniform(-1, 1, (n_in, hidden)) * np.sqrt(6.0 / (n_in + hidden))
    k1[0::3] *= 40.0
    return [x.astype(np.float32) for x in (k1, rng.uniform(-1, 1, hidden), rng.uniform(-1, 1, (hidden, n_actions)),
                                           rng.uniform(-0.1, 0.1, n_actions))]


def _check_launch(tag, env, orc, K, fin, rew, done, acts, ep0, cfg):
    """Step the oracles through one launch with its actions and compare every record at its done step."""
    W, H = env.width, env.height
    rew, done, acts = to_np(rew), to_np(done), to_np(acts)
    keys = list(zip(to_np(fin.k).tolist(), to_np(fin.env).tolist()))
    assert keys == sorted(keys), f"{tag}: records not in (k, env) order"
    assert set(keys) == {(int(k), int(n)) for k, n in zip(*np.nonzero(done))}, f"{tag}: records != done flags"
    where = {key: i for i, key in enumerate(keys)}
    hdr = to_np(fin.records[:, :_lib.FINAL_HEADER_WORDS])
    types = to_np(fin.types())
    obs = to_np(fin.obs) if not env.obs_bits else None
    for k in range(K):
        for n, e in enumerate(orc):
            o, r, d, _ = e.step(int(acts[k, n]))
            assert r == rew[k, n] and d == bool(done[k, n]), f"{tag}: trajectory k={k} env={n}"
            if not d:
                continue
            i = where[(k, n)]
            t = f"{tag}: record k={k} env={n}"
            p = e.planes()
            s = e.scalars()
            assert np.array_equal(types[i], p["type"]), f"{t}: types\n{types[i].T}\n{p['type'].T}"
            assert bool(fin.alive[i]) == bool(p["alive"]) and bool(fin.dead[i]) == bool(s[3]), f"{t}: alive / dead"
            assert bool(fin.digging[i]) == bool(s[4]), f"{t}: digging"
            assert bool(fin.visible[i]) == bool(p["apos"].any()), f"{t}: visible"
            if p["alive"]:
                assert tuple(hdr[i, [_lib.F_AX, _lib.F_AY]]) == (p["ax"], p["ay"]), f"{t}: agent"
            assert hdr[i, _lib.F_T] == s[9], f"{t}: episode length"
            assert hdr[i, _lib.F_EPISODE] == ep0[n], f"{t}: episode number"
            ep0[n] += 1
            if env.obs_bits:
                got = to_np(unpack_obs(fin.obs[i:i + 1].contiguous(), W, H, dtype=torch.uint8))[0]
            else:
                got = obs[i]
            assert np.array_equal(got, o), f"{t}: terminal observation"
            assert fin.render(i) == _oracle_render(p), f"{t}: render\n{fin.render(i)}\n{_oracle_render(p)}"
            if p["alive"] and not p["burning"].any():  # burn-out: the reward counts the grass cells
                grass = int((types[i] == 0).sum())
                assert r == cfg.get("contained_bonus", 1000) * (grass / (W * H)), f"{t}: burn-out reward"
            if s[3]:
                assert not bool(fin.alive[i]), f"{t}: a dead agent is alive"
            if env.METADATA["auto_reset"]:
                e.reset()
                s2 = e.scalars()
                assert tuple(to_np(fin.next_start[i]).tolist()) == (s2[1], s2[2]), f"{t}: next start"
            else:
                assert tuple(to_np(fin.next_start[i]).tolist()) == (-1, -1), f"{t}: next start without auto_reset"
    return len(keys)


def _run_policy(tag, env, orc, cfg, K, launches, policy):
    env.reset()
    for e in orc:
        e.reset()
    ep0 = to_np(env.get_state()["scalars"][:, _lib.S_EPISODE]).tolist()
    total = 0
    for j in range(launches):
        _, rew, done, acts, fin = env.rollout(K, policy=policy, return_actions=True, finals=True, obs=False)
        total += _check_launch(f"{tag} launch {j}", env, orc, K, fin, rew, done, acts, ep0, cfg)
    return total


@pytest.mark.parametrize("policy,n,W,H", [("stream", 4096, 14, 14), ("walk", 1024, 14, 14), ("mlp", 1024, 14, 14),
                                           ("stream", 512, 32, 32), ("mlp", 512, 32, 32), ("walk", 512, 24, 20)])
def test_warp_records_match_the_oracle(policy, n, W, H):
    """14x14: two envs per warp (16 lanes each); 32x32 and 24x20: one env per warp, 32 lanes, rows of more than 16 cells."""
    cfg = dict(width=W, height=H, seed=5, wind="random", make_rivers=True)
    env = BatchedForestFire(n, auto_reset=True, **cfg)
    orc = [wo.OracleEnv(cfg, env_id=i) for i in range(n)]
    if policy == "mlp":
        env.set_policy_mlp(*_net(W, H, env.n_actions), eps=0.3)
    total = _run_policy(f"warp {W}x{H} {policy}", env, orc, cfg, 16 if W == 14 else 40, 3, policy)
    assert total > 0


def test_warp_bits_observation_and_step():
    cfg = dict(width=12, height=10, seed=2)
    n = 256
    env = BatchedForestFire(n, auto_reset=True, obs_dtype="bits", **cfg)
    orc = [wo.OracleEnv(cfg, env_id=i) for i in range(n)]
    assert _run_policy("warp bits", env, orc, cfg, 24, 2, "stream") > 0
    # step(finals=True): info["final"]
    ep0 = to_np(env.get_state()["scalars"][:, _lib.S_EPISODE]).tolist()
    seen = 0
    for s in range(30):
        acts = torch.tensor([e.random_action() for e in orc], dtype=torch.int32, device="cuda")
        _, rew, done, info = env.step(acts, finals=True)
        fin = info["final"]
        seen += _check_launch(f"step {s}", env, orc, 1, fin, rew[None].clone(), done[None].clone(), acts[None], ep0, cfg)
    assert seen > 0


@pytest.mark.parametrize("W,H,n,K,geoms", [(48, 48, 64, 40, [(128, 1), (256, 2)]), (40, 20, 64, 40, [(128, 1), (128, 2)]),
                                           (128, 128, 16, 60, [(256, 4), (512, 1)])])
def test_tile_records_match_the_oracle_and_do_not_depend_on_geometry(monkeypatch, W, H, n, K, geoms):
    cfg = dict(width=W, height=H, seed=11, extra_ignitions=4, wind="random", make_rivers=True)
    recs = []
    for T, CS in geoms:
        monkeypatch.setenv("WF_TILE_T", str(T))
        monkeypatch.setenv("WF_TILE_CS", str(CS))
        env = BatchedForestFire(n, auto_reset=True, **cfg)
        assert env.kernel_family == "tile" and env.tile_geometry == (T, CS)
        if not recs:
            orc = [wo.OracleEnv(cfg, env_id=i) for i in range(n)]
            env.reset()
            for e in orc:
                e.reset()
            ep0 = to_np(env.get_state()["scalars"][:, _lib.S_EPISODE]).tolist()
            got = []
            for j in range(2):
                _, rew, done, acts, fin = env.rollout(K, policy="walk" if j else "stream", return_actions=True, finals=True)
                _check_launch(f"tile {W}x{H} launch {j}", env, orc, K, fin, rew, done, acts, ep0, cfg)
                got.append(to_np(fin.records))
        else:
            env.reset()
            got = [to_np(env.rollout(K, policy="walk" if j else "stream", finals=True, obs=False)[-1].records) for j in range(2)]
        recs.append(got)
        env.close()
    for a, b in zip(recs[0], recs[1]):
        assert np.array_equal(a, b), "records differ across tile geometries"
    if (W, H) == (48, 48):
        assert sum(len(r) for r in recs[0]) > 0


@pytest.mark.parametrize("W,H", [(14, 14), (48, 40)])
def test_without_auto_reset_one_record_per_env_at_its_done_step(W, H):
    cfg = dict(width=W, height=H, seed=4, extra_ignitions=2)
    n, K = 64, 120
    env = BatchedForestFire(n, auto_reset=False, **cfg)
    env.reset()
    _, rew, done, fin = env.rollout(K, finals=True, obs=False)
    done = to_np(done)
    first = {int(n_): int(np.argmax(done[:, n_])) for n_ in range(n) if done[:, n_].any()}
    assert {(k, e) for e, k in first.items()} == set(zip(to_np(fin.k).tolist(), to_np(fin.env).tolist()))
    st = env.get_state()
    sc = to_np(st["scalars"])
    for i, e in enumerate(to_np(fin.env).tolist()):
        assert np.array_equal(to_np(fin.types()[i]), to_np(st["type"][e])), f"env {e}: types"
        assert bool(fin.alive[i]) == bool(sc[e, _lib.S_ALIVE]) and bool(fin.dead[i]) == bool(sc[e, _lib.S_DEAD])
        assert bool(fin.visible[i]) == bool(sc[e, _lib.S_VISIBLE]) and bool(fin.digging[i]) == bool(sc[e, _lib.S_DIGGING])
        if sc[e, _lib.S_ALIVE]:
            assert tuple(to_np(fin.agent[i]).tolist()) == (sc[e, _lib.S_AX], sc[e, _lib.S_AY])
        assert int(fin.t[i]) == sc[e, _lib.S_T] and int(fin.episode[i]) == sc[e, _lib.S_EPISODE]
        assert tuple(to_np(fin.next_start[i]).tolist()) == (-1, -1)
    obs_now = to_np(env.observe())
    assert np.array_equal(to_np(fin.obs), obs_now[to_np(fin.env)])
    # a second launch: frozen envs never record again
    _, _, _, fin2 = env.rollout(8, finals=True, obs=False)
    assert not set(to_np(fin2.env).tolist()) & set(first)


@pytest.mark.parametrize("W", [14, 48])
def test_overflow_raises_with_the_true_count(W):
    cfg = dict(width=W, height=W, seed=6)
    n = 256 if W == 14 else 32
    a = BatchedForestFire(n, auto_reset=True, **cfg)
    b = BatchedForestFire(n, auto_reset=True, **cfg)
    a.reset()
    b.reset()
    K = 60
    _, _, done_b, fin_b = b.rollout(K, finals=True, obs=False)
    n_done = int(to_np(done_b).sum())
    assert n_done > 2
    with pytest.raises(_lib.WildfireError, match=f"{n_done} episodes ended in this call but finals_capacity is 2"):
        a.rollout(K, finals=True, finals_capacity=2, obs=False)
    # the same env afterwards, with ample capacity: unaffected
    _, _, _, fa = a.rollout(10, finals=True, obs=False)
    _, _, _, fb = b.rollout(10, finals=True, obs=False)
    assert np.array_equal(to_np(fa.records), to_np(fb.records))


@pytest.mark.parametrize("W,policy", [(14, "stream"), (14, "walk"), (14, "mlp"), (48, "stream"), (48, "mlp")])
def test_capture_changes_nothing_else(W, policy):
    cfg = dict(width=W, height=W, seed=8, extra_ignitions=1)
    n = 512 if W == 14 else 32
    envs = [BatchedForestFire(n, auto_reset=True, **cfg) for _ in range(2)]
    for env in envs:
        env.reset()
        if policy == "mlp":
            env.set_policy_mlp(*_net(W, W, env.n_actions, seed=3), eps=0.2)
    for j in range(3):
        a = envs[0].rollout(20, policy=policy, return_actions=True)
        b = envs[1].rollout(20, policy=policy, return_actions=True, finals=True)
        for x, y in zip(a, b[:4]):
            assert torch.equal(x, y), f"launch {j}: capture changed an output"
    assert envs[0].stats() == envs[1].stats()
    st0, st1 = envs[0].get_state(), envs[1].get_state()
    for k in ("type", "burning", "fm_inf", "fuel", "hits", "scalars"):
        assert torch.equal(st0[k], st1[k]), k


def test_host_step_refused_while_capture_is_on():
    env = BatchedForestFire(16, width=10, height=10, seed=1)
    env.reset()
    L = _lib.lib()
    buf = torch.empty((16, _lib.final_record_words(10, 10)), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.wf_set_final_capture(env._h, buf.data_ptr(), 16, cnt.data_ptr()))
    try:
        with pytest.raises(_lib.WildfireError, match="final-state capture"):
            env.step_host(np.zeros(16, np.int32))
        assert L.wf_host_session(env._h, 1) == _lib.WF_ERR_STATE
    finally:
        _lib.check(L.wf_set_final_capture(env._h, None, 0, None))
    env.step_host(np.zeros(16, np.int32))


# ---------------------------------------------------------------------------------------------------------------------
# the learners' maps / agent_pos logs (record_maps=True)
from tests.test_learn_gpu import _Sim, _agent  # noqa: E402
from tests.test_population_gpu import _state  # noqa: E402
from tests.test_resume_gpu import _resume_until_done  # noqa: E402
from wildfire_control_python_b200 import agents as A  # noqa: E402

ASCII = set("+@#0xA")


def _host_maps(rewards, best=-10000):
    """DQN.py:120-148's map rule on a list of returns: the indices of the episodes it renders, and the best return."""
    idx = []
    for i, r in enumerate(rewards):
        if r >= 0.9 * best or r > 300:
            idx.append(i)
            best = max(best, r)
    return idx, best


def _check_map_logs(ag, W, H, n_ep):
    idx, best = _host_maps(ag.logs["total_rewards"])
    assert [m[0] for m in ag.logs["maps"]] == idx and ag.logs["best_reward"] == best
    for _, m in ag.logs["maps"]:
        rows = m.split("\n")[1:-1]
        assert m[0] == "\n" and len(rows) == H and all(len(r) == W and set(r) <= ASCII for r in rows)
        assert m.count("A") <= 1
    if ag._SARSA:
        assert ag.logs["agent_pos"] == []
    else:
        assert len(ag.logs["agent_pos"]) == n_ep
        assert all(0 <= x < W and 0 <= y < H for x, y in ag.logs["agent_pos"])


@pytest.mark.parametrize("name,W,n_envs,n_ep", [("DQN", 14, 512, 400), ("DQN_SARSA", 14, 512, 400), ("DQN_DUEL", 48, 64, 40)])
def test_learn_batched_record_maps_is_an_output_only(name, W, n_envs, n_ep, tmp_path):
    runs = []
    for rm in (False, True):
        ag = _agent(name, W, W, seed=1)
        ag.out_dir = str(tmp_path / str(rm))
        runs.append((ag, ag.learn_batched(n_ep, n_envs=n_envs, k_steps=16, seed=3, record_maps=rm)))
    (a, sa), (b, sb) = runs
    assert sa == sb and _state(a) == _state(b) and a._until_sync == b._until_sync
    for key in ("total_rewards", "agent_deaths", "n_episodes"):
        assert a.logs[key] == b.logs[key], key
    assert a.logs["maps"] == [] and a.logs["agent_pos"] == []
    _check_map_logs(b, W, W, n_ep)
    assert len(b.logs["maps"]) > 0


def test_learn_population_record_maps_equals_each_learner_alone(tmp_path):
    W, G, K, n_ep, seed = 14, 64, 16, 150, 4

    def make(j, out, **kw):
        torch.manual_seed(j)
        ag = A.DQN(_Sim(W, W, **kw), verbose=False, device="cuda")
        ag.out_dir = str(out)
        return ag

    pop = [make(j, tmp_path / "pop") for j in range(2)]
    A.learn_population(pop, n_ep, envs_per_learner=G, k_steps=K, seed=seed, record_maps=True)
    for j in range(2):
        solo = make(j, tmp_path / f"solo{j}", env_id_base=j * G)
        solo.learn_batched(n_ep, n_envs=G, k_steps=K, seed=seed, replay_seed=seed + j, record_maps=True)
        for key in ("total_rewards", "agent_deaths", "maps", "agent_pos", "best_reward"):
            assert pop[j].logs[key] == solo.logs[key], (j, key)
        _check_map_logs(pop[j], W, W, n_ep)


def test_learn_batched_record_maps_resumes_byte_identically(tmp_path):
    W, n_ep, kw = 14, 200, dict(n_envs=256, k_steps=16, seed=6, record_maps=True)

    def make(i, out):
        ag = _agent("DQN", W, W, seed=1 if i == 0 else 100 + i)
        ag.out_dir = str(out)
        return ag

    whole = make(0, tmp_path / "whole")
    whole.learn_batched(n_ep, **kw)
    path = tmp_path / "run.ckpt"
    ag, _, stops = _resume_until_done(lambda i: make(i, tmp_path / "resumed"),
                                      lambda a: a.learn_batched(n_ep, checkpoint=path, time_limit=0, **kw), path)
    assert stops == len(whole.eps_per_launch) - 1 and stops > 0
    for key in ("total_rewards", "agent_deaths", "maps", "agent_pos", "best_reward"):
        assert ag.logs[key] == whole.logs[key], key
    assert _state(ag) == _state(whole)


def test_evaluate_batched_record_maps():
    ag = _agent("DQN", 14, 14, seed=2)
    ret, died = ag.evaluate_batched(n_envs=256, episodes_per_env=2, eps=0.2, seed=1, in_kernel=True)
    ret2, died2, maps = ag.evaluate_batched(n_envs=256, episodes_per_env=2, eps=0.2, seed=1, in_kernel=True, record_maps=True)
    assert np.array_equal(ret, ret2) and np.array_equal(died, died2) and len(maps) == len(ret)
    for m, d in zip(maps, died):
        rows = m.split("\n")[1:-1]
        assert len(rows) == 14 and all(len(r) == 14 and set(r) <= ASCII for r in rows)
        if d:
            assert "A" not in m
    with pytest.raises(ValueError, match="in_kernel"):
        ag.evaluate_batched(n_envs=64, in_kernel=False, record_maps=True)
