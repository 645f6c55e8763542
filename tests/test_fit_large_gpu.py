"""wf_replay_fit_large on the GPU (DQN.fit_batches_fused on grids larger than 32x32): against the torch fit_batch loop and
against wf_replay_fit, its determinism whatever the number of CTAs, its out-of-range rules, and learn_batched's use of it."""
import copy

import numpy as np
import pytest
import torch

from tests.test_learn_gpu import _agent, _flat, _random_replays, _warm
from wildfire_control_python_b200 import _lib, unpack_obs
from wildfire_control_python_b200 import agents as A

pytestmark = pytest.mark.gpu

BOUNDS = {"params": 1e-5, "target": 1e-5, "m": 2e-6, "v": 2e-7}
NAMES = ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"]


@pytest.fixture
def large_on_small_grids(monkeypatch):
    """fit_batches_fused runs wf_replay_fit_large on grids up to 32x32 too (it selects wf_replay_fit there)."""
    L = _lib.lib()
    monkeypatch.setattr(L, "wf_replay_fit", L.wf_replay_fit_large)


def _setup(name, W, H, B, R=64):
    ag = _agent(name, W, H, seed=W + H + B)
    n_frames = 4 * B
    data = _random_replays(ag, n_frames, R * B, seed=W * B + H)
    _warm(ag, data[0], n_frames, W * B)
    return ag, data


def _torch_loop(ag, data, R, phase):
    frames, s, sp, a, ap, r, d = data
    W, H = ag.obs_shape[0], ag.obs_shape[1]
    B = len(s) // R
    until, te = phase, ag.target_update_freq
    losses = []
    for i in range(R):
        sl = slice(B * i, B * i + B)
        losses.append(ag.fit_batch((unpack_obs(frames, W, H, s[sl], torch.uint8), a[sl], r[sl],
                                    unpack_obs(frames, W, H, sp[sl], torch.uint8), ap[sl], d[sl])))
        until -= 1
        if until == 0:
            until = te
            ag.target.load_state_dict(ag.model.state_dict())
    return np.array(losses), until


def _check_close(x, y, lx, ly):
    assert np.allclose(lx, ly, rtol=1e-3, atol=1e-5), np.abs(lx - ly).max()
    for what, p, q in zip(("params", "target", "m", "v"), _flat(x), _flat(y)):
        diff = np.abs(p - q)
        assert diff.max() <= BOUNDS[what], (what, diff.max(), int(diff.argmax()))


CASES = [(n, W, H, B) for n in NAMES for (W, H) in [(40, 40), (100, 70), (128, 128)] for B in (32, 256)]
CASES += [(n, 256, 256, 32) for n in ("DQN", "DQN_BOTH")]


@pytest.mark.parametrize("name,W,H,B", CASES)
def test_large_fit_matches_the_torch_loop(name, W, H, B):
    """64 replays in one launch against 64 fit_batch calls from the same warmed state (Adam t = 3, target != model), with
    target refreshes after replays 7, 27 and 47 (phase 7, target_update 20).  100x70 has 21000 inputs: its last
    observation word is partial.  Bounds as in test_learn_gpu.test_fused_replays_match_the_torch_loop."""
    R = 64
    ag, data = _setup(name, W, H, B, R)
    ref = copy.deepcopy(ag)
    ref_loss, until = _torch_loop(ref, data, R, 7)
    loss = ag.fit_batches_fused(*data, R, phase=7).cpu().numpy()
    assert ag._until_sync == until
    _check_close(ag, ref, loss, ref_loss)
    assert ag.optimizer.state[ag.model.dense_1.weight]["t"] == 3 + R


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("W,B", [(14, 32), (14, 256), (32, 32), (32, 256)])
def test_large_fit_matches_replay_fit(request, name, W, B):
    """The two kernels from the same state on grids both take: they sum in different orders, so they agree to the
    bounds of the torch comparison, not bit for bit."""
    R = 64
    ag, data = _setup(name, W, W, B, R)
    small = copy.deepcopy(ag)
    l_small = small.fit_batches_fused(*data, R, phase=7).cpu().numpy()
    request.getfixturevalue("large_on_small_grids")
    l_large = ag.fit_batches_fused(*data, R, phase=7).cpu().numpy()
    assert ag._until_sync == small._until_sync
    _check_close(ag, small, l_large, l_small)


@pytest.mark.parametrize("name,W,H", [("DQN_BOTH", 100, 70), ("DQN_SARSA", 48, 48)])
def test_large_fit_does_not_depend_on_the_number_of_ctas(monkeypatch, name, W, H):
    """Two calls are bit-identical, and so are calls forced to 1 and 7 CTAs (WF_FIT_CTAS): params, target, m, v and loss."""
    R, B = 16, 32
    ag, data = _setup(name, W, H, B, R)
    runs = []
    for ctas in (None, None, "1", "7"):
        if ctas is None:
            monkeypatch.delenv("WF_FIT_CTAS", raising=False)
        else:
            monkeypatch.setenv("WF_FIT_CTAS", ctas)
        x = copy.deepcopy(ag)
        loss = x.fit_batches_fused(*data, R, phase=5).cpu().numpy()
        runs.append([loss] + _flat(x))
    for other in runs[1:]:
        for p, q in zip(runs[0], other):
            assert p.tobytes() == q.tobytes()


def test_large_fit_out_of_range_rows_and_actions():
    """On 40x40: rows outside the frames are all-zero observations; a next action outside [0, A) bootstraps nothing (as
    if done); an action outside [0, A) replaces no target entry (the torch update with that sample's target =
    Q_target(s))."""
    B, W = 32, 40
    ag = _agent("DQN_SARSA", W, W, seed=5)
    frames, s, sp, a, ap, r, d = _random_replays(ag, 64, B, seed=6)
    _warm(ag, frames, 64, 6)
    zero_frames = torch.cat([frames, torch.zeros_like(frames[:1])])
    bad = torch.arange(B, device="cuda") % 4 == 0
    x, y = copy.deepcopy(ag), copy.deepcopy(ag)
    x.fit_batches_fused(frames, torch.where(bad, -5, s), torch.where(bad, 10**9, sp), a, ap, r, d, 1)
    y.fit_batches_fused(zero_frames, torch.where(bad, 64, s), torch.where(bad, 64, sp), a, ap, r, d, 1)
    for p, q in zip(_flat(x), _flat(y)):
        assert p.tobytes() == q.tobytes()
    x, y = copy.deepcopy(ag), copy.deepcopy(ag)
    x.fit_batches_fused(frames, s, sp, a, torch.where(bad, 99, ap), r, d, 1)
    y.fit_batches_fused(frames, s, sp, a, ap, r, d | bad, 1)
    for p, q in zip(_flat(x), _flat(y)):
        assert p.tobytes() == q.tobytes()
    x, ref = copy.deepcopy(ag), copy.deepcopy(ag)
    lx = float(x.fit_batches_fused(frames, s, sp, torch.where(bad, -1, a), ap, r, d, 1)[0])
    su, spu = unpack_obs(frames, W, W, s, torch.float32), unpack_obs(frames, W, W, sp, torch.float32)
    tgt = ref.replay_targets((su, a, r, spu, ap, d))
    with torch.no_grad():
        tgt[bad] = ref.target(su[bad])
    loss = torch.nn.functional.mse_loss(ref.model(su), tgt)
    ref.optimizer.zero_grad(set_to_none=True)
    loss.backward()
    ref.optimizer.step()
    assert lx == pytest.approx(float(loss), rel=1e-4)
    assert np.abs(_flat(x)[0] - _flat(ref)[0]).max() < 1e-5


def test_learn_batched_on_a_tile_grid_replays_only_in_the_kernel(monkeypatch, tmp_path):
    """learn_batched on 40x40 with DQN.fit_batch made to raise: the run replays (through wf_replay_fit_large), its
    weights move away from the initial ones, and two runs with one seed give the same weights."""
    def no_torch_replays(self, batch):
        raise AssertionError("learn_batched replayed through fit_batch")

    monkeypatch.setattr(A.DQN, "fit_batch", no_torch_replays)

    def run():
        ag = _agent("DQN", 40, 40, seed=1)
        ag.out_dir = str(tmp_path)
        init = torch.nn.utils.parameters_to_vector(ag.model.parameters()).detach().cpu().numpy()
        ag.collect_memories_batched(4, n_envs=64, k_steps=64, seed=2)
        assert len(ag.memory) > ag.METADATA["batch_size"]  # so the first launch replays
        ag.learn_batched(40, n_envs=64, k_steps=8, replays_per_launch=4, seed=3)
        assert ag.optimizer.state[ag.model.dense_1.weight]["t"] == 4 * len(ag.eps_per_launch)
        return init, _flat(ag)

    init, w1 = run()
    _, w2 = run()
    assert not np.array_equal(init, w1[0])
    for x, y in zip(w1, w2):
        assert x.tobytes() == y.tobytes()
