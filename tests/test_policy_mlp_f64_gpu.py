"""WF_POLICY_MLP against float64: every action the in-kernel Q-network chooses, on the warp family (all six MLP
instantiations: 16 or 32 lanes per env x bit-sliced hits / non-uniform wind / fuel > 31) and on the tile family, through
all three refresh paths (set_policy_mlp, set_policy_mlp_dev, set_policy_mlp_flat_dev with four group networks).

Explored steps must follow the EXPLORE stream (philox.explore_draw); greedy steps must pick an action whose float64 Q
(tests/f64_ref.py, on the observation the policy saw; the full V + A - mean(A) of a dueling head) is within a margin of
the float64 maximum; and every reward, done flag and observation must equal the oracle's, driven with the chosen actions.

Margins come from each path's error model.  Warp: float64 first layer, then float32 (__expf, __fdividef, fmaf, shuffle
sums): 1e-5 * (max_a sum_j |w2[a, j] s_j| + max |b2|), some 100 float32 ulps of the largest magnitude summed.  Tile: the
first layer is exact in int64 fixed point on top of `base` (bias + the all-free map, summed in float64 and stored as
float32), the rest float64: the margin is what rounding base_j (|base_j| * 2^-24) and each of the at most 2WH + 1 weights
(2^-33) can move sigmoid(z_j), through max_a |w2[a, j]|, doubled, plus 1e-9.  Worst measured gap (float64 max - Q of the
chosen action) on a B200 (1000 W power limit): 0 on both families -- every one of about 30 800 warp and 2 000 tile greedy
steps chose the float64 argmax.  GAPS collects (case, family, worst gap, worst gap / margin, greedy steps) as the tests
run, for recalibrating.

The weights are generated to discriminate (f64_ref.policy_weights), and each case checks on the frames it observed that
switching off the units of any one lane, or of any one register slot, changes at least 2 % of the greedy actions, that
more than one greedy action occurs, and that with A = 8 an action >= 5 is among them."""
import numpy as np
import pytest
import torch

from oracle import philox
from tests import f64_ref as R
from tests.gpu_util import make_pair, to_np

pytestmark = pytest.mark.gpu

GAPS = []


class _Shape:
    def __init__(self, W, H, hid, A, duel):
        self.width, self.height, self.hidden, self.n_actions, self.dueling = W, H, hid, A, duel


def _sigmoid_moves(z, dz):
    """The most sigmoid can move when z moves by at most dz (elementwise)."""
    s = R.sigmoid(z)
    return np.maximum(np.abs(R.sigmoid(z + dz) - s), np.abs(R.sigmoid(z - dz) - s))


def _margins(family, parts, shape, x):
    """Per observation: how far the kernel's Q may lie from float64 (see the module docstring)."""
    w1, b1 = parts["w1"].astype(np.float64), parts["b1"].astype(np.float64)
    w2, b2 = parts["w2"].astype(np.float64), parts["b2"].astype(np.float64)
    z = x @ w1.T + b1
    s = R.sigmoid(z)
    if family == "warp":
        return 1e-5 * ((s[:, None, :] * np.abs(w2)[None]).sum(-1).max(-1) + np.abs(b2).max())
    W, H = shape.width, shape.height
    base = b1 + w1[:, 2::3].sum(axis=1)
    dz = np.abs(base) * 2.0 ** -24 + (2 * W * H + 1) * 2.0 ** -33
    return 2.0 * (_sigmoid_moves(z, dz[None]) * np.abs(w2).max(axis=0)[None]).sum(-1) + 1e-9


def _set(gpu, path, nets, shape, eps):
    if path == "flat":
        gpu.set_policy_mlp_flat_dev(torch.from_numpy(np.stack(nets)).cuda(), shape.hidden, bool(shape.dueling), eps)
        return
    (net,), (e,) = nets, eps
    p = R.split(net, shape)
    if path == "host":
        gpu.set_policy_mlp(p["w1"].T.copy(), p["b1"], p["w2"].T.copy(), p["b2"], eps=e)
    else:
        gpu.set_policy_mlp_dev(*(torch.from_numpy(np.ascontiguousarray(p[k])).cuda() for k in ("w1", "b1", "w2", "b2")), eps=e)


def _check(tag, cfg, nets, shape, eps, N, K, launches, auto_reset, path):
    """The rollout, step by step, against float64 Q, the EXPLORE stream and the oracle (nets[m] drives envs
    m * N / M ...).  Returns the number of episodes that ended."""
    W, H = cfg["width"], cfg["height"]
    family = "tile" if W > 32 or H > 32 else "warp"
    lanes = 32 if family == "tile" or W > 16 else 16
    M = len(nets)
    G = N // M
    gpu, orc = make_pair(N, cfg, auto_reset=auto_reset)
    A = gpu.n_actions
    _set(gpu, path, nets, shape, eps)
    obs0 = to_np(gpu.reset())
    for e in orc:
        e.reset()
    outs = [gpu.rollout(K // launches, policy="mlp", return_actions=True) for _ in range(launches)]
    obs, rew, done, acts = (np.concatenate([to_np(o[j]) for o in outs]) for j in range(4))
    gpu.close()
    seen = np.concatenate([obs0[None], obs[:-1]]).reshape(K, N, -1)
    q, margin = np.empty((K, N, A)), np.empty((K, N))
    for m, net in enumerate(nets):
        x = seen[:, m * G:(m + 1) * G].reshape(-1, seen.shape[-1]).astype(np.float64)
        q[:, m * G:(m + 1) * G] = R.q_values(net, shape, x).reshape(K, G, A)
        margin[:, m * G:(m + 1) * G] = _margins(family, R.split(net, shape), shape, x).reshape(K, G)
    thr = [0xFFFFFFFF if e >= 1.0 else int(e * 4294967296.0) for e in eps]
    n_explored = n_greedy = n_ended = 0
    worst, worst_rel = 0.0, 0.0
    acted = np.zeros((K, N), bool)
    for i, e in enumerate(orc):
        episode, t, frozen = 0, 0, None
        for k in range(K):
            if frozen is not None:
                assert rew[k, i] == 0.0 and done[k, i] and np.array_equal(obs[k, i], frozen), (tag, i, k)
                continue
            acted[k, i] = True
            u0, u1 = philox.explore_draw(cfg["seed"], i, episode, t)
            a = int(acts[k, i])
            if u0 < thr[i // G]:
                assert a == u1 % A, (tag, i, k)
                n_explored += 1
            else:
                gap = q[k, i].max() - q[k, i, a] if 0 <= a < A else np.inf
                assert gap <= margin[k, i], (tag, i, k, a, q[k, i], margin[k, i])
                worst, worst_rel = max(worst, gap), max(worst_rel, gap / margin[k, i])
                n_greedy += 1
            o, r, d, _ = e.step(a)
            assert rew[k, i] == r and bool(done[k, i]) == d, (tag, i, k)
            t += 1
            if d:
                n_ended += 1
                if auto_reset:
                    o = e.reset()
                    episode, t = episode + 1, 0
                else:
                    frozen = o
            assert np.array_equal(obs[k, i], o), (tag, i, k)
    GAPS.append((tag, family, worst, worst_rel, n_greedy))
    if all(e >= 1.0 for e in eps):
        assert n_greedy == 0
    else:
        assert n_greedy > 0.4 * acted.sum()
    if all(e == 0.0 for e in eps):
        assert n_explored == 0
    # the weights discriminate on what the policy saw
    for m, net in enumerate(nets):
        x = seen[:, m * G:(m + 1) * G][acted[:, m * G:(m + 1) * G]]
        lane, slot, greedy = R.sensitivity(net, shape, x, lanes)
        assert R.discriminates(net, shape, x, lanes), (tag, m, lane, slot, greedy)
    return n_ended


def _nets(seed, W, H, hid, A, duel=0, M=1, lanes=16):
    return [R.policy_weights(seed + 7919 * m, W, H, hid, A, duel, lanes=lanes) for m in range(M)]


# (config, hidden, eps, launches, auto_reset, refresh path): L = 16 for W <= 16, else 32; the default wind is uniform
# with fuel 20 (bit-sliced hits), a directional or random wind is not, fuel 40 needs 8 fuel bits.
WARP = [
    (dict(width=10, height=10, seed=1), 1, 0.3, 2, True, "host"),
    (dict(width=16, height=10, seed=2, wind=[0.85, (1, 0)], n_actions=8), 16, 0.0, 3, True, "dev"),
    (dict(width=16, height=16, seed=3, fuel=40, allow_dig_toggle=True, n_actions=5, make_rivers=True, a_speed=2,
          extra_ignitions=2), 33, 0.3, 2, True, "host"),
    (dict(width=10, height=10, seed=4, fuel=40, wind="random", n_actions=7), 64, 1.0, 2, False, "dev"),
    (dict(width=16, height=16, seed=5), 64, 0.0, 2, False, "dev"),
    (dict(width=17, height=10, seed=6, n_actions=8, extra_ignitions=3), 64, 0.3, 3, True, "host"),
    (dict(width=24, height=20, seed=7, wind="random", allow_dig_toggle=True, n_actions=5, make_rivers=True), 50, 0.0, 2,
     False, "dev"),
    (dict(width=31, height=13, seed=8, fuel=40, n_actions=8, a_speed=2), 1, 0.3, 2, True, "dev"),
    (dict(width=32, height=32, seed=9, n_actions=1), 33, 0.3, 2, True, "host"),
    (dict(width=32, height=32, seed=10, wind=[0.85, (0, 1)], make_rivers=True), 16, 0.3, 2, True, "host"),
    (dict(width=24, height=20, seed=11, fuel=40, n_actions=7, extra_ignitions=2), 64, 0.3, 3, True, "host"),
]


def _wid(c):
    cfg = c[0]
    return (f"{cfg['width']}x{cfg['height']}-h{c[1]}-A{cfg.get('n_actions', 4)}-eps{c[2]}-{c[5]}"
            f"{'' if c[4] else '-frozen'}")


@pytest.mark.parametrize("case", WARP, ids=[_wid(c) for c in WARP])
def test_warp_policy_matches_float64(case):
    cfg, hid, eps, launches, auto_reset, path = case
    W, H = cfg["width"], cfg["height"]
    A = cfg.get("n_actions", 4)
    shape = _Shape(W, H, hid, A, 0)
    nets = _nets(cfg["seed"], W, H, hid, A, lanes=16 if W <= 16 else 32)
    ended = _check(_wid(case), cfg, nets, shape, [eps], 32, 96, launches, auto_reset, path)
    assert ended > 0


GROUPS = [
    (dict(width=14, height=14, seed=21, allow_dig_toggle=True, n_actions=5), 50, 1, [0.0, 0.3, 1.0, 0.3]),
    (dict(width=24, height=20, seed=22, wind="random", n_actions=8), 64, 0, [0.3, 0.0, 0.3, 0.3]),
    (dict(width=32, height=32, seed=23, fuel=40), 17, 1, [0.3, 0.3, 0.0, 0.3]),
]


@pytest.mark.parametrize("case", GROUPS, ids=[f"{c[0]['width']}x{c[0]['height']}-h{c[1]}-duel{c[2]}" for c in GROUPS])
def test_group_networks_match_float64(case):
    """set_policy_mlp_flat_dev with four networks of the flat layout: every group against its own network (a dueling
    network against its full Q), with auto-resets over two launches."""
    cfg, hid, duel, eps = case
    W, H = cfg["width"], cfg["height"]
    A = cfg.get("n_actions", 4)
    shape = _Shape(W, H, hid, A, duel)
    nets = _nets(cfg["seed"], W, H, hid, A, duel, M=4, lanes=16 if W <= 16 else 32)
    assert _check(f"groups-{W}x{H}", cfg, nets, shape, eps, 64, 64, 2, True, "flat") > 0


def _near_bound(net, shape, seed):
    """Units 3 and 40 with first-layer entries at 0.999 * 2^31 / (2 W H + 1), random signs: the largest magnitudes the
    tile kernel's exact int64 sums accept."""
    p = {k: v.copy() for k, v in R.split(net, shape).items()}
    bound = np.float32(0.999 * 2.0 ** 31 / (2 * shape.width * shape.height + 1))
    rng = np.random.default_rng(seed)
    for j in (3, 40):
        p["w1"][j] = rng.choice([-bound, bound], p["w1"].shape[1])
    return R.join(p, False).astype(np.float32)


TILE = [
    (dict(width=40, height=40, seed=31, n_actions=8, extra_ignitions=4), 1, 0.3, "host", False),
    (dict(width=48, height=40, seed=32, n_actions=1, wind=[0.85, (1, 0)], extra_ignitions=4), 64, 0.3, "dev", False),
    (dict(width=40, height=40, seed=33, n_actions=8, extra_ignitions=4), 64, 0.3, "host", True),
    (dict(width=36, height=33, seed=34, fuel=40, allow_dig_toggle=True, n_actions=5, extra_ignitions=4), 64, 0.0, "dev",
     False),
]


@pytest.mark.parametrize("case", TILE, ids=[f"{c[0]['width']}x{c[0]['height']}-h{c[1]}-A{c[0]['n_actions']}"
                                            f"{'-bound' if c[4] else ''}" for c in TILE])
def test_tile_policy_matches_float64(case):
    cfg, hid, eps, path, near_bound = case
    W, H = cfg["width"], cfg["height"]
    A = cfg["n_actions"]
    shape = _Shape(W, H, hid, A, 0)
    nets = _nets(cfg["seed"], W, H, hid, A, lanes=32)
    if near_bound:
        nets = [_near_bound(nets[0], shape, cfg["seed"])]
    assert _check(f"tile-{W}x{H}-h{hid}", cfg, nets, shape, [eps], 4, 160, 2, True, path) > 0
