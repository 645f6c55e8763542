"""Plain float64 statements of what the device Q-network kernels compute, for the tests that pin those kernels.

Nothing here calls the package's learners or kernels: the math is restated from the reference's rule (DQN.py:156-185,
DQN_SARSA.py:103-132, Keras 2's clipped Adam) on the flat parameter layout of include/wildfire.h,

    dense_1.weight [hidden][n_in] | dense_1.bias | dense_2.weight [A][hidden] | dense_2.bias
    | (dueling) dense_3.weight [hidden][n_in] | dense_3.bias | dense_4.weight [1][hidden] | dense_4.bias

(``parameters_to_vector(model.parameters())``, n_in = W * H * 3), with gradients written out by hand.  ``dtype`` lets the
same code run in float32: that twin measures how far an honest float32 evaluation of the same update lands from float64,
which is what the kernels' deviations are bounded against.

Also: generators of replay inputs (bit frames, rows, actions, rewards, with out-of-range rows and actions) and of
discriminating policy weights, whose greedy action varies with the observation and depends on every lane and register
slot of hidden units the in-kernel policy deals them out to.
"""
from __future__ import annotations

import numpy as np


def n_in(shape) -> int:
    return int(shape.width) * int(shape.height) * 3


def param_count(shape) -> int:
    n, hid, A = n_in(shape), int(shape.hidden), int(shape.n_actions)
    return hid * (n + 1 + A) + A + (hid * (n + 2) + 1 if shape.dueling else 0)


def split(flat, shape) -> dict:
    """Views of the flat layout: w1 [hid, n_in], b1, w2 [A, hid], b2 and, dueling, w3, b3, w4 [1, hid], b4."""
    n, hid, A = n_in(shape), int(shape.hidden), int(shape.n_actions)
    flat = np.asarray(flat)
    assert flat.shape == (param_count(shape),), (flat.shape, param_count(shape))
    out, o = {}, 0
    parts = [("w1", (hid, n)), ("b1", (hid,)), ("w2", (A, hid)), ("b2", (A,))]
    if shape.dueling:
        parts += [("w3", (hid, n)), ("b3", (hid,)), ("w4", (1, hid)), ("b4", (1,))]
    for name, shp in parts:
        size = int(np.prod(shp))
        out[name] = flat[o:o + size].reshape(shp)
        o += size
    return out


def join(parts: dict, dueling: bool) -> np.ndarray:
    names = ["w1", "b1", "w2", "b2"] + (["w3", "b3", "w4", "b4"] if dueling else [])
    return np.concatenate([np.asarray(parts[k]).reshape(-1) for k in names])


def from_keras(k1, b1, k2, b2):
    """The Keras orientation of ``set_policy_mlp`` (kernel1 [n_in, hid], kernel2 [hid, A]) as w1, b1, w2, b2."""
    return {"w1": np.asarray(k1).T, "b1": np.asarray(b1), "w2": np.asarray(k2).T, "b2": np.asarray(b2)}


def sigmoid(z):
    return 1.0 / (1.0 + np.exp(-np.clip(z, -500, 500)))


def _parts(params, shape):
    if isinstance(params, (tuple, list)):
        return from_keras(*params)
    return split(params, shape)


def hidden(params, shape, x, dtype=np.float64):
    """Hidden activations of the advantage (plain) stream, [n, hidden]."""
    p = _parts(params, shape)
    x = np.asarray(x, dtype).reshape(len(x), -1)
    return sigmoid(x @ p["w1"].astype(dtype).T + p["b1"].astype(dtype))


def q_values(params, shape, x, dtype=np.float64):
    """Q [n, A] of observations ``x`` ([n, n_in] or [n, W, H, 3], 0/1) under flat ``params`` (or a Keras-oriented
    (kernel1, bias1, kernel2, bias2) tuple: a plain head); a dueling head gives V + A - mean(A)."""
    return _forward({k: v.astype(dtype) for k, v in _parts(params, shape).items()}, np.asarray(x, dtype).reshape(len(x), -1),
                    bool(shape.dueling) and not isinstance(params, (tuple, list)))[0]


def _forward(p, x, duel):
    h = sigmoid(x @ p["w1"].T + p["b1"])
    adv = h @ p["w2"].T + p["b2"]
    if not duel:
        return adv, h, None
    hv = sigmoid(x @ p["w3"].T + p["b3"])
    val = hv @ p["w4"].T + p["b4"]
    return val + (adv - adv.mean(axis=1, keepdims=True)), h, hv


def _gradients(p, x, y, duel):
    """MSE over all B * A elements and its gradient with respect to every part, by the chain rule."""
    q, h, hv = _forward(p, x, duel)
    e = q - y
    loss = (e * e).sum() / e.size
    dq = 2.0 * e / e.size
    g = {}
    dadv = dq - dq.mean(axis=1, keepdims=True) if duel else dq
    g["w2"] = dadv.T @ h
    g["b2"] = dadv.sum(axis=0)
    dz = (dadv @ p["w2"]) * h * (1.0 - h)
    g["w1"] = dz.T @ x
    g["b1"] = dz.sum(axis=0)
    if duel:
        dval = dq.sum(axis=1, keepdims=True)
        g["w4"] = dval.T @ hv
        g["b4"] = dval.sum(axis=0)
        dzv = (dval @ p["w4"]) * hv * (1.0 - hv)
        g["w3"] = dzv.T @ x
        g["b3"] = dzv.sum(axis=0)
    return loss, g


def unpack_bits(frames, width, height) -> np.ndarray:
    """[n_frames, words] int32 WF_OBS_BITS rows -> [n_frames, n_in] uint8 (element k = bit k % 32 of word k // 32)."""
    f = np.ascontiguousarray(np.asarray(frames, np.int32)).view(np.uint32).astype("<u4")
    bits = np.unpackbits(f.view(np.uint8), axis=1, bitorder="little")
    return bits[:, :int(width) * int(height) * 3]


def pack_bits(x) -> np.ndarray:
    """[n, n_in] 0/1 -> [n, ceil(n_in / 32)] int32 in the WF_OBS_BITS layout (zero padding)."""
    x = (np.asarray(x).reshape(len(x), -1) != 0).astype(np.uint8)
    words = (x.shape[1] + 31) // 32
    x = np.pad(x, ((0, 0), (0, words * 32 - x.shape[1])))
    return np.packbits(x, axis=1, bitorder="little").view("<u4").astype(np.uint32).view(np.int32).reshape(len(x), words)


def _obs(X, rows, dtype):
    rows = np.asarray(rows, np.int64)
    ok = (rows >= 0) & (rows < len(X))
    out = np.zeros((len(rows), X.shape[1]), dtype)
    out[ok] = X[rows[ok]]
    return out


def _loss_and_gradient(P, T, shape, gamma, X, s_row, sp_row, a, ap, r, d, dtype):
    """One replay's targets (from the target network T), its MSE and the flat gradient at P."""
    B, A, duel = len(s_row), int(shape.n_actions), bool(shape.dueling)
    xs, xsp = _obs(X, s_row, dtype), _obs(X, sp_row, dtype)
    tp = split(T, shape)
    y, _, _ = _forward(tp, xs, duel)
    qn, _, _ = _forward(tp, xsp, duel)
    rew, act = np.asarray(r).astype(dtype), np.asarray(a, np.int64)
    if ap is None:
        upd = rew + gamma * qn.max(axis=1)
    else:
        nact = np.asarray(ap, np.int64)
        upd = np.where((nact >= 0) & (nact < A), rew + gamma * qn[np.arange(B), np.clip(nact, 0, A - 1)], rew)
    upd = np.where(np.asarray(d).astype(bool), rew, upd)
    ok = (act >= 0) & (act < A)
    y = y.copy()
    y[np.nonzero(ok)[0], act[ok]] = upd[ok]
    loss, g = _gradients(split(P, shape), xs, y, duel)
    return loss, join(g, duel).astype(dtype)


def replay_fit(state, shape, hp, frames_bits, s_row, sp_row, a, ap, r, d, n_replays, dtype=np.float64):
    """``n_replays`` consecutive DQN replays (what wf_replay_fit promises), replay i on transitions i * B ... i * B + B - 1.

    ``state``: (params, target, m, v) flat arrays; ``hp``: anything with the fields of ``wf_fit_params`` (gamma, lr, beta_1,
    beta_2, epsilon, clipvalue, adam_t, target_every, phase); ``ap`` None = max bootstrap, else SARSA.  Per replay:
      targets  Q_target(s) with the taken action's entry replaced by r (done) or r + gamma * bootstrap(s'), bootstrap =
               max_a Q_target(s', a) or Q_target(s', a'); a row outside the frames is an all-zero observation, an action
               outside [0, A) replaces no entry, a next action outside [0, A) bootstraps nothing (the target is r);
      fit      the MSE over B * A and its gradient; Keras 2 Adam: g clipped to [-clipvalue, clipvalue], t = adam_t + i + 1,
               m = b1 m + (1 - b1) g, v = b2 v + (1 - b2) g^2, lr_t = lr sqrt(1 - b2^t) / (1 - b1^t) in double,
               p -= lr_t m / (sqrt(v) + epsilon);
      sync     ``phase`` replays until the first target refresh (target = model after that replay's update), then every
               ``target_every``.
    Returns (params, target, m, v, losses) in ``dtype``."""
    B = len(s_row) // n_replays
    X = unpack_bits(frames_bits, shape.width, shape.height).astype(dtype)
    P, T, M, V = (np.array(s, dtype) for s in state)
    gamma = dtype(hp.gamma)
    b1, b2, eps, clip = dtype(hp.beta_1), dtype(hp.beta_2), dtype(hp.epsilon), dtype(hp.clipvalue)
    until, losses = int(hp.phase), []
    for i in range(n_replays):
        sl = slice(i * B, i * B + B)
        loss, grad = _loss_and_gradient(P, T, shape, gamma, X, s_row[sl], sp_row[sl], a[sl], None if ap is None else ap[sl],
                                        r[sl], d[sl], dtype)
        losses.append(loss)
        t = int(hp.adam_t) + i + 1
        lr_t = hp.lr * np.sqrt(1.0 - hp.beta_2 ** t) / (1.0 - hp.beta_1 ** t)
        grad = np.clip(grad, -clip, clip)
        M = b1 * M + (dtype(1) - b1) * grad
        V = b2 * V + (dtype(1) - b2) * grad * grad
        P = P - dtype(lr_t) * (M / (np.sqrt(V) + eps))
        until -= 1
        if until == 0:
            until = int(hp.target_every)
            T = P.copy()
    return P, T, M, V, np.array(losses, dtype)


def gradient(params, target, shape, gamma, frames_bits, s_row, sp_row, a, ap, r, d, dtype=np.float64):
    """(loss, unclipped flat gradient) of one replay at ``params``: what a kernel's m holds after one replay with
    beta_1 = 0 and no clipping."""
    X = unpack_bits(frames_bits, shape.width, shape.height).astype(dtype)
    return _loss_and_gradient(np.asarray(params, dtype), np.asarray(target, dtype), shape, dtype(gamma), X, s_row, sp_row, a,
                              ap, r, d, dtype)


# ---------------------------------------------------------------------------------------------------------------------
# generators
def random_replays(rng, shape, n_frames, n, p_bit=0.35, out_of_range=True):
    """Bit frames and ``n`` transitions: rows (with ``out_of_range``, some below 0 or past the last frame), actions and next
    actions in [-1, A] (so both edges are out of range), rewards of scale 3 and about 10 % done flags."""
    A = int(shape.n_actions)
    x = rng.random((n_frames, n_in(shape))) < p_bit
    frames = pack_bits(x)
    lo, hi = (-3, n_frames + 3) if out_of_range else (0, n_frames)
    s_row = rng.integers(lo, hi, n).astype(np.int64)
    sp_row = rng.integers(lo, hi, n).astype(np.int64)
    alo, ahi = (-1, A + 1) if out_of_range else (0, A)
    act = rng.integers(alo, ahi, n).astype(np.int32)
    nact = rng.integers(alo, ahi, n).astype(np.int32)
    rew = (rng.standard_normal(n) * 3).astype(np.float32)
    done = (rng.random(n) < 0.1).astype(np.uint8)
    return frames, s_row, sp_row, act, nact, rew, done


def random_state(rng, shape, scale=1.0):
    """(params, target, m, v) float32: Glorot-sized first layers, unit-sized second layers, a target near the model and
    zero Adam moments."""
    n, hid = n_in(shape), int(shape.hidden)
    g = np.sqrt(6.0 / (n + hid))
    parts = {"w1": rng.uniform(-g, g, (hid, n)), "b1": rng.uniform(-0.5, 0.5, hid),
             "w2": rng.uniform(-1, 1, (int(shape.n_actions), hid)) * scale, "b2": rng.uniform(-0.5, 0.5, int(shape.n_actions))}
    if shape.dueling:
        parts.update({"w3": rng.uniform(-g, g, (hid, n)), "b3": rng.uniform(-0.5, 0.5, hid),
                      "w4": rng.uniform(-1, 1, (1, hid)) * scale, "b4": rng.uniform(-0.5, 0.5, 1)})
    P = join(parts, shape.dueling).astype(np.float32)
    T = (P + rng.standard_normal(P.shape) * 0.01).astype(np.float32)
    return P, T, np.zeros_like(P), np.zeros_like(P)


def synthetic_observations(rng, width, height, n):
    """[n, W, H, 3] observations like the environment's: one agent cell, a few burning cells in clusters, the non-free
    cells (channel 2 = 0) where fire is or has been."""
    W, H = int(width), int(height)
    o = np.zeros((n, W, H, 3), np.uint8)
    o[..., 2] = 1
    for i in range(n):
        o[i, rng.integers(W), rng.integers(H), 0] = 1
        cx, cy, rad = rng.integers(W), rng.integers(H), rng.integers(0, 4)
        xs, ys = np.meshgrid(np.arange(W), np.arange(H), indexing="ij")
        dist = np.abs(xs - cx) + np.abs(ys - cy)
        o[i, ..., 1] = (dist == rad)
        o[i, ..., 2] = dist > rad
    return o


def policy_net(rng, width, height, hid, A, dueling=False):
    """One candidate network (flat layout, float32): the agent channel dominates the first layer so that the greedy action
    follows the agent's cell, the fire channel matters too, the free channel is small and the first-layer bias centres
    the empty map; the second-layer biases give every action's Q the same mean and then shift them so that every Q value
    is negative (an action the network does not have must not win as a 0)."""
    n = int(width) * int(height) * 3
    w1 = rng.standard_normal((hid, n)) * 0.05
    w1[:, 0::3] = rng.standard_normal((hid, n // 3)) * 2.0
    w1[:, 1::3] = rng.standard_normal((hid, n // 3)) * 0.5
    b1 = -w1[:, 2::3].sum(axis=1) + rng.standard_normal(hid) * 0.5
    w2 = rng.choice([-1.0, 1.0], (A, hid)) * rng.uniform(0.5, 1.0, (A, hid))  # no unit with a negligible weight
    b2 = rng.uniform(-0.1, 0.1, A) - 0.5 * w2.sum(axis=1)  # every action's Q of the same mean (s_j is about 1/2 on average)
    b2 -= np.abs(w2).sum(axis=1).max() + 0.5
    parts = {"w1": w1, "b1": b1, "w2": w2, "b2": b2}
    if dueling:
        parts.update({"w3": rng.standard_normal((hid, n)) * 0.5, "b3": rng.standard_normal(hid),
                      "w4": rng.uniform(-1, 1, (1, hid)), "b4": rng.uniform(-1, 1, 1)})
    return join(parts, dueling).astype(np.float32)


def sensitivity(params, shape, x, lanes):
    """How much every hidden unit the in-kernel policy deals out matters, in float64 on observations ``x``: the share of
    observations whose greedy action changes when the units of one lane (j % lanes == l) or of one register slot
    (j // lanes == i) are switched off (their second-layer weights zeroed), the smallest over lanes and over slots, and
    the set of greedy actions.  A dueling head's greedy action is the advantage stream's."""
    p = _parts(params, shape)
    h = hidden(params, shape, x)
    w2, b2 = p["w2"].astype(np.float64), p["b2"].astype(np.float64)
    greedy = np.argmax(h @ w2.T + b2, axis=1)
    hid = h.shape[1]

    def changed(mask):
        return float(np.mean(np.argmax(h @ (w2 * ~mask).T + b2, axis=1) != greedy))

    j = np.arange(hid)
    lane = min(changed(j % lanes == x_) for x_ in range(min(lanes, hid)))
    slot = min(changed(j // lanes == i) for i in range((hid + lanes - 1) // lanes))
    return lane, slot, set(int(g) for g in np.unique(greedy))


def discriminates(params, shape, x, lanes, min_share=0.02):
    """The checks a network must pass to make a policy test bite (see ``sensitivity``): more than one greedy action, with
    A = 8 an action >= 5 among them, and every lane and slot changing at least ``min_share`` of the greedy actions.
    A one-action network has nothing to discriminate."""
    A = int(shape.n_actions)
    if A == 1:
        return True
    lane, slot, acts = sensitivity(params, shape, x, lanes)
    return len(acts) > 1 and (A < 8 or max(acts) >= 5) and lane >= min_share and slot >= min_share


def policy_weights(seed, width, height, hid, A, dueling=False, lanes=16, tries=50):
    """Discriminating policy weights (``policy_net``): the first candidate from ``seed`` that passes ``discriminates`` with
    twice the share a test asks for on 512 synthetic observations (``synthetic_observations``), so that it still passes
    on the frames a rollout shows it.  Flat layout, float32."""
    class _S:
        pass
    shape = _S()
    shape.width, shape.height, shape.hidden, shape.n_actions, shape.dueling = width, height, hid, A, int(dueling)
    rng = np.random.default_rng(seed)
    x = synthetic_observations(np.random.default_rng(seed + 1), width, height, 512)
    for _ in range(tries):
        net = policy_net(rng, width, height, hid, A, dueling)
        if discriminates(net, shape, x, lanes, min_share=0.04):
            return net
    raise AssertionError(f"no discriminating network for {width}x{height}, hidden {hid}, A {A}")
