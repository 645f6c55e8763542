"""wf_replay_fit, wf_replay_fit_large and wf_replay_fit_many against the float64 reference (tests/f64_ref.py), through
the C ABI so that hidden, n_actions, batch, grid and every hyper-parameter are free.

Gradient read-out: one replay from zero moments with adam_t = 0, beta_1 = beta_2 = 0 and clipvalue = inf leaves the
kernel's gradient in m (and its square in v); with epsilon = 1 the weight step lr * g / (|g| + 1) follows the gradient's
scale, so a wrong 1 / (B * A) or a dropped sample shows in m, v, params and the loss.  Schedule: 5 replays with a target
refresh inside, under one of eight hyper-parameter sets.

Bounds: a kernel's largest deviation from float64 is compared with the largest deviation of the reference run in float32
(the "twin": the same update, honestly rounded) on the same inputs: kernel <= C_TWIN * twin + a floor of FLOOR_ULPS
float32 ulps of the largest reference element.  Measured on a B200 (1000 W power limit), the largest kernel / twin ratio
over the cases of each mode:

    mode       params  target  m     v     loss
    read-out   1.0     -       4.7   6.3   31 (7.4e-7 against 2.4e-8: inside the floor; the kernel sums the loss in order)
    schedule   1.03    1.0     1.9   2.0   4.3
    many       1.06    1.0     2.8   2.3   7.8

and the largest kernel deviations 4.6e-7 (read-out m), 2.5e-7 (schedule params), 1.1e-7 (many params).  C_TWIN = 10.
MEASURED collects (mode, case, quantity, kernel deviation, twin deviation) as the tests run, for recalibrating."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests import f64_ref as R
from wildfire_control_python_b200 import _lib

pytestmark = pytest.mark.gpu

C_TWIN = 10.0
FLOOR_ULPS = 4.0
MEASURED = []


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else t.data_ptr()


def _dev(x, dt):
    return torch.as_tensor(np.ascontiguousarray(x)).to(dt).cuda()


def _check(mode, case, what, kernel, ref64, twin):
    kernel, ref64, twin = (np.asarray(x, np.float64) for x in (kernel, ref64, twin))
    dk, dt = float(np.abs(kernel - ref64).max()), float(np.abs(twin - ref64).max())
    floor = FLOOR_ULPS * 2.0 ** -24 * float(np.abs(ref64).max())
    MEASURED.append((mode, case, what, dk, dt))
    assert np.isfinite(kernel).all(), (mode, case, what)
    assert dk <= C_TWIN * dt + floor, (mode, case, what, dk, dt, floor, int(np.abs(kernel - ref64).argmax()))


def _inputs(seed, sh, sarsa, n_rep):
    rng = np.random.default_rng(seed)
    B = sh.batch
    data = R.random_replays(rng, sh, max(16, 2 * B), n_rep * B)
    state = R.random_state(rng, sh)
    frames, s, sp, a, ap, r, d = data
    return rng, state, (frames, s, sp, a, ap if sarsa else None, r, d)


def _fit(fn, sh, hp, n_rep, state, data):
    """One call of wf_replay_fit / wf_replay_fit_large; (params, target, m, v, loss) on the host."""
    frames, s, sp, a, ap, r, d = data
    st = [_dev(x, torch.float32) for x in state]
    cols = [_dev(frames, torch.int32), _dev(s, torch.int64), _dev(sp, torch.int64), _dev(a, torch.int32),
            None if ap is None else _dev(ap, torch.int32), _dev(r, torch.float32), _dev(d, torch.uint8)]
    loss = torch.full((n_rep,), -1.0, device="cuda")
    f = getattr(_lib.lib(), fn)
    _lib.check(f(C.byref(sh), C.byref(hp), n_rep, *[_p(t) for t in st], _p(cols[0]), len(frames), *[_p(t) for t in cols[1:]],
                 _p(loss), _stream()))
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in st] + [loss.cpu().numpy()]


# ---------------------------------------------------------------------------------------------------------------------
# (entry point, W, H, hidden, dueling, A, B, sarsa): a pairwise cover of hidden x dueling x A x B x SARSA x grid
READOUT = [
    ("wf_replay_fit", 10, 10, 1, 0, 1, 1, 0), ("wf_replay_fit", 10, 10, 17, 1, 4, 31, 1),
    ("wf_replay_fit", 16, 10, 50, 0, 5, 33, 0), ("wf_replay_fit", 16, 10, 64, 1, 8, 256, 1),
    ("wf_replay_fit", 17, 10, 1, 1, 5, 256, 0), ("wf_replay_fit", 17, 10, 17, 0, 8, 1, 1),
    ("wf_replay_fit", 31, 13, 50, 1, 1, 31, 0), ("wf_replay_fit", 31, 13, 64, 0, 4, 33, 1),
    ("wf_replay_fit", 32, 32, 1, 0, 8, 33, 1), ("wf_replay_fit", 32, 32, 17, 1, 5, 1, 0),
    ("wf_replay_fit", 32, 32, 50, 0, 4, 256, 1), ("wf_replay_fit", 32, 32, 64, 1, 8, 256, 0),
    ("wf_replay_fit", 10, 10, 64, 0, 1, 256, 1), ("wf_replay_fit", 16, 10, 50, 1, 8, 31, 0),
    ("wf_replay_fit", 17, 10, 64, 1, 4, 33, 1), ("wf_replay_fit", 31, 13, 17, 0, 5, 256, 0),
    ("wf_replay_fit_large", 33, 33, 1, 1, 8, 31, 1), ("wf_replay_fit_large", 33, 33, 64, 1, 8, 256, 0),
    ("wf_replay_fit_large", 33, 33, 17, 0, 4, 1, 0), ("wf_replay_fit_large", 48, 40, 50, 0, 5, 33, 1),
    ("wf_replay_fit_large", 48, 40, 64, 1, 1, 31, 0), ("wf_replay_fit_large", 48, 40, 1, 0, 4, 256, 1),
    ("wf_replay_fit_large", 100, 70, 17, 1, 5, 256, 0), ("wf_replay_fit_large", 100, 70, 64, 0, 8, 33, 1),
    ("wf_replay_fit_large", 100, 70, 50, 1, 4, 1, 1), ("wf_replay_fit_large", 10, 10, 50, 1, 8, 33, 0),
    ("wf_replay_fit_large", 17, 10, 64, 0, 5, 31, 1), ("wf_replay_fit_large", 31, 13, 17, 1, 1, 256, 1),
    ("wf_replay_fit_large", 32, 32, 1, 0, 5, 33, 0), ("wf_replay_fit_large", 48, 40, 17, 1, 8, 256, 1),
]


def _id(c):
    return f"{c[0][14:] or 'small'}-{c[1]}x{c[2]}-h{c[3]}{'d' if c[4] else ''}-A{c[5]}-B{c[6]}{'-sarsa' if c[7] else ''}"


@pytest.mark.parametrize("case", READOUT, ids=[_id(c) for c in READOUT])
def test_gradient_readout_matches_float64(case):
    """One replay in read-out mode: m = the kernel's gradient against the float64 gradient (every element), v against
    its square, the loss against the float64 MSE, params against P0 - lr * g / (|g| + 1)."""
    fn, W, H, hid, duel, A_, B, sarsa = case
    sh = _lib.WfMlpShape(width=W, height=H, hidden=hid, n_actions=A_, dueling=duel, batch=B)
    hp = _lib.WfFitParams(gamma=0.95, lr=1e-3, beta_1=0.0, beta_2=0.0, epsilon=1.0, clipvalue=math.inf, adam_t=0,
                          target_every=7, phase=7)
    _, state, data = _inputs(READOUT.index(case), sh, sarsa, 1)
    P, T, M, V, loss = _fit(fn, sh, hp, 1, state, data)
    l64, g64 = R.gradient(state[0], state[1], sh, hp.gamma, *data)
    l32, g32 = R.gradient(state[0], state[1], sh, hp.gamma, *data, dtype=np.float32)
    tag = _id(case)
    _check("readout", tag, "m", M, g64, g32)
    _check("readout", tag, "v", V, g64 * g64, g32.astype(np.float64) ** 2)
    _check("readout", tag, "loss", loss, [l64], [l32])
    step = lambda g, dt: (state[0].astype(dt) - dt(1e-3) * g / (np.abs(g) + dt(1))).astype(np.float64)  # noqa: E731
    _check("readout", tag, "params", P, step(g64, np.float64), step(g32, np.float32))
    assert np.array_equal(T, state[1])  # no refresh
    assert np.abs(g64).max() > 0


# ---------------------------------------------------------------------------------------------------------------------
HP_SETS = [
    dict(clipvalue=1e-3, target_every=3, phase=2),                    # most elements clipped
    dict(gamma=0.0, target_every=4, phase=3),
    dict(gamma=1.0, target_every=2, phase=1),
    dict(target_every=1, phase=1),                                    # refresh after every replay
    dict(target_every=3, phase=2),
    dict(adam_t=10**6, target_every=5, phase=4),
    dict(beta_1=0.5, beta_2=0.9, target_every=3, phase=3),
    dict(epsilon=1e-7, target_every=4, phase=2),                      # the production epsilon
]


def _hp(j):
    hp = dict(gamma=0.99, lr=2e-3, beta_1=0.9, beta_2=0.999, epsilon=1.0, clipvalue=1.0, adam_t=3, target_every=3, phase=2)
    hp.update(HP_SETS[j])
    return _lib.WfFitParams(**hp)


def _warm(rng, state):
    """Adam moments of an earlier run (so adam_t > 0 is consistent with them)."""
    P, T, _, _ = state
    return P, T, (rng.standard_normal(P.shape) * 1e-3).astype(np.float32), (rng.random(P.shape) * 1e-5).astype(np.float32)


# (entry point, W, H, hidden, dueling, A, B, sarsa, hyper-parameter set)
SCHEDULE = [
    ("wf_replay_fit", 14, 14, 50, 0, 4, 32, 0, 0), ("wf_replay_fit", 17, 10, 64, 1, 8, 33, 1, 1),
    ("wf_replay_fit", 32, 32, 17, 0, 5, 256, 1, 2), ("wf_replay_fit", 10, 10, 1, 1, 1, 31, 0, 3),
    ("wf_replay_fit", 31, 13, 64, 0, 7, 64, 1, 4), ("wf_replay_fit", 24, 20, 33, 1, 4, 1, 0, 5),
    ("wf_replay_fit", 16, 16, 50, 1, 5, 100, 1, 6), ("wf_replay_fit", 20, 12, 64, 1, 8, 256, 0, 7),
    ("wf_replay_fit_large", 33, 33, 64, 1, 8, 33, 1, 0), ("wf_replay_fit_large", 48, 40, 50, 0, 4, 32, 0, 3),
    ("wf_replay_fit_large", 100, 70, 17, 1, 5, 31, 1, 5), ("wf_replay_fit_large", 40, 40, 64, 0, 7, 256, 0, 7),
]


@pytest.mark.parametrize("case", SCHEDULE, ids=[_id(c[:8]) + f"-hp{c[8]}" for c in SCHEDULE])
def test_replay_schedule_matches_float64(case):
    """5 replays with the target refreshed inside the run: params, target, m, v and every loss against float64."""
    fn, W, H, hid, duel, A_, B, sarsa, j = case
    n_rep = 5
    sh = _lib.WfMlpShape(width=W, height=H, hidden=hid, n_actions=A_, dueling=duel, batch=B)
    hp = _hp(j)
    rng, state, data = _inputs(100 + SCHEDULE.index(case), sh, sarsa, n_rep)
    state = _warm(rng, state)
    got = _fit(fn, sh, hp, n_rep, state, data)
    ref = R.replay_fit(state, sh, hp, *data, n_rep)
    twin = R.replay_fit(state, sh, hp, *data, n_rep, dtype=np.float32)
    tag = _id(case[:8]) + f"-hp{j}"
    for what, x, y, z in zip(("params", "target", "m", "v", "loss"), got, ref, twin):
        _check("schedule", tag, what, x, y, z)
    assert not np.array_equal(got[1], state[1])  # the target was refreshed


def test_replay_fit_many_matches_float64_per_learner():
    """64 learners (kMaxLearners) in one wf_replay_fit_many launch, each with its own state, transitions and hyper-
    parameter set (the eight above in turn), half of them SARSA: every learner against its float64 reference."""
    L = _lib.lib()
    n, n_rep = _lib.MAX_LEARNERS, 4
    sh = _lib.WfMlpShape(width=16, height=10, hidden=33, n_actions=5, dueling=1, batch=33)
    rng = np.random.default_rng(7)
    frames = R.random_replays(rng, sh, 80, 1)[0]
    fr = _dev(frames, torch.int32)
    learners, refs, keep = [], [], []
    for k in range(n):
        _, s, sp, a, ap, r, d = R.random_replays(rng, sh, 80, n_rep * sh.batch)
        if k % 2:
            ap = None
        state = _warm(rng, R.random_state(rng, sh))
        hp = _hp(k % len(HP_SETS))
        st = [_dev(x, torch.float32) for x in state]
        cols = [_dev(s, torch.int64), _dev(sp, torch.int64), _dev(a, torch.int32), None if ap is None else _dev(ap, torch.int32),
                _dev(r, torch.float32), _dev(d, torch.uint8)]
        loss = torch.full((n_rep,), -1.0, device="cuda")
        keep.append((st, cols, loss))
        learners.append(_lib.WfFitLearner(*[_p(t) for t in st], *[_p(t) for t in cols], _p(loss), hp))
        data = (frames, s, sp, a, ap, r, d)
        refs.append((hp, state, data))
    desc = (_lib.WfFitLearner * n)(*learners)
    _lib.check(L.wf_replay_fit_many(C.byref(sh), n, desc, n_rep, _p(fr), len(frames), _stream()))
    torch.cuda.synchronize()
    for k, ((st, _, loss), (hp, state, data)) in enumerate(zip(keep, refs)):
        got = [t.cpu().numpy() for t in st] + [loss.cpu().numpy()]
        ref = R.replay_fit(state, sh, hp, *data, n_rep)
        twin = R.replay_fit(state, sh, hp, *data, n_rep, dtype=np.float32)
        for what, x, y, z in zip(("params", "target", "m", "v", "loss"), got, ref, twin):
            _check("many", f"learner{k}-hp{k % len(HP_SETS)}", what, x, y, z)
