"""The float64 reference of the Q-network kernels (tests/f64_ref.py) against what it restates: the golden N1 fixture
(a NumPy restatement of the reference's Keras update), the torch learners of agents.py run in float64, explicit
statements of the out-of-range rules, and the sensitivity of the generated policy weights.  No GPU needed."""
import numpy as np
import pytest
import torch

from tests import f64_ref as R
from tests.test_agents import FakeSim, _load_n1
from wildfire_control_python_b200 import _lib
from wildfire_control_python_b200 import agents as A

NAMES = ["DQN", "DQN_SARSA", "DQN_DUEL", "DQN_BOTH"]
DUEL = {"DQN": 0, "DQN_SARSA": 0, "DQN_DUEL": 1, "DQN_BOTH": 1}
SARSA = {"DQN": False, "DQN_SARSA": True, "DQN_DUEL": False, "DQN_BOTH": True}


def _shape(W=10, H=10, hid=50, A_=4, duel=0, B=32):
    return _lib.WfMlpShape(width=W, height=H, hidden=hid, n_actions=A_, dueling=duel, batch=B)


def _hp(**kw):
    hp = dict(gamma=0.999, lr=0.005, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipvalue=1.0, adam_t=0, target_every=20, phase=20)
    hp.update(kw)
    return _lib.WfFitParams(**hp)


def _flat_from_keras(w, duel):
    parts = {}
    for k, (wn, bn) in {"1": ("w1", "b1"), "2": ("w2", "b2"), "3": ("w3", "b3"), "4": ("w4", "b4")}.items():
        if f"dense_{k}/kernel:0" in w:
            parts[wn] = np.asarray(w[f"dense_{k}/kernel:0"]).T
            parts[bn] = np.asarray(w[f"dense_{k}/bias:0"])
    return R.join(parts, duel)


@pytest.mark.parametrize("name", NAMES)
def test_reference_reproduces_the_n1_fixture(name):
    """Two consecutive replays from the fixture's weights and target: loss and every stored weight, with the tolerances
    test_agents._check_n1 uses."""
    fx = _load_n1(name)
    duel = DUEL[name]
    sh = _shape(duel=duel)
    P = _flat_from_keras({k[3:]: v for k, v in fx.items() if k.startswith("w0/")}, duel)
    T = _flat_from_keras({k[7:]: v for k, v in fx.items() if k.startswith("target/")}, duel)
    state = (P, T, np.zeros_like(P), np.zeros_like(P))
    for t in (1, 2):
        b = {k: fx[f"t{t}/batch_{k}"] for k in ("s", "a", "r", "sp", "ap", "d")}
        B = len(b["a"])
        frames = R.pack_bits(np.concatenate([b["s"], b["sp"]]))
        rows = np.arange(2 * B)
        out = R.replay_fit(state, sh, _hp(adam_t=t - 1), frames, rows[:B], rows[B:], b["a"], b["ap"] if SARSA[name] else None,
                           b["r"].astype(np.float32), b["d"], 1)
        assert out[4][0] == pytest.approx(float(fx[f"t{t}/loss"]), rel=1e-4)
        got = R.split(out[0], sh)
        for k in sorted(k[5:] for k in fx if k.startswith(f"t{t}/w/")):
            layer, what = k.split("/")
            n = layer[-1]
            have = got[("w" if what.startswith("kernel") else "b") + n]
            have = have.T if what.startswith("kernel") else have
            have = have[::16] if have.shape[0] == 300 else have
            want = fx[f"t{t}/w/{k}"]
            assert np.allclose(have, want, rtol=0, atol=2e-6), (name, t, k, np.abs(have - want).max())
        state = out[:4]


class _F64(torch.nn.Module):
    """A learner's network in float64 (fit_batch feeds it float32 observations)."""

    def __init__(self, net):
        super().__init__()
        self.net = net.double()

    def forward(self, x):
        return self.net(x.double())


@pytest.mark.parametrize("name", NAMES)
def test_reference_matches_the_torch_learner_in_float64(name):
    """8 replays of agents.DQN*.fit_batch with model, target and optimiser in float64, a target refresh after replay 3,
    from a target that differs from the model: params, target, Adam m and v, and every loss."""
    torch.manual_seed(3)
    ag = getattr(A, name)(FakeSim(), verbose=False, device="cpu")
    ag.model, ag.target = _F64(ag.model), _F64(ag.target)
    with torch.no_grad():
        for p in ag.target.parameters():
            p.add_(0.02 * torch.randn_like(p))
    sh = _shape(duel=DUEL[name])
    rng = np.random.default_rng(5)
    n_rep, B, phase = 8, 32, 3
    frames, s, sp, a, ap, r, d = R.random_replays(rng, sh, 64, n_rep * B, out_of_range=False)
    p2v = torch.nn.utils.parameters_to_vector
    state = tuple(p2v(m.parameters()).detach().numpy() for m in (ag.model, ag.target)) + (np.zeros(R.param_count(sh)),) * 2
    X = torch.as_tensor(R.unpack_bits(frames, 10, 10)).view(-1, 10, 10, 3)
    losses, until = [], phase
    for i in range(n_rep):
        sl = slice(i * B, i * B + B)
        batch = (X[s[sl]], torch.as_tensor(a[sl]).long(), torch.as_tensor(r[sl]), X[sp[sl]], torch.as_tensor(ap[sl]).long(),
                 torch.as_tensor(d[sl]).bool())
        losses.append(ag.fit_batch(batch))
        until -= 1
        if until == 0:
            until = 20
            ag.target.load_state_dict(ag.model.state_dict())
    want = R.replay_fit(state, sh, _hp(phase=phase), frames, s, sp, a, ap if SARSA[name] else None, r, d, n_rep)
    st = [ag.optimizer.state[p] for p in ag.model.parameters()]
    have = [p2v(x).detach().numpy() for x in (list(ag.model.parameters()), list(ag.target.parameters()), [q["m"] for q in st],
                                              [q["v"] for q in st])] + [np.array(losses)]
    for what, x, y in zip(("params", "target", "m", "v", "loss"), have, want):
        assert np.allclose(x, y, rtol=1e-9, atol=1e-12), (what, np.abs(x - y).max())
    assert not np.array_equal(want[0], state[0]) and not np.array_equal(want[1], want[0])


def _one(state, sh, frames, s, sp, a, ap, r, d):
    return R.replay_fit(state, sh, _hp(adam_t=4), frames, s, sp, a, ap, r, d, 1)


@pytest.mark.parametrize("duel", [0, 1])
def test_out_of_range_rules(duel):
    """Each rule of fit_batches_fused against an explicit statement: a row outside the frames is the all-zero row, an
    out-of-range next action is a done flag, and an out-of-range action leaves Q_target(s) as the whole target row (the
    loss of a per-sample loop in the reference's style)."""
    sh = _shape(W=12, H=10, hid=9, A_=5, duel=duel)
    rng = np.random.default_rng(11 + duel)
    B = 40
    frames, s, sp, a, ap, r, d = R.random_replays(rng, sh, 30, B, out_of_range=False)
    state = R.random_state(rng, sh)
    bad = np.arange(B) % 4 == 0
    zero = np.concatenate([frames, np.zeros_like(frames[:1])])
    x = _one(state, sh, frames, np.where(bad, -5, s), np.where(bad, 10**9, sp), a, ap, r, d)
    y = _one(state, sh, zero, np.where(bad, 30, s), np.where(bad, 30, sp), a, ap, r, d)
    for p, q in zip(x, y):
        assert np.array_equal(p, q)
    x = _one(state, sh, frames, s, sp, a, np.where(bad, 5, ap), r, d)
    y = _one(state, sh, frames, s, sp, a, ap, r, d | bad)
    for p, q in zip(x, y):
        assert np.array_equal(p, q)
    a_bad = np.where(bad, -1, np.where(np.arange(B) % 4 == 1, 5, a))
    for ap_ in (None, ap):
        loss = _one(state, sh, frames, s, sp, a_bad, ap_, r, d)[4][0]
        X = R.unpack_bits(frames, 12, 10).astype(np.float64)
        q = R.q_values(state[0], sh, X[s])
        qt, qn = R.q_values(state[1], sh, X[s]), R.q_values(state[1], sh, X[sp])
        se = 0.0
        for i in range(B):
            pred = qt[i].copy()
            if 0 <= a_bad[i] < 5:
                if d[i]:
                    pred[a_bad[i]] = r[i]
                elif ap_ is None:
                    pred[a_bad[i]] = r[i] + 0.999 * qn[i].max()
                else:
                    pred[a_bad[i]] = r[i] + 0.999 * qn[i][ap_[i]] if 0 <= ap_[i] < 5 else r[i]
            se += ((q[i] - pred) ** 2).sum()
        assert loss == pytest.approx(se / (B * 5), rel=1e-12)


@pytest.mark.parametrize("W,H,hid,A_,lanes,duel", [(10, 10, 1, 4, 16, 0), (16, 10, 16, 8, 16, 0), (24, 20, 33, 5, 32, 1),
                                                 (32, 32, 64, 8, 32, 0), (14, 14, 64, 7, 16, 1), (40, 40, 64, 8, 32, 0)])
def test_generated_policy_weights_discriminate(W, H, hid, A_, lanes, duel):
    """The generated policy weights pass the sensitivity check on observations they were not drawn against: more than
    one greedy action (at A = 8 one >= 5), and switching off any lane's or any register slot's units changes at least 2 %
    of the greedy actions."""
    sh = _shape(W, H, hid, A_, duel)
    net = R.policy_weights(W * 100 + hid, W, H, hid, A_, duel, lanes=lanes)
    x = R.synthetic_observations(np.random.default_rng(99), W, H, 1024)
    lane, slot, acts = R.sensitivity(net, sh, x, lanes)
    assert R.discriminates(net, sh, x, lanes), (lane, slot, acts)
    p = R.split(net, sh)
    assert (R.hidden(net, sh, x) @ p["w2"].T + p["b2"] < 0).all()  # the acting stream: a missing action read as 0 would win
