"""CPU: the offline-scorer oracle (tests/offline_metrics_oracle.py) against hand-worked values, the sums -> metrics
step (``engine.offline_scores``) and the argument checks of ``CQL.offline_metrics``.

The hand-worked networks are exact piecewise-linear MLPs: critic i computes Q_i(x, a) = k_i a + u_i x0 + c_i and the
actor mu(x) = m0 + m1 x1 (one ReLU unit each, biased to stay active), so every scorer has a closed form that numpy
evaluates in float64 without the oracle's code: the windowed advantage sums as explicit power sums, not recursions.
"""
from types import SimpleNamespace

import numpy as np
import pandas as pd
import pytest
import torch

from replay_cql_b200.engine import OFFLINE_SUM_KEYS, offline_scores
from replay_cql_b200.models import CQL
from tests import offline_metrics_oracle as OM

GAMMA = 0.99
CRITICS = [(1.5, 0.25, 0.5), (0.5, -0.5, -1.25), (2.0, 0.75, 0.0), (1.0, 0.0, 2.5)]   # (k, u, c)
ACTOR = (0.3, -0.2)                                                                     # (m0, m1)
LENGTHS = [1, 2, 5, 1023, 1024, 1025, 2049]
PREP = {"scaler": {"type": "standard", "mean": [2.0, 1.0], "std": [1.5, 0.75]},
        "action_scaler": {"type": "min_max", "minimum": [1.0], "maximum": [5.0]},
        "reward_scaler": {"type": "standard", "mean": [0.5], "std": [0.5]}}


def _net(in_f, out_f):
    z = lambda *s: torch.zeros(*s, dtype=torch.float32)
    return {"W1": z(256, in_f), "b1": z(256), "W2": z(256, 256), "b2": z(256), "W3": z(out_f, 256), "b3": z(out_f)}


def _state(n_critics):
    critics = []
    for k, u, c in CRITICS[:n_critics]:
        net = _net(3, 1)
        net["W1"][0, 2], net["b1"][0] = 1.0, 10.0       # h0 = a + 10
        net["W1"][1, 0], net["b1"][1] = 1.0, 100.0      # h1 = x0 + 100
        net["W2"][0, 0] = net["W2"][1, 1] = 1.0
        net["W3"][0, 0], net["W3"][0, 1] = k, u
        net["b3"][0] = c - 10.0 * k - 100.0 * u
        critics.append(net)
    actor = _net(2, 2)
    m0, m1 = ACTOR
    actor["W1"][0, 1], actor["b1"][0] = 1.0, 100.0
    actor["W2"][0, 0] = 1.0
    actor["W3"][0, 0], actor["b3"][0] = m1, m0 - 100.0 * m1
    return {"actor": actor, "critics": critics}


def _rows(lengths, last_terminal=True, seed=0):
    """Episode-ordered one-step rows; s' = the next row's s, a terminal row's s' = (0, 0) (the MDP builder's rows)."""
    rng = np.random.default_rng(seed)
    n = sum(lengths)
    obs = np.stack([rng.integers(0, 5, n), rng.integers(0, 3, n)], 1).astype(np.float32)
    obs += rng.choice([0.0, 0.25, 0.5], size=(n, 2)).astype(np.float32)
    rows = np.zeros((n, 8), np.float32)
    rows[:, 0:2] = obs
    rows[:, 2] = rng.integers(1, 6, n).astype(np.float32)
    rows[:, 3] = (rng.random(n) < 0.3).astype(np.float32)
    ends = np.cumsum(lengths) - 1
    rows[ends, 6] = 1.0
    if not last_terminal:
        rows[-1, 6] = 0.0
    nxt = np.concatenate([obs[1:], np.zeros((1, 2), np.float32)])
    rows[:, 4:6] = np.where(rows[:, 6:7] != 0, 0.0, nxt)
    return rows


def _reference(rows, n_critics, thr=None, prep=None):
    """Closed-form float64 sums of the hand-worked networks."""
    prep = prep or {}
    r = rows.astype(np.float64)
    obs, nobs, a, rew, term = r[:, 0:2].copy(), r[:, 4:6].copy(), r[:, 2], r[:, 3], r[:, 6]
    if prep.get("scaler"):
        mu, sd = np.array(prep["scaler"]["mean"]), np.array(prep["scaler"]["std"]) + 1e-3
        obs, nobs = (obs - mu) / sd, (nobs - mu) / sd
    a_in = a
    lo = hi = None
    if prep.get("action_scaler"):
        lo, hi = prep["action_scaler"]["minimum"][0], prep["action_scaler"]["maximum"][0]
        a_in = (a - lo) / (hi - lo) * 2 - 1
    rew_in = rew
    if prep.get("reward_scaler"):
        rew_in = (rew - prep["reward_scaler"]["mean"][0]) / (prep["reward_scaler"]["std"][0] + 1e-3)
    K, U, Cc = (np.array([x[j] for x in CRITICS[:n_critics]])[:, None] for j in range(3))
    qi = lambda x0, act: K * act + U * x0 + Cc
    m0, m1 = ACTOR
    pi, npi = np.tanh(m0 + m1 * obs[:, 1]), np.tanh(m0 + m1 * nobs[:, 1])
    q = qi(obs[:, 0], a_in).mean(0)
    qv = qi(obs[:, 0], pi)
    v, sig = qv.mean(0), qv.std(0)
    y = rew_in + GAMMA * qi(nobs[:, 0], npi).mean(0) * (1 - term)
    pi_rev = pi if lo is None else (pi + 1) / 2 * (hi - lo) + lo
    adv = q - v
    g = float(np.float32(GAMMA))
    ends = list(np.flatnonzero(term != 0))
    if not ends or ends[-1] != len(r) - 1:
        ends.append(len(r) - 1)
    A, init, succ_q, succ_n, first = 0.0, 0.0, 0.0, 0, 0
    for e in ends:
        for w0 in range(first, e + 1, OM.WINDOW):
            w1 = min(e + 1, w0 + OM.WINDOW)
            for t in range(w0, w1):
                A += float(np.sum(g ** np.arange(w1 - t) * adv[t:w1]))
        init += v[first]
        if thr is not None and rew[first:e + 1].sum() >= thr:
            succ_q += q[first:e + 1].sum()
            succ_n += e + 1 - first
        first = e + 1
    return dict(td_error=np.sum((q - y) ** 2), discounted_advantage=A, value=v.sum(), value_std=sig.sum(),
                initial_value=init, action_diff=np.sum((a - pi_rev) ** 2), success_q=succ_q, all_q=q.sum(),
                n_rows=len(r), n_episodes=len(ends), n_success_rows=succ_n)


def _close(got, want, rtol=2e-5):
    for k in OFFLINE_SUM_KEYS:
        if k.startswith("n_"):
            assert got[k] == want[k], k
        else:
            scale = max(1.0, abs(want[k]), abs(want.get("all_q", 0.0)) * 1e-3)
            assert abs(got[k] - want[k]) <= rtol * scale, (k, got[k], want[k])


@pytest.mark.parametrize("n_critics", [1, 2, 4])
def test_hand_worked_episodes_and_windows(n_critics):
    rows = _rows(LENGTHS)
    got = OM.evaluate(_state(n_critics), rows, GAMMA, return_threshold=300.0)
    want = _reference(rows, n_critics, thr=300.0)
    assert got["n_episodes"] == len(LENGTHS) and got["n_rows"] == sum(LENGTHS)
    assert 0 < got["n_success_rows"] < got["n_rows"]          # the long episodes qualify, the short ones do not
    _close(got, want)
    if n_critics == 1:
        assert got["value_std"] == 0.0


def test_window_restarts_the_advantage_recursion():
    """A 1025-row episode = a 1024-row window + a 1-row window: its sum differs from one unbroken recursion."""
    rows = _rows([1025])
    got = OM.evaluate(_state(2), rows, GAMMA)
    _close(got, _reference(rows, 2))
    q_minus_v = []
    st = _state(2)
    with torch.no_grad():
        t = torch.from_numpy(rows)
        from oracle import cql_oracle as O
        pi = O.predict_action(st, t[:, 0:2])
        q_minus_v = (O.predict_value(st, t[:, 0:2], t[:, 2:3]) - O.predict_value(st, t[:, 0:2], pi)).double().numpy()
    g = float(np.float32(GAMMA))
    unbroken = sum(float(np.sum(g ** np.arange(1025 - t) * q_minus_v[t:])) for t in range(1025))
    assert abs(got["discounted_advantage"] - unbroken) > 1e-3 * max(1.0, abs(unbroken))


def test_table_end_without_terminal_row():
    rows = _rows([3, 7, 4], last_terminal=False)
    assert rows[-1, 6] == 0 and np.all(rows[-1, 4:6] == 0)
    got = OM.evaluate(_state(2), rows, GAMMA, return_threshold=1.0)
    want = _reference(rows, 2, thr=1.0)
    assert got["n_episodes"] == 3
    _close(got, want)


def test_soft_opc_nan_when_no_episode_qualifies():
    rows = _rows([4, 6, 9])
    none = OM.evaluate(_state(2), rows, GAMMA, return_threshold=1e6)
    assert none["n_success_rows"] == 0 and none["success_q"] == 0.0
    assert np.isnan(offline_scores(none, soft_opc=True)["soft_opc"])
    every = OM.evaluate(_state(2), rows, GAMMA, return_threshold=-1.0)
    assert every["n_success_rows"] == every["n_rows"]
    assert abs(offline_scores(every, soft_opc=True)["soft_opc"]) < 1e-12
    assert "soft_opc" not in offline_scores(OM.evaluate(_state(2), rows, GAMMA), soft_opc=False)


def test_scalers_applied_as_pinned():
    rows = _rows([5, 1024, 12], seed=3)
    got = OM.evaluate(_state(4), rows, GAMMA, prep=PREP, return_threshold=4.0)
    _close(got, _reference(rows, 4, thr=4.0, prep=PREP))
    plain = OM.evaluate(_state(4), rows, GAMMA, return_threshold=4.0)
    for k in ("td_error", "value", "action_diff"):
        assert abs(got[k] - plain[k]) > 1e-3 * max(1.0, abs(plain[k])), k


def test_offline_scores_are_means():
    s = dict(td_error=8.0, discounted_advantage=-4.0, value=12.0, value_std=2.0, initial_value=3.0, action_diff=6.0,
             success_q=5.0, all_q=10.0, n_rows=4, n_episodes=2, n_success_rows=2)
    out = offline_scores(s, soft_opc=True)
    assert out == {"td_error": 2.0, "discounted_sum_of_advantage": -1.0, "average_value_estimation": 3.0,
                   "value_estimation_std": 0.5, "initial_state_value_estimation": 1.5, "continuous_action_diff": 1.5,
                   "soft_opc": 2.5 - 2.5}


def _fake_engine(n_steps=1, n_transitions=10):
    return SimpleNamespace(hp=SimpleNamespace(n_steps=n_steps), n_transitions=n_transitions)


def test_offline_metrics_argument_validation():
    m = CQL()
    with pytest.raises(AttributeError, match="not fitted"):
        m.offline_metrics()
    m.engine = _fake_engine()
    for bad in (float("nan"), float("inf"), "5", True, [1.0]):
        with pytest.raises(ValueError, match="return_threshold"):
            m.offline_metrics(return_threshold=bad)
    m.engine = _fake_engine(n_steps=3)
    with pytest.raises(ValueError, match="n-step"):
        m.offline_metrics()
    m.engine = _fake_engine(n_transitions=0)
    with pytest.raises(ValueError, match="no replay table"):
        m.offline_metrics()
    with pytest.raises(ValueError, match="empty log"):
        m.offline_metrics(pd.DataFrame({"user_idx": [], "item_idx": [], "relevance": [], "timestamp": []}))
