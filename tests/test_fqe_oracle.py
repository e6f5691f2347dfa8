"""CPU: the FQE oracle (tests/fqe_oracle.py) and the argument checks of ``replay_cql_b200.ope.FQE``.

* float32 and float64 oracles agree update by update (plain, terminal-heavy and n-step rows, scalers on);
* a second witness -- ``nn.Linear`` stacks, ``torch.optim.Adam`` and ``F.mse_loss`` -- equals the oracle over several
  updates that include target synchronisations;
* closed form: on an all-terminal minibatch the target is exactly r and the loss is sum_c mean_b (Q_c(s, a) - r)^2;
* the target schedule: a copy of the critics after updates 1, 1 + I, 1 + 2I, unchanged in between;
* ``FQE(...)`` rejects bad arguments with ``ValueError`` and an unfitted model with ``AttributeError``, before any GPU work.
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import cql_oracle as O
from replay_cql_b200 import layout
from replay_cql_b200.models import CQL
from replay_cql_b200.ope import FQE
from tests import fqe_oracle as Q

PREP = {"scaler": {"type": "standard", "mean": [3.0, 1.8], "std": [1.7, 1.1]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
        "reward_scaler": {"type": "standard", "mean": [0.3], "std": [0.45]}}


def rows_of(B, seed, term_frac=0.2, nstep=False):
    rng = np.random.default_rng(seed)
    r = np.zeros((B, 8), np.float32)
    r[:, 0:2] = rng.integers(0, 6000, (B, 2)) * np.float32(1e-3)
    r[:, 2] = rng.integers(1, 6, B) + np.float32(1e-3) * rng.standard_normal(B)
    r[:, 3] = rng.integers(0, 2, B)
    r[:, 6] = rng.random(B) < term_frac
    r[:, 4:6] = np.where(r[:, 6:7] != 0, 0, rng.integers(0, 6000, (B, 2)) * np.float32(1e-3))
    if nstep:
        r[:, 3] = rng.random(B) * 3
        r[:, 7] = np.float32(0.99) ** rng.integers(1, 4, B)
    return r


def state(C, seed=3, dtype=torch.float32):
    return Q.from_flat(layout.init_state(C, seed), C, dtype=dtype)


@pytest.mark.parametrize("kind", ["plain", "terminal", "nstep", "prep"])
@pytest.mark.parametrize("C", [1, 3])
def test_float32_matches_float64(kind, C):
    """Per update, restarted from the float32 state: loss and gradients within 1e-4.  The updated weights are gated at
    2 lr: Adam's early steps move a weight whose gradient is near zero by about lr whatever its sign, so they carry the
    sign of a gradient the two precisions may round differently."""
    lr = 1e-3
    rows = rows_of(64, 5, term_frac=0.9 if kind == "terminal" else 0.2, nstep=kind == "nstep")
    prep = PREP if kind == "prep" else None
    s32 = state(C)
    for step in range(3):
        s64 = Q.cast(s32, torch.float64)
        l32, g32 = Q.update(s32, rows, 0.99, lr, 2, nstep=kind == "nstep", prep=prep)
        l64, g64 = Q.update(s64, rows, 0.99, lr, 2, nstep=kind == "nstep", prep=prep)
        assert abs(l32 - l64) <= 1e-5 * max(1.0, abs(l64))
        for c in range(C):
            for k in Q.NET_KEYS:
                assert float((g32[c][k].double() - g64[c][k]).abs().max()) <= 1e-4 * float(g64[c][k].abs().max()) + 1e-12
                a, b = s32["critics"][c][k].double(), s64["critics"][c][k]
                assert float((a - b).abs().max()) <= 2 * lr, (step, c, k)


def _seq(net):
    """nn.Sequential(Linear, ReLU, Linear, ReLU, Linear) carrying an oracle network's tensors (d3rlpy's encoder + head)."""
    in_f, out_f = net["W1"].shape[1], net["W3"].shape[0]
    seq = nn.Sequential(nn.Linear(in_f, O.H), nn.ReLU(), nn.Linear(O.H, O.H), nn.ReLU(), nn.Linear(O.H, out_f))
    seq = seq.to(net["W1"].dtype)
    with torch.no_grad():
        for lin, (w, b) in zip((seq[0], seq[2], seq[4]), (("W1", "b1"), ("W2", "b2"), ("W3", "b3"))):
            lin.weight.copy_(net[w])
            lin.bias.copy_(net[b])
    return seq


@pytest.mark.parametrize("nstep", [False, True])
def test_second_witness_nn_modules_adam_mse(nstep):
    C, I, lr, gamma = 2, 2, 1e-3, 0.97
    st = state(C, dtype=torch.float64)
    actor = _seq(st["actor"])
    critics = [_seq(c) for c in st["critics"]]
    targets = [copy.deepcopy(c) for c in critics]
    opt = torch.optim.Adam([p for c in critics for p in c.parameters()], lr=lr, betas=(0.9, 0.999), eps=1e-8)
    for step in range(5):
        rows = rows_of(48, 10 + step, nstep=nstep)
        t = torch.from_numpy(rows).double()
        s, a, r, s1, term, disc = t[:, 0:2], t[:, 2:3], t[:, 3], t[:, 4:6], t[:, 6], t[:, 7]
        with torch.no_grad():
            pi = torch.tanh(actor(s1)[:, 0:1])
            q_t = torch.stack([q(torch.cat([s1, pi], 1))[:, 0] for q in targets]).min(0).values
            y = r + (disc if nstep else gamma) * q_t * (1 - term)
        loss = sum(F.mse_loss(q(torch.cat([s, a], 1))[:, 0], y) for q in critics)
        opt.zero_grad()
        loss.backward()
        opt.step()
        if step % I == 0:
            for q, tq in zip(critics, targets):
                tq.load_state_dict(q.state_dict())
        l_o, _ = Q.update(st, rows, gamma, lr, I, nstep=nstep)
        assert abs(l_o - float(loss.detach())) <= 1e-12 * max(1.0, abs(l_o))
        for c in range(C):
            for mod, net in ((critics[c], st["critics"][c]), (targets[c], st["targ"][c])):
                for lin, (w, b) in zip((mod[0], mod[2], mod[4]), (("W1", "b1"), ("W2", "b2"), ("W3", "b3"))):
                    assert float((lin.weight.detach() - net[w]).abs().max()) <= 1e-12, (step, c, w)
                    assert float((lin.bias.detach() - net[b]).abs().max()) <= 1e-12, (step, c, b)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_all_terminal_target_is_the_reward(dtype):
    rows = rows_of(77, 8, term_frac=1.0)
    rows[:, 3] = np.float32(0.625)
    st = state(2, dtype=dtype)
    y = Q.td_target(st, rows, 0.99)
    assert torch.equal(y, torch.full_like(y, 0.625))
    s, a, _, _, _, _ = Q.minibatch(rows, dtype)
    with torch.no_grad():
        want = sum(((O.critic_forward(c, s, a)[:, 0] - 0.625) ** 2).mean() for c in st["critics"])
    loss, _ = Q.update(st, rows, 0.99, 1e-4, 100)
    assert abs(loss - float(want)) <= 1e-12 * max(1.0, float(want))


def test_target_schedule():
    I = 3
    st = state(2)
    prev = None
    for k in range(1, 9):                       # 1-based update index
        Q.update(st, rows_of(32, k), 0.99, 1e-3, I)
        same = all(torch.equal(t[key], c[key]) for t, c in zip(st["targ"], st["critics"]) for key in Q.NET_KEYS)
        if (k - 1) % I == 0:
            assert same, k
        else:
            assert not same, k
            assert all(torch.equal(t[key], p[key]) for t, p in zip(st["targ"], prev) for key in Q.NET_KEYS), k
        prev = [{key: x.clone() for key, x in t.items()} for t in st["targ"]]


class _Fitted:
    """Stands in for a fitted model: argument checks must fail before the model's engine is touched."""
    engine = object()


@pytest.mark.parametrize("kw", [
    {"n_critics": 0}, {"n_critics": 11}, {"n_critics": 2.0}, {"batch_size": 0}, {"target_update_interval": 0},
    {"n_steps": 0}, {"n_steps": 65}, {"learning_rate": 0.0}, {"learning_rate": -1e-4}, {"learning_rate": float("nan")},
    {"learning_rate": float("inf")}, {"precision": "fp64"},
])
def test_fqe_rejects_bad_arguments(kw):
    with pytest.raises(ValueError):
        FQE(_Fitted(), **kw)
    with pytest.raises(ValueError):              # arguments first, then the model
        FQE(CQL(), **kw)


def test_fqe_rejects_an_unfitted_model():
    with pytest.raises(AttributeError, match="not fitted"):
        FQE(CQL())
