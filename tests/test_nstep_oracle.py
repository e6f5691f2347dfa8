"""CPU: the n-step restatement of the replay rows (d3rlpy ``n_steps``, DESIGN.md section 1), the oracle update's
per-row discount, and ``CQL(n_steps=...)`` argument handling."""
import json

import numpy as np
import pytest
import torch

from oracle import cql_oracle as O
from tests import helpers as Hp
from tests.nstep_oracle import discount_config, n_step_transitions


def _steps(lengths, rewards, terminal_tail=True):
    """Episode-ordered steps: user u = episode index, item = 10 + global step index."""
    obs, term = [], []
    for u, L in enumerate(lengths):
        for j in range(L):
            obs.append((u, 10 + len(obs)))
            term.append(1.0 if j == L - 1 and (terminal_tail or u < len(lengths) - 1) else 0.0)
    n = len(obs)
    act = np.arange(n, dtype=np.float32) / 8
    return np.asarray(obs, np.float32), act, np.asarray(rewards, np.float32), np.asarray(term, np.float32)


def test_hand_worked_episodes_1_2_5_with_n3():
    """gamma = 0.5 keeps every sum exact: the rows are written out by hand."""
    obs, act, rew, term = _steps([1, 2, 5], [1, 1, 0, 1, 0, 1, 0, 1])
    got = n_step_transitions(obs, act, rew, term, n_steps=3, gamma=0.5)
    z = (0.0, 0.0)
    #        t  R     next_obs   term  discount
    want = [(0, 1.0, z, 1.0, 0.5),          # episode of one step: k = 1
            (1, 1.0, z, 1.0, 0.25),         # k = 2: 1 + 0.5 * 0, bootstraps past the episode's terminal step (term = 1)
            (2, 0.0, z, 1.0, 0.5),
            (3, 1.25, (2, 16), 0.0, 0.125),  # k = 3: 1 + 0.5 * 0 + 0.25 * 1, s' = the step after t + 2
            (4, 0.5, (2, 17), 0.0, 0.125),
            (5, 1.25, z, 1.0, 0.125),       # window ends on the terminal step: its zeros and term = 1
            (6, 0.5, z, 1.0, 0.25),
            (7, 1.0, z, 1.0, 0.5)]
    for t, R, nx, tm, disc in want:
        row = (obs[t, 0], obs[t, 1], act[t], R, nx[0], nx[1], tm, disc)
        assert np.array_equal(got[t], np.asarray(row, np.float32)), (t, got[t], row)


def test_non_terminal_table_tail():
    """The table's end closes the last episode: windows shrink there, s' of the last step is zeros with term = 0."""
    obs, act, rew, term = _steps([2, 4], [0, 1, 1, 1, 1, 1], terminal_tail=False)
    assert term[-1] == 0
    got = n_step_transitions(obs, act, rew, term, n_steps=3, gamma=0.5)
    assert np.array_equal(got[2], np.asarray([1, 12, act[2], 1.75, 1, 15, 0, 0.125], np.float32))
    assert np.array_equal(got[3], np.asarray([1, 13, act[3], 1.75, 0, 0, 0, 0.125], np.float32))
    assert np.array_equal(got[4], np.asarray([1, 14, act[4], 1.5, 0, 0, 0, 0.25], np.float32))
    assert np.array_equal(got[5], np.asarray([1, 15, act[5], 1.0, 0, 0, 0, 0.5], np.float32))


def test_one_step_window_is_the_one_step_row():
    """n_steps = 1 (or k = 1) gives R = r and discount = (float32) gamma exactly, s' = the next step's observation."""
    rng = np.random.default_rng(3)
    n = 200
    obs = rng.integers(0, 100, (n, 2)).astype(np.float32)
    act, rew = rng.standard_normal(n).astype(np.float32), rng.random(n).astype(np.float32)
    term = (rng.random(n) < 0.2).astype(np.float32)
    got = n_step_transitions(obs, act, rew, term, n_steps=1, gamma=0.99)
    assert np.array_equal(got[:, 3], rew) and np.all(got[:, 7] == np.float32(0.99)) and np.array_equal(got[:, 6], term)
    nxt = np.zeros_like(obs)
    nxt[:-1] = obs[1:]
    nxt[term != 0] = 0
    nxt[-1] = 0
    assert np.array_equal(got[:, 4:6], nxt)


def test_float64_accumulation_order():
    """R and the discount are summed in float64 in the pinned order and rounded once to float32."""
    obs, act, rew, term = _steps([7], [0.3, 0.7, 0.1, 0.9, 0.5, 0.2, 0.4])
    rew32 = rew.astype(np.float64)
    g32 = float(np.float32(0.99))
    got = n_step_transitions(obs, act, rew, term, n_steps=5, gamma=0.99)
    R, g = 0.0, 1.0
    for j in range(5):
        R, g = R + g * rew32[j], g * g32
    assert got[0, 3] == np.float32(R) and got[0, 7] == np.float32(g)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_oracle_update_discount_gamma_equals_no_discount(dtype):
    """A per-row discount of gamma on every row takes exactly the step of the update with the scalar gamma."""
    cfg = O.OracleConfig(n_critics=2, n_action_samples=4)
    B = 48
    batch = {k: v.to(dtype) for k, v in Hp.make_batch(B, seed=21, scale=1e-3).items()}
    noise = {k: v.to(dtype) for k, v in O.make_noise(B, cfg.n_action_samples, seed=22).items()}
    st0 = O.cast_state(O.init_state(cfg, seed=7), dtype)
    a, b = O.cast_state(st0, dtype), O.cast_state(st0, dtype)
    ma, ga = O.update(cfg, a, batch, noise, want_grads=True)
    disc = torch.full((B, 1), cfg.gamma, dtype=dtype)
    mb, gb = O.update(discount_config(cfg, disc), b, batch, noise, want_grads=True)
    assert ma == mb
    assert np.array_equal(Hp.oracle_state_to_flat(a), Hp.oracle_state_to_flat(b))
    for c in range(cfg.n_critics):
        for k in O.NET_KEYS:
            assert torch.equal(ga["critics"][c][k], gb["critics"][c][k])


def test_oracle_update_reads_the_discount():
    """A different discount changes the TD target (and so the critic loss)."""
    cfg = O.OracleConfig(n_critics=2, n_action_samples=4)
    B = 32
    batch = Hp.make_batch(B, seed=5, scale=1e-3)
    noise = O.make_noise(B, cfg.n_action_samples, seed=6)
    st = O.init_state(cfg, seed=7)
    m1, _ = O.update(cfg, O.cast_state(st, torch.float32), batch, noise)
    m2, _ = O.update(discount_config(cfg, torch.full((B, 1), 0.5)), O.cast_state(st, torch.float32), batch, noise)
    assert m1["critic_loss"] != m2["critic_loss"] and m1["temp_loss"] == m2["temp_loss"]


def test_cql_n_steps_argument():
    from replay_cql_b200 import _lib
    from replay_cql_b200.models import CQL
    for bad in (0, -1, _lib.MAX_N_STEPS + 1, 2.5):
        with pytest.raises(ValueError, match="n_steps"):
            CQL(n_steps=bad)
    assert CQL().n_steps == 1 and CQL()._hyper_params().n_steps == 1
    m = CQL(n_steps=3)
    args = json.loads(json.dumps(m._init_args))
    assert args["n_steps"] == 3
    m2 = CQL(**args)
    assert m2._init_args == m._init_args and m2._hyper_params().n_steps == 3
    assert CQL(n_steps=_lib.MAX_N_STEPS).n_steps == _lib.MAX_N_STEPS


def test_header_max_n_steps_matches_binding():
    import re
    from pathlib import Path
    from replay_cql_b200 import _lib
    text = (Path(__file__).resolve().parent.parent / "include" / "cql_b200.h").read_text()
    assert int(re.search(r"#define CQL_MAX_N_STEPS (\d+)", text).group(1)) == _lib.MAX_N_STEPS
