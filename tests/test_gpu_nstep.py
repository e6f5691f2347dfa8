"""GPU: n-step TD returns (d3rlpy ``n_steps``, DESIGN.md section 1) from the replay table through the update to the model.

* every table producer (chunked ingestion, the one-call builder, ``load_transitions``, ``synth_table``) writes exactly
  the oracle's n-step rows (``tests.nstep_oracle.n_step_transitions``);
* with k = 1 on every row, and for one-step host batches, n_steps > 1 takes bit for bit the steps of n_steps = 1;
* ``update_batch`` on rows of a real n = 3 expansion matches the CPU oracle with the per-row discount, under the gates
  of ``tests/test_gpu_update_shapes.py``;
* the sampled update, the provided-rows update and the phase-split path agree bit for bit on an n-step table;
* ``CQL(n_steps=3)`` fits, predicts and resumes exactly from a checkpoint.
"""
import json
import os

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import cql_oracle as O
from replay_cql_b200.mdp import build_mdp, build_mdp_on_device
from replay_cql_b200.model_handler import load, save
from replay_cql_b200.models import CQL
from replay_cql_b200.synthetic import make_log
from tests import helpers as Hp
from tests.nstep_oracle import discount_config, n_step_transitions
from tests.test_gpu_update_shapes import _Step, _compare_step

pytestmark = pytest.mark.gpu
GAMMA = 0.99            # CqlHyperParams / OracleConfig default


def _log(n, seed=0):
    """Users with episode lengths 1, n - 1, n, n + 1, long and 5 (the last user), tied timestamps, shuffled rows."""
    rng = np.random.default_rng(seed)
    lens = [1, max(1, n - 1), n, n + 1, 37, 2, 1, 5]
    cols = {"user_idx": [], "item_idx": [], "timestamp": [], "relevance": []}
    for u, L in enumerate(lens):
        cols["user_idx"] += [u] * L
        cols["item_idx"] += rng.integers(0, 300, L).tolist()
        cols["timestamp"] += rng.integers(0, L // 2 + 1, L).tolist()            # ties
        cols["relevance"] += rng.integers(1, 6, L).astype(float).tolist()
    log = pd.DataFrame(cols).sample(frac=1.0, random_state=seed).reset_index(drop=True)
    return log, rng.standard_normal(len(log)) * 1e-3


def _want(steps, n):
    return n_step_transitions(steps.obs, steps.act, steps.rew, steps.term, n, GAMMA)


def _same(got, want):
    bad = np.nonzero(~np.all(got == want, axis=1))[0]
    assert got.shape == want.shape and bad.size == 0, (bad[:5], got[bad[:3]], want[bad[:3]])


@pytest.mark.parametrize("n", [2, 3, 10])
def test_every_table_producer_writes_the_oracle_rows(engine_factory, n):
    log, noise = _log(n, seed=n)
    host = build_mdp(log, top_k=3, action_noise=noise)             # one-step steps, bit-exact with the device builder
    want = _want(host, n)
    assert (want[:, 7] == np.float32(GAMMA ** 1)).any() and (want[:, 7] < np.float32(GAMMA) ** (n - 1)).any()
    eng = engine_factory(batch_size=64, n_steps=n)
    # chunked ingestion; its host outputs stay the one-step episode steps
    obs, act, rew, term, order = build_mdp_on_device(eng, log, top_k=3, action_noise=noise, want_outputs=True)
    assert np.array_equal(obs, host.obs) and np.array_equal(act, host.act) and np.array_equal(term, host.term)
    _same(eng.export_transitions(), want)
    # the one-call builder
    eng.build_mdp_on_device(log["user_idx"], log["item_idx"], log["timestamp"], log["relevance"], top_k=3,
                            action_noise=noise)
    _same(eng.export_transitions(), want)
    # host steps
    eng.load_transitions(host.obs, host.act, host.rew, host.term)
    _same(eng.export_transitions(), want)
    # a table whose last episode has no terminal step
    cut = len(host.term) - 2
    assert host.term[cut - 1] == 0
    eng.load_transitions(host.obs[:cut], host.act[:cut], host.rew[:cut], host.term[:cut])
    _same(eng.export_transitions(), n_step_transitions(host.obs[:cut], host.act[:cut], host.rew[:cut], host.term[:cut],
                                                       n, GAMMA))
    # the synthetic table: n_steps = n == the oracle expansion of the same table at n_steps = 1
    one = engine_factory(batch_size=64)
    one.synth_table(6000, 45, 300, seed=4)
    rows1 = one.export_transitions()
    assert np.all(rows1[:, 7] == 0)
    eng.synth_table(6000, 45, 300, seed=4)
    _same(eng.export_transitions(), n_step_transitions(rows1[:, 0:2], rows1[:, 2], rows1[:, 3], rows1[:, 6], n, GAMMA))


def test_one_step_windows_reduce_to_n_steps_1(engine_factory):
    """Every user has one row (k = 1 everywhere): n_steps = 3 takes bit for bit the sampled steps of n_steps = 1.  One-step
    host batches (update_batch, update_batches: discount gamma staged) do the same on non-terminal rows."""
    rng = np.random.default_rng(1)
    U = 3000
    log = pd.DataFrame({"user_idx": np.arange(U), "item_idx": rng.integers(0, 300, U), "timestamp": np.zeros(U, np.int64),
                        "relevance": rng.integers(1, 6, U).astype(float)})
    a, b = engine_factory(batch_size=64, seed=5), engine_factory(batch_size=64, seed=5, n_steps=3)
    for e in (a, b):
        build_mdp_on_device(e, log, top_k=1)
    ta, tb = a.export_transitions(), b.export_transitions()
    assert np.array_equal(ta[:, :7], tb[:, :7]) and np.all(ta[:, 7] == 0) and np.all(tb[:, 7] == np.float32(GAMMA))
    ma, mb = a.update(5), b.update(5)
    assert ma == mb
    assert np.array_equal(a.get_state(), b.get_state())
    for x, y in zip(a.get_optimizer(), b.get_optimizer()):
        assert np.array_equal(x, y)
    batches = [Hp.batch_to_numpy(Hp.make_batch(64, seed=40 + i, scale=1e-3)) for i in range(3)]
    assert all(a.update_batch(bt)[0] == b.update_batch(bt)[0] for bt in batches)
    assert a.update_batches(batches) == b.update_batches(batches)
    assert np.array_equal(a.get_state(), b.get_state())


def _nstep_batch(B, seed, n_steps=3):
    """B rows drawn from a real n-step expansion of scaled (unsaturated) random episodes of 1..12 steps."""
    rng = np.random.default_rng(seed)
    N = 4 * B + 64
    term = np.zeros(N, np.float32)
    pos = 0
    while True:
        pos += int(rng.integers(1, 13))
        if pos > N:
            break
        term[pos - 1] = 1
    obs = np.stack([rng.integers(0, 6040, N), rng.integers(0, 3706, N)], 1).astype(np.float32) * np.float32(1e-3)
    act = ((rng.integers(1, 6, N) + 1e-3 * rng.standard_normal(N)) / 5).astype(np.float32)
    rew = rng.integers(0, 2, N).astype(np.float32)
    rows = n_step_transitions(obs, act, rew, term, n_steps, GAMMA)[rng.choice(N, B, replace=False)]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    return {"obs": t(rows[:, 0:2]), "act": t(rows[:, 2:3]), "rew": t(rows[:, 3:4]), "next_obs": t(rows[:, 4:6]),
            "term": t(rows[:, 6:7]), "discount": t(rows[:, 7:8])}


PARITY = [(37, 3, 7), (129, 2, 10), (1024, 2, 10)]


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("B,C,n", PARITY, ids=[f"B{b}-C{c}-n{n}" for b, c, n in PARITY])
def test_nstep_update_batch_matches_oracle(engine_factory, B, C, n, precision):
    """Two steps from a state with non-zero Adam moments; every metric, gradient, updated tensor and Adam moment against
    the CPU oracle with the rows' discounts (gamma, gamma^2, gamma^3, terminal rows), under the shape tests' gates."""
    cfg = O.OracleConfig(n_critics=C, n_action_samples=n)
    st = O.init_state(cfg, seed=7)
    O.update(cfg, st, Hp.make_batch(64, seed=17, scale=1e-3), O.make_noise(64, n, seed=18))       # Adam warm-up
    eng = engine_factory(batch_size=B, n_critics=C, n_action_samples=n, precision=precision, n_steps=3)
    budgeted = []
    for s in range(2):
        batch = _nstep_batch(B, seed=3000 + 10 * B + s)
        g = float(np.float32(GAMMA))
        powers = {float(np.float32(g)), float(np.float32(g * g)), float(np.float32(g * g * g))}
        assert powers <= set(batch["discount"].numpy().ravel().tolist())
        assert batch["term"].numpy().any() and not batch["term"].numpy().all()
        # the oracle takes the rows' discounts as its gamma; update_batch reads them from batch['discount']
        step = _Step(discount_config(cfg, batch["discount"]), st, batch, O.make_noise(B, n, seed=4000 + 10 * B + s))
        _compare_step(eng, step, precision, (B, C, n), s, budgeted)
    print(f"\n[{precision} B={B} C={C} n={n} n_steps=3] comparisons that needed the float64 budget: {len(budgeted)}")
    for b in budgeted:
        print("   ", b)


def _nstep_table(n_steps=3, seed=8):
    log, noise = _log(7, seed=seed)
    big = pd.concat([log.assign(user_idx=log["user_idx"] + 8 * r) for r in range(40)], ignore_index=True)
    return build_mdp(big, top_k=3, action_noise=np.tile(noise, 40))


def test_sampled_update_equals_provided_rows_and_phase_split(engine_factory):
    """On an n = 3 table: update(1) == update_batch(rows = sample_rows(B, pos=0), Philox noise) -- at world size 1 both
    draw step 0's streams -- and update(3) == three phase sequences, bit for bit."""
    steps = _nstep_table()
    B = 64
    kw = dict(batch_size=B, seed=9, n_steps=3, precision="f16x3")
    a, b, c = engine_factory(**kw), engine_factory(**kw), engine_factory(**kw)
    for e in (a, b, c):
        e.load_transitions(steps.obs, steps.act, steps.rew, steps.term)
    rows = b.sample_rows(B, pos=0).cpu().numpy()
    assert (rows[:, 7] != np.float32(GAMMA)).any()
    ma = a.update(1)
    mb, _ = b.update_batch({"obs": rows[:, 0:2], "act": rows[:, 2], "rew": rows[:, 3], "next_obs": rows[:, 4:6],
                            "term": rows[:, 6], "discount": rows[:, 7]})
    assert ma == mb
    assert np.array_equal(a.get_state(), b.get_state())
    for x, y in zip(a.get_optimizer(), b.get_optimizer()):
        assert np.array_equal(x, y)
    a.update(2)
    for _ in range(3):
        c.update_data_parallel(lambda buf: None)
    torch.cuda.synchronize()
    assert a.read_metrics() == c.read_metrics()
    assert np.array_equal(a.get_state(), c.get_state())
    for x, y in zip(a.get_optimizer(), c.get_optimizer()):
        assert np.array_equal(x, y)


def test_cql_n_steps_fit_predict():
    """CQL(n_steps=3) on the ML-1M-shaped log: fits, predicts, and learns something else than n_steps = 1."""
    log = make_log("ml1m")
    kw = dict(top_k=10, batch_size=1024, seed=3, n_steps_per_epoch=30)
    m3, m1 = CQL(n_steps=3, **kw), CQL(**kw)
    m3.fit(log)
    m1.fit(log)
    rows = m3.engine.export_transitions()
    g = float(np.float32(GAMMA))
    assert (rows[:, 7] == np.float32(g * g * g)).mean() > 0.5
    assert all(np.isfinite(v) for v in m3.last_metrics.values())
    assert not np.array_equal(m3.engine.get_state(), m1.engine.get_state())
    recs = m3.predict(log[log["user_idx"] < 50], k=5, users=list(range(50)))
    assert recs["user_idx"].nunique() == 50 and recs.groupby("user_idx").size().max() == 5
    m3.engine.close()
    m1.engine.close()


@pytest.mark.parametrize("with_table", [False, True])
def test_nstep_exact_resume_after_save_load(tmp_path, with_table):
    """fit(N) -> save -> load -> resume(M) == fit(N + M) bit for bit with n_steps = 3: the n-step table travels verbatim
    in the checkpoint or is rebuilt from the log at the model's n_steps."""
    log = make_log("tiny")
    N, M = 37, 23
    kw = dict(top_k=3, batch_size=64, seed=11, n_epochs=1, save_replay_table=with_table, n_steps=3)
    full = CQL(n_steps_per_epoch=N + M, **kw)
    full.fit(log)
    part = CQL(n_steps_per_epoch=N, **kw)
    part.fit(log)
    path = str(tmp_path / "ckpt")
    save(part, path)
    part.engine.close()
    resumed = load(path)
    assert resumed.n_steps == 3 and resumed.engine.get_optimizer()[2] == N
    if with_table:
        assert np.array_equal(resumed.engine.export_transitions(), full.engine.export_transitions())
        resumed.resume(n_steps=M)
    else:
        assert resumed.engine.n_transitions == 0
        resumed.resume(log, n_steps=M)
        assert np.array_equal(resumed.engine.export_transitions(), full.engine.export_transitions())
    assert np.array_equal(resumed.engine.get_state(), full.engine.get_state())
    m1, v1, s1 = resumed.engine.get_optimizer()
    m2, v2, s2 = full.engine.get_optimizer()
    assert s1 == s2 == N + M and np.array_equal(m1, m2) and np.array_equal(v1, v2)
    pd.testing.assert_frame_equal(resumed.predict(log, k=5), full.predict(log, k=5))
    full.engine.close()
    resumed.engine.close()


def test_checkpoint_without_n_steps_loads_as_one_step(tmp_path):
    """A checkpoint written before n_steps existed (no such init argument, table rows with slot 7 = 0) loads as n_steps = 1
    with its table bit for bit."""
    log = make_log("tiny")
    m = CQL(top_k=3, batch_size=64, seed=11, n_steps_per_epoch=5, save_replay_table=True)
    m.fit(log)
    path = str(tmp_path / "old")
    save(m, path)
    with open(os.path.join(path, "init_args.json")) as f:
        args = json.load(f)
    del args["n_steps"]
    with open(os.path.join(path, "init_args.json"), "w") as f:
        json.dump(args, f)
    old = load(path)
    assert old.n_steps == 1
    assert np.array_equal(old.engine.export_transitions(), m.engine.export_transitions())
    assert np.array_equal(old.engine.get_state(), m.engine.get_state())
    m.engine.close()
    old.engine.close()
