"""GPU: d3rlpy's scalers (``scaler``, ``action_scaler``, ``reward_scaler``; DESIGN.md section 1) from the replay table's
statistics through the update and the scorers to ``CQL(...)``.

* every table producer's column statistics match the oracle fit, and are the same bits for the same steps;
* a handle with preprocessing on raw rows takes bit for bit the steps of a handle without it on the rows the oracle
  transformed -- sampled, provided-batch and phase-split updates, n_steps 1 and 3, every precision;
* parameters set (or cleared) after the update graphs were captured reach the next update;
* ``update_batch`` with all three scalers meets the oracle gates of ``tests/test_gpu_update_shapes.py``;
* the scorers use the scaled observations and (policy mode) return relevance in rating units;
* ``CQL(scaler=..., action_scaler=..., reward_scaler=...)`` fits, predicts, saves, loads and resumes exactly.
"""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import cql_oracle as O
from oracle import recs_oracle
from replay_cql_b200.mdp import build_mdp, build_mdp_on_device
from replay_cql_b200.model_handler import load, save
from replay_cql_b200.models import CQL
from replay_cql_b200.synthetic import make_log
from tests import helpers as Hp
from tests import scaler_oracle as S
from tests.test_gpu_scoring import _lists_match, _oracle_state
from tests import test_gpu_update_shapes as U
from tests.test_gpu_update_shapes import _Step, _compare_step

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
TOL = 1e-5
PREP = {"scaler": {"type": "standard", "mean": [3000.5, 1850.25], "std": [1740.0, 1070.0]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
        "reward_scaler": {"type": "standard", "mean": [0.3], "std": [0.45]}}
PREP_MM = {"scaler": {"type": "min_max", "minimum": [0.0, 0.0], "maximum": [6039.0, 3705.0]},
           "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
           "reward_scaler": {"type": "min_max", "minimum": [0.0], "maximum": [2.0]}}


def _steps(seed=0):
    log = make_log("tiny", seed=seed)
    noise = np.random.default_rng(seed).standard_normal(len(log)) * 1e-3
    return log, noise, build_mdp(log, top_k=3, action_noise=noise)


def _check_stats(got, want, rew=True):
    cols = range(4) if rew else range(3)
    for c in cols:
        assert got["count"][c] == want["count"][c]
        assert got["min"][c] == want["min"][c] and got["max"][c] == want["max"][c], c
        assert np.isclose(got["mean"][c], want["mean"][c], rtol=1e-12, atol=0), (c, got["mean"][c], want["mean"][c])
        std = np.sqrt(got["m2"][c] / got["count"][c])
        assert np.isclose(std, want["std"][c], rtol=1e-12, atol=0), (c, std, want["std"][c])
    assert got["rew_available"] == rew


def _same_bits(a, b, cols=range(4)):
    for k in ("count", "min", "max", "mean", "m2"):
        assert np.array_equal(np.asarray(a[k])[list(cols)], np.asarray(b[k])[list(cols)]), k


@pytest.mark.parametrize("n_steps", [1, 3])
def test_statistics_of_every_table_producer(engine_factory, n_steps):
    log, noise, host = _steps()
    want = S.fit(host.obs, host.act, host.rew, host.term)
    eng = engine_factory(batch_size=64, n_steps=n_steps)
    assert eng.table_stats()["count"].sum() == 0 and not eng.table_stats()["rew_available"]
    got = []
    build_mdp_on_device(eng, log, top_k=3, action_noise=noise)                      # chunked ingestion
    got.append(eng.table_stats())
    eng.build_mdp_on_device(log["user_idx"], log["item_idx"], log["timestamp"], log["relevance"], top_k=3,
                            action_noise=noise)
    got.append(eng.table_stats())
    eng.load_transitions(host.obs, host.act, host.rew, host.term)
    got.append(eng.table_stats())
    for g in got:
        _check_stats(g, want)
        _same_bits(g, got[0])
    # verbatim rows: one-step rows give the same bits; n-step rows keep obs / act and mark the reward unavailable
    eng.set_table_rows(eng.export_transitions())
    s = eng.table_stats()
    if n_steps == 1:
        _same_bits(s, got[0])
        assert s["rew_available"]
    else:
        _same_bits(s, got[0], cols=range(3))
        assert not s["rew_available"]
        with pytest.raises(ValueError, match="unavailable"):
            eng.set_preprocessing(reward_scaler="standard")
        eng.set_preprocessing(scaler="min_max", reward_scaler=PREP["reward_scaler"])     # the dict form still works
    # the synthetic table == load_transitions of the same one-step rows
    one = engine_factory(batch_size=64)
    one.synth_table(6000, 45, 300, seed=4)
    r1 = one.export_transitions()
    eng.synth_table(6000, 45, 300, seed=4)
    a = eng.table_stats()
    eng.load_transitions(r1[:, 0:2], r1[:, 2], r1[:, 3], r1[:, 6])
    _same_bits(a, eng.table_stats())
    _check_stats(a, S.fit(r1[:, 0:2], r1[:, 2], r1[:, 3], r1[:, 6]))


def _rows_to_batch(rows, discount=False):
    out = {"obs": rows[:, 0:2], "act": rows[:, 2], "rew": rows[:, 3], "next_obs": rows[:, 4:6], "term": rows[:, 6]}
    if discount:
        out["discount"] = rows[:, 7]
    return {k: np.ascontiguousarray(v) for k, v in out.items()}


def _same_learners(a, b):
    assert np.array_equal(a.get_state(), b.get_state())
    for x, y in zip(a.get_optimizer(), b.get_optimizer()):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "bf16", "f16x3"])
@pytest.mark.parametrize("n_steps", [1, 3])
def test_scaled_handle_equals_unscaled_handle_on_transformed_rows(engine_factory, precision, n_steps):
    """P on raw rows == no P on T(rows), bit for bit: state, both Adam moments and metrics."""
    _, _, host = _steps()
    B = 64
    kw = dict(batch_size=B, seed=5, precision=precision, n_steps=n_steps)
    a, b = engine_factory(**kw), engine_factory(**kw)
    a.load_transitions(host.obs, host.act, host.rew, host.term)
    a.set_preprocessing(**PREP)
    raw = a.export_transitions()
    b.set_table_rows(S.transform_rows(PREP, raw))
    assert a.update(3) == b.update(3)
    _same_learners(a, b)
    rng = np.random.default_rng(n_steps)
    picks = [raw[rng.choice(len(raw), B, replace=False)] for _ in range(3)]
    for rows in picks:                       # table rows (with their discount when n_steps > 1)
        assert a.update_batch(_rows_to_batch(rows, n_steps > 1))[0] == \
            b.update_batch(_rows_to_batch(S.transform_rows(PREP, rows), n_steps > 1))[0]
    _same_learners(a, b)
    for i, rows in enumerate(picks):         # caller-provided noise (the second staged-batch graph)
        nz = Hp.noise_to_numpy(O.make_noise(B, 10, seed=70 + i))
        assert a.update_batch(_rows_to_batch(rows, n_steps > 1), nz)[0] == \
            b.update_batch(_rows_to_batch(S.transform_rows(PREP, rows), n_steps > 1), nz)[0]
    _same_learners(a, b)
    one_step = [_rows_to_batch(r) for r in picks]
    scaled = [_rows_to_batch(S.transform_rows(PREP, r)) for r in picks]
    assert a.update_batches(one_step) == b.update_batches(scaled)
    _same_learners(a, b)
    for x, y in zip(one_step, scaled):       # phase split on uploaded batches (phase 4), and sampled (phase 0)
        a.upload_batch(x)
        a.update_data_parallel(lambda buf: None, uploaded_batch=True)
        b.upload_batch(y)
        b.update_data_parallel(lambda buf: None, uploaded_batch=True)
    for _ in range(2):                       # phase 4 replayed on one upload: the staged rows stay raw
        a.update_data_parallel(lambda buf: None, uploaded_batch=True)
        b.update_data_parallel(lambda buf: None, uploaded_batch=True)
    a.update_data_parallel(lambda buf: None)
    b.update_data_parallel(lambda buf: None)
    torch.cuda.synchronize()
    assert a.read_metrics() == b.read_metrics()
    _same_learners(a, b)


def test_parameters_set_after_graph_capture(engine_factory):
    _, _, host = _steps(1)
    kw = dict(batch_size=64, seed=6)
    a, b = engine_factory(**kw), engine_factory(**kw)
    for e in (a, b):
        e.load_transitions(host.obs, host.act, host.rew, host.term)
    raw = a.export_transitions()
    bt = _rows_to_batch(raw[:64])
    assert a.update(2) == b.update(2) and a.update_batch(bt)[0] == b.update_batch(bt)[0]     # graphs captured
    a.set_preprocessing(**PREP_MM)
    b.set_table_rows(S.transform_rows(PREP_MM, raw))
    assert a.update(2) == b.update(2)
    assert a.update_batch(bt)[0] == b.update_batch(_rows_to_batch(S.transform_rows(PREP_MM, raw[:64])))[0]
    _same_learners(a, b)
    a.set_preprocessing()                                          # cleared: the unscaled bits again
    assert all(v is None for v in a.get_preprocessing().values())
    b.set_table_rows(raw)
    assert a.update(2) == b.update(2) and a.update_batch(bt)[0] == b.update_batch(bt)[0]
    _same_learners(a, b)


class _RawBatchEngine:
    """The engine as ``_compare_step`` sees it: the step's batch is the oracle's transformed one; the engine, which applies
    the scalers itself, gets the raw batch that was transformed."""

    def __init__(self, eng, raw, prep):
        self.eng, self.raw, self.scaled = eng, Hp.batch_to_numpy(raw), Hp.batch_to_numpy(S.transform_batch(prep, raw))

    def update_batch(self, batch, noise=None, want_grads=False):
        for k, v in self.scaled.items():
            assert np.array_equal(np.asarray(batch[k]), v), k
        return self.eng.update_batch(self.raw, noise, want_grads=want_grads)

    def __getattr__(self, name):
        return getattr(self.eng, name)


GATES = [(37, 3, 7), (1024, 2, 10)]


# Looser gates of the standard-scaler cases, in the style of tests/test_gpu_update_shapes.py's LOOSER (same key and
# value layout, applied to that module's tables for this test only), measured on a B200 with these seeds by
# tests/_diag_scaler_gates.py: each miss is one ReLU flip, reproduced by toggling that one mask in the float64 oracle.
# ("Call" counts the oracle update's network evaluations in order.)
SCALER_LOOSER = {
    ("tf32x3", (37, 3, 7), 0, ("critic", 1)): (
        ("W2",), 5e-4, ("grads", "moments", "state"),
        "layer-2 flip: critic 1, call 31, row 198, unit 193, pre-activation 1.48e-7 of the row's largest.  Against the "
        "float64 oracle the GPU's dW2 / db2 are off by 1.06e-4 / 1.20e-4 (max-norm) and the updated W2 by 1.77e-4; with "
        "that mask toggled by 2.7e-7 / 3.0e-7 and 5.3e-7."),
    ("tf32x3", (1024, 2, 10), 1, ("actor",)): (
        ("W2",), 5e-3, ("grads", "moments", "state"),
        "layer-2 flip: actor, call 26, row 104, unit 71, pre-activation 4.75e-8 of the row's largest.  Against the "
        "float64 oracle the GPU's dW2 is off by 2.47e-3 (max-norm) and the updated W2 by 1.08e-4; with that mask toggled "
        "by 1.4e-6 and 1.2e-7.  The flip also lifts the step's median gradient L2 error to 2.63e-5 (MEDIAN_LOOSER)."),
    ("f16x3", (1024, 2, 10), 1, ("actor",)): (
        ("W2",), 5e-3, ("grads", "moments", "state"),
        "the same flip as tf32x3 (actor, call 26, row 104, unit 71, 4.75e-8): dW2 off by 2.47e-3 and W2 by 1.08e-4 "
        "against the float64 oracle, by 8.7e-7 and 1.2e-7 with the mask toggled."),
}
SCALER_MEDIAN_LOOSER = {("tf32x3", (1024, 2, 10), 1): 3e-5}
PREPS = [pytest.param(p, q, id=f"{p}-{q}") for p in ("standard", "min_max") for q in ("fp32", "tf32x3", "f16x3")]


@pytest.mark.parametrize("prep,precision", PREPS)
@pytest.mark.parametrize("B,C,n", GATES, ids=[f"B{b}-C{c}-n{n}" for b, c, n in GATES])
def test_scaled_update_batch_matches_oracle(engine_factory, monkeypatch, B, C, n, precision, prep):
    """Raw minibatches (ids, ratings 1..5, terminal rows with s' = 0) through the engine's scalers against the CPU oracle
    on the transformed minibatches, two steps from a state with non-zero Adam moments.  Every gate of the shape tests;
    the standard-scaler cases take the named allowances of SCALER_LOOSER."""
    if prep == "standard":
        for key, val in SCALER_LOOSER.items():
            monkeypatch.setitem(U.LOOSER, key, val)
        for key, val in SCALER_MEDIAN_LOOSER.items():
            monkeypatch.setitem(U.MEDIAN_LOOSER, key, val)
    cfg = O.OracleConfig(n_critics=C, n_action_samples=n)
    st = O.init_state(cfg, seed=7)
    O.update(cfg, st, Hp.make_batch(64, seed=17, scale=1e-3), O.make_noise(64, n, seed=18))       # Adam warm-up
    eng = engine_factory(batch_size=B, n_critics=C, n_action_samples=n, precision=precision)
    P = PREP if prep == "standard" else PREP_MM
    eng.set_preprocessing(**P)
    budgeted = []
    for s in range(2):
        raw = Hp.make_batch(B, seed=5000 + 10 * B + s, term_frac=0.2)
        assert raw["term"].numpy().any()
        step = _Step(cfg, st, S.transform_batch(P, raw), O.make_noise(B, n, seed=6000 + 10 * B + s))
        _compare_step(_RawBatchEngine(eng, raw, P), step, precision, (B, C, n), s, budgeted)
    print(f"\n[{precision} B={B} C={C} n={n} scalers] comparisons that needed the float64 budget: {len(budgeted)}")


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("mode", ["q", "policy"])
def test_scoring_with_scalers(engine_factory, precision, mode):
    flat, st = _oracle_state(11)
    eng = engine_factory(batch_size=64, precision=precision)
    eng.set_state(flat)
    prep = eng.set_preprocessing(scaler=PREP["scaler"], action_scaler=PREP["action_scaler"])
    rng = np.random.default_rng(3)
    users = np.sort(rng.choice(6040, size=6, replace=False)).astype(np.int32)
    items = np.sort(rng.choice(3706, size=2500, replace=False)).astype(np.int32)
    seen = {int(u): set(rng.choice(items, size=40, replace=False).tolist()) for u in users}
    indptr = np.zeros(int(users.max()) + 2, dtype=np.int64)
    flat_seen = []
    for u in range(int(users.max()) + 1):
        flat_seen.extend(sorted(seen.get(u, ())))
        indptr[u + 1] = len(flat_seen)
    flat_seen = np.asarray(flat_seen, dtype=np.int32)

    def score(obs):
        r = O.relevance(st, S.obs_fwd(prep["scaler"], torch.from_numpy(np.asarray(obs, np.float32))), mode)
        return (S.act_rev(prep["action_scaler"], r) if mode == "policy" else r).numpy()

    k = 10
    ri, rs = recs_oracle.brute_force_topk(score, users, items, seen, k)
    ti, ts = eng.score_topk(users, items, k, indptr, flat_seen, mode=mode)
    _lists_match(ti, ts, ri, rs)
    dev = torch.device("cuda", eng.device)
    di, ds = eng.score_topk_device(torch.from_numpy(users).to(dev), torch.from_numpy(items).to(dev), k,
                                   torch.from_numpy(indptr).to(dev), torch.from_numpy(flat_seen).to(dev), mode=mode)
    assert np.array_equal(di.cpu().numpy(), ti) and np.array_equal(ds.cpu().numpy(), ts)
    pu, pi = rng.integers(0, 6040, 700).astype(np.int32), rng.integers(0, 3706, 700).astype(np.int32)
    ps = eng.score_pairs(pu, pi, mode=mode)
    want = score(np.stack([pu, pi], 1).astype(np.float32)).reshape(-1)
    assert np.max(np.abs(ps - want)) <= TOL * max(1.0, float(np.max(np.abs(want))))
    if mode == "policy":                 # relevance in rating units, inside the action range (to the ulp the reverse
        for v in (ts[np.isfinite(ts)], ps):  # transform's last addition may round a saturated tanh past maximum)
            assert v.min() >= np.float32(0.99) and v.max() <= np.nextafter(np.float32(5.01), np.float32(np.inf))
    # cleared: the same bits as a handle that never had preprocessing
    fresh = engine_factory(batch_size=64, precision=precision)
    fresh.set_state(flat)
    eng.set_preprocessing()
    for e_args in ((users, items, k, indptr, flat_seen),):
        x, y = eng.score_topk(*e_args, mode=mode), fresh.score_topk(*e_args, mode=mode)
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])
    assert np.array_equal(eng.score_pairs(pu, pi, mode=mode), fresh.score_pairs(pu, pi, mode=mode))


SCALED = dict(scaler="standard", action_scaler="min_max", reward_scaler="standard")


def test_cql_scalers_fit_predict_save_load(tmp_path):
    log = make_log("tiny")
    kw = dict(top_k=3, batch_size=64, seed=3, n_steps_per_epoch=25)
    m, plain = CQL(**SCALED, **kw), CQL(**kw)
    m.fit(log)
    plain.fit(log)
    rows = m.engine.export_transitions()
    assert np.array_equal(rows, plain.engine.export_transitions())           # the table stays raw
    o = S.fit(rows[:, 0:2], rows[:, 2], rows[:, 3], rows[:, 6])
    prep = m.engine.get_preprocessing()
    for arg, kind, cols in (("scaler", "standard", (0, 1)), ("action_scaler", "min_max", (2,)),
                            ("reward_scaler", "standard", (3,))):
        want = S.params(kind, cols, o)
        for key in want:
            if key != "type":
                assert np.allclose(prep[arg][key], want[key], rtol=2 ** -22, atol=0), (arg, key)   # one float32 ulp
    assert not np.array_equal(m.engine.get_state(), plain.engine.get_state())
    assert all(np.isfinite(v) for v in m.last_metrics.values())
    recs = m.predict(log, k=5)
    assert len(recs) > 0
    path = str(tmp_path / "scaled")
    save(m, path)
    back = load(path)
    assert back.engine.get_preprocessing() == prep
    pd.testing.assert_frame_equal(back.predict(log, k=5), recs)
    pol = CQL(**dict(SCALED, score="policy"), **kw)
    pol.fit(log)
    pr = pol.predict(log, k=5)["relevance"].to_numpy()
    assert pr.min() >= rows[:, 2].min() and pr.max() <= np.nextafter(rows[:, 2].max(), np.float32(np.inf))
    for e in (m, plain, back, pol):
        e.engine.close()


@pytest.mark.parametrize("with_table", [False, True])
def test_scaled_exact_resume_after_save_load(tmp_path, with_table):
    log = make_log("tiny")
    N, M = 31, 17
    kw = dict(top_k=3, batch_size=64, seed=12, n_epochs=1, save_replay_table=with_table, **SCALED)
    full = CQL(n_steps_per_epoch=N + M, **kw)
    full.fit(log)
    part = CQL(n_steps_per_epoch=N, **kw)
    part.fit(log)
    path = str(tmp_path / "ckpt")
    save(part, path)
    part.engine.close()
    resumed = load(path)
    assert resumed.engine.get_preprocessing() == full.engine.get_preprocessing()
    if with_table:
        resumed.resume(n_steps=M)
    else:
        assert resumed.engine.n_transitions == 0
        resumed.resume(log, n_steps=M)
    assert np.array_equal(resumed.engine.get_state(), full.engine.get_state())
    m1, v1, s1 = resumed.engine.get_optimizer()
    m2, v2, s2 = full.engine.get_optimizer()
    assert s1 == s2 == N + M and np.array_equal(m1, m2) and np.array_equal(v1, v2)
    pd.testing.assert_frame_equal(resumed.predict(log, k=5), full.predict(log, k=5))
    full.engine.close()
    resumed.engine.close()


def test_checkpoint_without_scalers_loads_unscaled(tmp_path):
    """A checkpoint written before the scalers existed (no such init arguments, no parameters in meta.json)."""
    log = make_log("tiny")
    m = CQL(top_k=3, batch_size=64, seed=11, n_steps_per_epoch=5)
    m.fit(log)
    path = str(tmp_path / "old")
    save(m, path)
    with open(os.path.join(path, "init_args.json")) as f:
        args = json.load(f)
    for k in ("scaler", "action_scaler", "reward_scaler"):
        del args[k]
    with open(os.path.join(path, "init_args.json"), "w") as f:
        json.dump(args, f)
    old = load(path)
    assert old.scaler is None and all(v is None for v in old.engine.get_preprocessing().values())
    pd.testing.assert_frame_equal(old.predict(log, k=5), m.predict(log, k=5))
    m.engine.close()
    old.engine.close()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_fit_gives_the_same_parameters_on_every_rank():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29541", "tests/_scalers_dp_check.py"],
                         cwd=ROOT, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    lines = sorted(l for l in out.stdout.splitlines() if l.startswith("rank "))
    assert len(lines) == 2
    assert lines[0].split(" ", 2)[2] == lines[1].split(" ", 2)[2], lines
