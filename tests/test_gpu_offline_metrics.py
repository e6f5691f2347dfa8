"""GPU: d3rlpy's offline scorers (``cql_offline_eval``, ``CQL.offline_metrics``; DESIGN.md section 1).

* the sums match the oracle (tests/offline_metrics_oracle.py) at every FP32-grade precision, critic count 1..4, table
  sizes around the forward chunk and the 1024-row window, with the scalers off and on (gates: DESIGN.md tolerance table);
* two calls, a side stream, and a table loaded verbatim versus built by the MDP builder give the same bits;
* a permutation of whole episodes gives the same sums within float64 reordering;
* the call leaves the model as it was: fit -> offline_metrics -> resume equals fit -> resume;
* n_steps = 3 needs the log and then equals an n_steps = 1 model with the same networks; save / load keeps the result;
* two GPUs: sharded evaluation equals one engine's.
"""
import functools
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import cql_oracle as O
from replay_cql_b200 import _lib, layout
from replay_cql_b200.engine import OFFLINE_SUM_KEYS, offline_scores
from replay_cql_b200.mdp import build_mdp_on_device
from replay_cql_b200.model_handler import load, save
from replay_cql_b200.models import CQL
from replay_cql_b200.synthetic import make_log
from tests import helpers as Hp
from tests import offline_metrics_oracle as OM

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
CHUNK = 1 << 18                      # OE_CHUNK of csrc/offline_eval.cuh
TOL = 1e-5                           # per value, relative to max|Q| (DESIGN.md tolerance table)
GAMMA = 0.99
PREP = {"scaler": {"type": "standard", "mean": [3.0, 1.8], "std": [1.7, 1.1]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
        "reward_scaler": {"type": "standard", "mean": [0.3], "std": [0.45]}}


@functools.lru_cache(maxsize=None)
def _rows(n, seed=0):
    """n one-step rows: episodes of 1..3000 steps (the last one without a terminal row when it is cut by n), ids
    scaled by 1e-3 (the policy is not saturated), s' = the next s; ~0.1 % of the non-terminal rows carry an s' that is
    not the next row's s (the explicit-s' path)."""
    rng = np.random.default_rng(seed)
    lens, total = [], 0
    while total < n:
        lens.append(int(min(n - total, rng.choice([1, 2, 5, 1023, 1024, 1025, int(rng.integers(3, 3000))]))))
        total += lens[-1]
    obs = np.stack([rng.integers(0, 6040, n), rng.integers(0, 3706, n)], 1).astype(np.float32) * np.float32(1e-3)
    rows = np.zeros((n, 8), np.float32)
    rows[:, 0:2] = obs
    rows[:, 2] = rng.integers(1, 6, n).astype(np.float32) + np.float32(1e-3) * rng.standard_normal(n).astype(np.float32)
    rows[:, 3] = (rng.random(n) < 0.2).astype(np.float32)
    ends = np.cumsum(lens) - 1
    rows[ends, 6] = 1.0
    if n > 2 and seed % 2 == 0:
        rows[-1, 6] = 0.0                                        # the table ends inside an episode
    nxt = np.concatenate([obs[1:], np.zeros((1, 2), np.float32)])
    rows[:, 4:6] = np.where(rows[:, 6:7] != 0, 0.0, nxt)
    odd = np.flatnonzero((rows[:, 6] == 0) & (rng.random(n) < 1e-3))
    rows[odd, 4:6] = rows[odd, 4:6] + np.float32(0.125)
    return rows


@functools.lru_cache(maxsize=None)
def _flat(C, seed=1):
    return layout.init_state(C, seed, 1.0, 1.0)


@functools.lru_cache(maxsize=None)
def _oracle(C, n, prep_on, thr=2.0):
    st = Hp.flat_to_oracle_state(_flat(C), O.OracleConfig(n_critics=C))
    rows = _rows(n)
    sums = OM.evaluate(st, rows, GAMMA, prep=PREP if prep_on else None, return_threshold=thr)
    with torch.no_grad():
        t = torch.from_numpy(rows)
        obs = t[:, 0:2] if not prep_on else (t[:, 0:2] - torch.tensor(PREP["scaler"]["mean"])) / (
            torch.tensor(PREP["scaler"]["std"]) + np.float32(1e-3))
        qmax = float(O.q_ensemble(st["critics"], obs, O.predict_action(st, obs)).abs().max())
    return sums, max(1.0, qmax)


def _engine(engine_factory, precision, C, prep_on):
    eng = engine_factory(batch_size=64, n_critics=C, precision=precision, gamma=GAMMA)
    eng.set_state(_flat(C))
    if prep_on:
        eng.set_preprocessing(**PREP)
    return eng


def _check(got, want, qmax, what):
    """Metric gates: TOL x the metric's scale -- max|Q| for the values, max|Q|^2 and max|a|^2 for the squares, and
    max|Q| / (1 - gamma) for the windowed advantage sums."""
    g, w = offline_scores(got, True), offline_scores(want, True)
    for k in OFFLINE_SUM_KEYS:
        if k.startswith("n_"):
            assert got[k] == want[k], (what, k)
    scale = {"td_error": qmax * qmax, "continuous_action_diff": 36.0, "discounted_sum_of_advantage": qmax / (1 - GAMMA)}
    for k, v in w.items():
        if np.isnan(v):
            assert np.isnan(g[k]), (what, k)
            continue
        assert abs(g[k] - v) <= TOL * scale.get(k, qmax), (what, k, g[k], v)


@pytest.mark.parametrize("prep_on", [False, True])
@pytest.mark.parametrize("C", [1, 2, 3, 4])
@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_small_tables_against_oracle(engine_factory, precision, C, prep_on):
    eng = _engine(engine_factory, precision, C, prep_on)
    for n in (1, 2, 2100, 5000):
        eng.set_table_rows(_rows(n))
        want, qmax = _oracle(C, n, prep_on)
        got = eng.offline_metrics(2.0)
        _check(got, want, qmax, (precision, C, prep_on, n))
        if C == 1:
            assert got["value_std"] == 0.0


@pytest.mark.parametrize("n", [CHUNK - 1, CHUNK + 1, 2 * CHUNK + 3])
@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_chunk_boundaries_against_oracle(engine_factory, precision, n):
    eng = _engine(engine_factory, precision, 2, True)
    eng.set_table_rows(_rows(n))
    want, qmax = _oracle(2, n, True)
    _check(eng.offline_metrics(2.0), want, qmax, (precision, n))


def test_ml1m_shape_against_oracle(engine_factory):
    n = 1_000_209
    eng = _engine(engine_factory, "f16x3", 2, False)
    eng.set_table_rows(_rows(n))
    want, qmax = _oracle(2, n, False)
    _check(eng.offline_metrics(2.0), want, qmax, "ml1m")


def test_bits_do_not_depend_on_call_stream_or_table_producer(engine_factory):
    log = make_log("tiny", seed=3)
    for precision in ("fp32", "f16x3"):
        a = _engine(engine_factory, precision, 2, True)
        build_mdp_on_device(a, log, top_k=3)
        first = a.offline_metrics(1.0)
        assert a.offline_metrics(1.0) == first
        side = torch.cuda.Stream()
        assert a.offline_metrics(1.0, stream=side.cuda_stream) == first
        b = _engine(engine_factory, precision, 2, True)
        b.set_table_rows(a.export_transitions())
        assert b.offline_metrics(1.0) == first
        big = _engine(engine_factory, precision, 2, False)      # several chunks
        big.set_table_rows(_rows(2 * CHUNK + 3))
        assert big.offline_metrics() == big.offline_metrics()


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_episode_permutation(engine_factory, precision):
    rows = _rows(200_000, seed=1)                                  # one chunk, every episode ends with a terminal row
    ends = np.flatnonzero(rows[:, 6] != 0)
    assert ends[-1] == len(rows) - 1
    eps = np.split(np.arange(len(rows)), ends[:-1] + 1)
    perm = np.random.default_rng(5).permutation(len(eps))
    shuffled = rows[np.concatenate([eps[i] for i in perm])]
    eng = _engine(engine_factory, precision, 3, True)
    eng.set_table_rows(rows)
    a = eng.offline_metrics(1.5)
    eng.set_table_rows(shuffled)
    b = eng.offline_metrics(1.5)
    for k in OFFLINE_SUM_KEYS:
        assert abs(a[k] - b[k]) <= 1e-12 * max(1.0, abs(a[k])), (k, a[k], b[k])


def _fit(**kw):
    m = CQL(top_k=3, batch_size=64, seed=11, n_steps_per_epoch=5, **kw)
    m.fit(make_log("tiny", seed=2))
    return m


def _learner(m):
    return m.engine.get_state(), m.engine.get_optimizer()


def test_no_side_effects_on_training():
    a, b = _fit(scaler="min_max"), _fit(scaler="min_max")
    launches = a.engine.launch_count
    a.offline_metrics(return_threshold=1.0)
    a.offline_metrics(make_log("tiny", seed=2))
    assert a.engine.launch_count > launches
    a.resume(n_steps=7)
    b.resume(n_steps=7)
    (sa, (ma, va, ka)), (sb, (mb, vb, kb)) = _learner(a), _learner(b)
    assert np.array_equal(sa, sb) and np.array_equal(ma, mb) and np.array_equal(va, vb) and ka == kb
    assert a.last_metrics == b.last_metrics


def test_n_steps_model_needs_the_log_and_matches_one_step():
    log = make_log("tiny", seed=2)
    m3 = _fit(n_steps=3)
    with pytest.raises(ValueError, match="n-step"):
        m3.offline_metrics()
    with pytest.raises(_lib.CqlArgumentError, match="n-step"):
        m3.engine.offline_metrics()
    m1 = _fit()
    m1.engine.set_state(m3.engine.get_state())
    assert m3.offline_metrics(log, return_threshold=1.0) == m1.offline_metrics(log, return_threshold=1.0)
    assert m1.offline_metrics(log) == m1.offline_metrics()          # the same builder rebuilds the fitted table


def test_save_load_keeps_the_result(tmp_path):
    log = make_log("tiny", seed=2)
    m = _fit(action_scaler="min_max")
    before = m.offline_metrics(log, return_threshold=1.0)
    save(m, str(tmp_path / "m"))
    m2 = load(str(tmp_path / "m"))
    with pytest.raises(ValueError, match="no replay table"):
        m2.offline_metrics()
    assert m2.offline_metrics(log, return_threshold=1.0) == before


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_equal_one():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29541", "tests/_offline_metrics_dp_check.py"],
                         cwd=ROOT, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    res = {int(l.split()[1]): json.loads(l.split(" result ", 1)[1]) for l in out.stdout.splitlines() if " result " in l}
    assert set(res) == {0, 1}
    assert res[0]["table"] == res[1]["table"] and res[0]["log"] == res[1]["log"]
    for part in ("table", "log"):
        for k, v in res[0]["single"].items():
            assert abs(res[0][part][k] - v) <= 1e-12 * max(1.0, abs(v)), (part, k)
