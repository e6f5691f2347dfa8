"""GPU: critic ensembles of 5..10 and 11..32 action samples (``CQL_MAX_CRITICS`` = 10, ``CQL_MAX_ACTION_SAMPLES`` = 32).

With 3n + 1 > 32 rows per (critic, batch element) ``k_lse`` takes its wide path (``k_lse<true>``, lane l holds rows
l, l + 32, ...).  The update matrix below reaches the f16x3 dispatch cells with the new shapes (148-SM B200; critic rows =
B (3n + 1)):

    B, C, n        critic rows   critic fwd / bwd   actor-step fwd / dx-bwd1
    1, 5, 11       34            small              small
    37, 7, 16      1 813         regular            small
    300, 10, 21    19 200        pair               small
    1024, 10, 32   99 328        pair               regular
    8192, 5, 11    278 528       pair               pair

The parity gates are those of ``tests/test_gpu_update_shapes.py`` (same helpers, same float64 budget rule).  Scoring,
the offline scorers and the model-level checks reuse the gates of ``test_gpu_scoring_shapes.py``,
``test_gpu_offline_metrics.py`` and ``test_gpu_sampler_and_model.py`` at the new critic counts.
"""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch

from replay_cql_b200 import _lib
from replay_cql_b200.engine import CqlEngine, CqlHyperParams
from tests import test_gpu_offline_metrics as OMT
from tests import test_gpu_scoring_shapes as SS
from tests import test_gpu_update_shapes as US

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

CASES = [(1, 5, 11), (37, 7, 16), (300, 10, 21), (1024, 10, 32), (8192, 5, 11)]
SMALLER = CASES[:4]
_ids = lambda cases: [f"B{b}-C{c}-n{n}" for b, c, n in cases]


# ---------------------------------------------------------------- 1. update parity against the float32 oracle
# Looser gates, each for named tensors of one case, in the format of test_gpu_update_shapes.LOOSER, with what was measured
# on a B200 (148 SMs) with these seeds.  All are layer-2 ReLU flips (test_gpu_update_shapes.py, note above LOOSER): the
# error of the tensor sits in one row -- one hidden unit -- and the float32 oracle has a pre-activation of that unit
# within 1e-6 of its row's largest, which any other summation order may put on the other side of zero.
_FLIP = "layer-2 flip, critic {c} unit {u}: pre-activation {m} of its row's largest at {where} in the oracle; "
LOOSER = {
    ("f16x3", (1024, 10, 32), 0, ("critic", 6)): (
        ("W2",), 1e-3, ("state",),
        _FLIP.format(c=6, u=239, m="4.0e-8", where="sample row 14306") +
        "updated W2 misses by 3.2e-4, 98 % of the squared error in row 239 (tf32x3: the same 3.2e-4, 99.8 %)"),
    ("f16x3", (1024, 10, 32), 1, ("critic", 8)): (
        ("W2",), 1e-3, ("state",),
        _FLIP.format(c=8, u=9, m="5.6e-8", where="sample row 8657") +
        "updated W2 misses by 1.1e-4, 87 % of the squared error in row 9 (tf32x3: 96 %)"),
    ("tf32x3", (1024, 10, 32), 0, ("critic", 2)): (
        ("W1", "W2", "b2"), 1e-2, ("grads", "moments", "state"),
        _FLIP.format(c=2, u=29, m="6.1e-7", where="data row 564 (the row that carries the TD and the conservative dQ)") +
        "dW2 misses by 6.8e-3 (max) / 1.2e-3 (L2) and db2 by 4.5e-3, > 99 % of the squared error in row 29; dW1 by "
        "1.1e-3 (L2, spread over the rows: dz2 of unit 29 feeds every unit of layer 1); updated W2 by 1.6e-4"),
}
LOOSER[("tf32x3", (1024, 10, 32), 0, ("critic", 6))] = LOOSER[("f16x3", (1024, 10, 32), 0, ("critic", 6))]
LOOSER[("tf32x3", (1024, 10, 32), 1, ("critic", 8))] = LOOSER[("f16x3", (1024, 10, 32), 1, ("critic", 8))]


@pytest.fixture
def looser(monkeypatch):
    monkeypatch.setattr(US, "LOOSER", {**US.LOOSER, **LOOSER})


@pytest.mark.parametrize("B,C,n", CASES, ids=_ids(CASES))
def test_f16x3_update_matches_oracle_large_ensemble(engine_factory, looser, B, C, n):
    US._run_case(engine_factory, B, C, n, "f16x3")


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
@pytest.mark.parametrize("B,C,n", SMALLER, ids=_ids(SMALLER))
def test_fp32_grade_update_matches_oracle_large_ensemble(engine_factory, looser, B, C, n, precision):
    US._run_case(engine_factory, B, C, n, precision)


@pytest.mark.parametrize("B,C,n", [(37, 7, 16), (1024, 10, 32)], ids=_ids([(37, 7, 16), (1024, 10, 32)]))
def test_bf16_losses_large_ensemble(engine_factory, B, C, n):
    """bf16: the six losses within its stated 2e-2 of the float32 oracle."""
    US.test_bf16_losses_at_shape(engine_factory, B, C, n)


# ---------------------------------------------------------------- 2. determinism at (C, n) = (10, 32)
CHILD = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from replay_cql_b200.engine import CqlEngine, CqlHyperParams
out = {}
for tag in ("a", "b"):
    eng = CqlEngine(CqlHyperParams(batch_size=1024, n_critics=10, n_action_samples=32, seed=777, precision="f16x3"), device=0)
    eng.synth_table(1_000_003, 6040, 3706, seed=777)
    eng.update(20, want_metrics=False)
    m, v, step = eng.get_optimizer()
    out.update({tag + "_state": eng.get_state(), tag + "_adam_m": m, tag + "_adam_v": v, tag + "_step": np.int64(step),
                tag + "_metrics": np.array(list(eng.read_metrics().values()), dtype=np.float32)})
    eng.close()
np.savez(sys.argv[2], **out)
"""
ARMS = {"default": {}, "no_fold": {"CQL_NO_FOLD": "1"}, "no_pdl": {"CQL_NO_PDL": "1"}}


def test_two_handles_and_switches_are_bit_identical(tmp_path):
    """Two handles with one seed take bit-identical steps (20 sampled f16x3 updates at B = 1024, C = 10, n = 32: the wide
    k_lse path); CQL_NO_FOLD=1 and CQL_NO_PDL=1 leave every bit of state, moments and metrics as they are."""
    out = {}
    for arm, extra in ARMS.items():
        env = {k: v for k, v in os.environ.items() if not k.startswith("CQL_")}
        env.update(extra)
        path = tmp_path / f"{arm}.npz"
        p = subprocess.run([sys.executable, "-c", CHILD, str(ROOT), str(path)], cwd=ROOT, env=env, capture_output=True,
                           text=True, timeout=900)
        assert p.returncode == 0, f"{arm}:\n{p.stdout}\n{p.stderr}"
        out[arm] = np.load(path)
    ref = out["default"]
    assert int(ref["a_step"]) == 20
    assert np.all(np.isfinite(ref["a_metrics"])), ref["a_metrics"]
    for key in ("state", "adam_m", "adam_v", "step", "metrics"):
        assert np.array_equal(ref["a_" + key], ref["b_" + key]), f"two handles: {key}"
        for arm in ("no_fold", "no_pdl"):
            assert np.array_equal(ref["a_" + key], out[arm]["a_" + key]), f"{arm}: {key} differs from the default schedule"


# ---------------------------------------------------------------- 3. scoring at C = 5 and 10
TOPK_CASES = [(1, 1, 1, False), (3, 129, 33, False), (4, 4097, 10, False)]       # k = 1, 33, 10
TOPK = [pytest.param(p, C, m, c, id=f"{p}-C{C}-{m}-{SS._case_id(c)}") for C in (5, 10) for m in ("q", "policy")
        for c in TOPK_CASES for p in SS.PRECISIONS]


@pytest.mark.parametrize("precision,C,mode,case", TOPK)
def test_topk_matches_oracle_large_ensemble(engine_factory, precision, C, mode, case):
    """Ordered, unseen, complete lists; each score within 1e-5 max|Q| of the oracle's; score_topk == score_pairs."""
    SS.test_topk_matches_oracle_at_shape(engine_factory, precision, C, mode, case)


@pytest.mark.parametrize("precision,C,mode",
                         [pytest.param(p, C, m, id=f"{p}-C{C}-{m}") for C in (5, 10) for m in ("q", "policy")
                          for p in SS.PRECISIONS])
def test_score_pairs_matches_oracle_large_ensemble(engine_factory, precision, C, mode):
    SS.test_score_pairs_matches_oracle(engine_factory, precision, C, mode)


@pytest.mark.parametrize("k", [1, 10, 33])
@pytest.mark.parametrize("precision", SS.PRECISIONS)
def test_user_row_alone_equals_among_many_large_ensemble(engine_factory, precision, k):
    C = 10
    _, users, items, seen = SS._invariance_inputs()
    indptr, flat_seen = SS._csr(users, seen)
    flat, _, _ = SS._state(C)
    eng = SS._engine(engine_factory, precision, C, flat)
    many = eng.score_topk(users, items, k, indptr, flat_seen)
    for r in (0, users.size // 2, users.size - 1):
        alone = eng.score_topk(users[r:r + 1], items, k, indptr, flat_seen)
        SS._same((many[0][r:r + 1], many[1][r:r + 1]), alone, f"row {r} alone vs among many")


# ---------------------------------------------------------------- 4. offline scorers at C = 10
@pytest.mark.parametrize("prep_on", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_offline_metrics_large_ensemble(engine_factory, precision, prep_on):
    """Every scorer, value_estimation_std included, against tests/offline_metrics_oracle.py under its gates."""
    OMT.test_small_tables_against_oracle(engine_factory, precision, 10, prep_on)


# ---------------------------------------------------------------- 5. model level
def test_exact_resume_and_predict_large_ensemble(tmp_path):
    """CQL(n_critics=10, n_action_samples=32): fit(N) -> save -> load -> resume(M) is bit-identical to fit(N + M), and
    predict agrees with predict_pairs."""
    from replay_cql_b200.model_handler import load, save
    from replay_cql_b200.models import CQL
    from replay_cql_b200.synthetic import make_log
    log = make_log("tiny")
    N, M = 17, 11
    kw = dict(top_k=3, batch_size=64, seed=5, n_epochs=1, save_replay_table=True, n_critics=10, n_action_samples=32)
    full = CQL(n_steps_per_epoch=N + M, **kw)
    full.fit(log)
    part = CQL(n_steps_per_epoch=N, **kw)
    part.fit(log)
    path = str(tmp_path / "ckpt")
    save(part, path)
    part.engine.close()
    resumed = load(path)
    assert resumed.n_critics == 10 and resumed.n_action_samples == 32
    assert resumed.engine.hp.n_critics == 10 and resumed.engine.hp.n_action_samples == 32
    resumed.resume(n_steps=M)
    assert np.array_equal(resumed.engine.get_state(), full.engine.get_state())
    m1, v1, s1 = resumed.engine.get_optimizer()
    m2, v2, s2 = full.engine.get_optimizer()
    assert s1 == s2 == N + M and np.array_equal(m1, m2) and np.array_equal(v1, v2)
    recs = full.predict(log, k=4, filter_seen_items=False)
    pd.testing.assert_frame_equal(resumed.predict(log, k=4, filter_seen_items=False), recs)
    pairs = full.predict_pairs(recs[["user_idx", "item_idx"]], log)
    merged = recs.merge(pairs, on=["user_idx", "item_idx"], suffixes=("_a", "_b"))
    assert len(merged) == len(recs) > 0
    scale = max(1.0, merged["relevance_a"].abs().max())
    assert (merged["relevance_a"] - merged["relevance_b"]).abs().max() <= SS.TOL * scale
    full.engine.close()
    resumed.engine.close()


# ---------------------------------------------------------------- 6. memory
def test_over_budget_configuration_is_rejected_before_allocating():
    """B = 2^20 with C = 10 and n = 32 needs about a terabyte: cql_create sizes its buffers first and returns code 3 with
    the requirement, without allocating; a normal handle created afterwards works."""
    torch.cuda.init()
    free0, _ = torch.cuda.mem_get_info(0)
    with pytest.raises(_lib.CqlArgumentError, match=r"need [0-9.]+ GiB of device memory"):
        CqlEngine(CqlHyperParams(batch_size=1 << 20, n_critics=10, n_action_samples=32), device=0)
    free1, _ = torch.cuda.mem_get_info(0)
    assert free1 >= free0 - (256 << 20), (free0, free1)       # (other processes may share the GPU)
    eng = CqlEngine(CqlHyperParams(batch_size=64, n_critics=10, n_action_samples=32), device=0)
    try:
        eng.synth_table(10_007, 100, 50, seed=3)
        m = eng.update(3)
        assert all(np.isfinite(v) for v in m.values()), m
    finally:
        eng.close()


# ---------------------------------------------------------------- 7. two GPUs, fused peer exchange
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_large_ensemble_match_oracle():
    """(C, n) = (10, 32), world size 2 with the fused peer exchange: both replicas bit-identical, and equal within the
    update gates to the float32 oracle whose gradients are averaged over the two ranks' batches."""
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", "tests/_large_ensemble_dp_check.py"],
                       cwd=ROOT, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True,
                       timeout=1200)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert p.stdout.count("dp-ok") == 2, p.stdout
