"""GPU: fitted Q evaluation (``cql_fqe_*``, ``replay_cql_b200.ope.FQE``; DESIGN.md section 1 "FQE").

* one update on caller rows (``cql_fqe_update_rows``) against the float32 oracle (tests/fqe_oracle.py): precision x
  critic count x batch size, plus terminal rows, n-step rows and the scalers; loss and updated critics at 1e-4 (float64-
  budget rule; WEIGHT_LOOSER lists the measured exceptions), Adam moments and gradients at the update tests' gates;
* the sampled path draws the rows ``cql_sample_rows`` returns for the same positions; per-step restarted oracle
  comparisons over updates that span target synchronisations;
* bits: the target is a copy of the critics after synchronising updates and unchanged otherwise, the actor slot never
  changes, ``fit(N); fit(M)`` equals ``fit(N + M)``, two runs and a side stream agree, and the CQL model is untouched;
* behaviour: constant reward on an all-terminal table, and two-step episodes rewarded at the terminal;
* ``offline_metrics`` and ``predict_value`` against the oracles on FQE's networks; the launch count per update.
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
from replay_cql_b200 import layout
from replay_cql_b200.engine import CqlEngine, CqlHyperParams, offline_scores
from replay_cql_b200.models import CQL
from replay_cql_b200.ope import FQE
from replay_cql_b200.synthetic import make_log
from tests import fqe_oracle as Q
from tests import helpers as Hp
from tests import offline_metrics_oracle as OM

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
GAMMA = 0.99
LR = 1e-4
PREP = {"scaler": {"type": "standard", "mean": [3.0, 1.8], "std": [1.7, 1.1]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
        "reward_scaler": {"type": "standard", "mean": [0.3], "std": [0.45]}}
# launches per FQE update (DESIGN.md section 5)
LAUNCHES = {"fp32": 10, "tf32x3": 13, "f16x3": 8}


# Updated-weight entries measured above 1e-4 of their tensor (first Adam step, from zero moments, lr 1e-4).  In every one
# the worst entry's float32-oracle gradient is 5e-12 .. 2e-8, 2e-10 .. 3e-7 of the tensor's largest, where the step
# lr * g / (|g| + 1e-8) is ill-conditioned: the GPU's gradient there differs from the oracle's by 2e-9 .. 7e-8 (inside
# the gradient gates, which are relative to the largest entry) and the entry moves by 6e-6 .. 3e-5 more or less than the
# oracle's.  tf32x3 C = 10, B = 100, critic 4 W2[62, 134]: g 1.5e-8 (oracle) / 8.1e-8 (GPU), step 8.9e-5 against 6.0e-5
# (float32 oracle) and 5.3e-5 (float64 oracle); the float32 oracle itself is 1.1e-4 from the float64 one on that tensor.
# key: the comparison's tag -> {(critic, tensor): gate}, each gate the measured error rounded up.
WEIGHT_LOOSER = {
    ("tf32x3", 10, 100, "plain"): {(4, "W2"): 6e-4},        # measured 4.7e-4 (float64 oracle: 5.8e-4)
    ("tf32x3", 10, 1024, "plain"): {(2, "W3"): 1.5e-4},     # 1.2e-4
    ("tf32x3", 10, 8192, "plain"): {(7, "W2"): 2e-4},       # 1.4e-4
    ("tf32x3", "sampled", 0): {(1, "W2"): 2e-4},            # 1.7e-4
    ("f16x3", 2, 1024, "plain"): {(1, "W2"): 1.5e-4},       # 1.0e-4
    ("f16x3", 10, 100, "plain"): {(4, "W2"): 5e-4},         # 3.8e-4 (float64 oracle: 4.9e-4)
}


def rows_of(B, seed, term_frac=0.1, nstep=False):
    """B table rows: ids scaled by 1e-3 (the policy is not saturated), ratings 1..5, 0/1 rewards, terminal rows with
    s' = (0, 0); n-step rows carry returns and discounts gamma^k."""
    rng = np.random.default_rng(seed)
    r = np.zeros((B, 8), np.float32)
    r[:, 0:2] = rng.integers(0, 6000, (B, 2)) * np.float32(1e-3)
    r[:, 2] = rng.integers(1, 6, B) + np.float32(1e-3) * rng.standard_normal(B).astype(np.float32)
    r[:, 3] = rng.integers(0, 2, B)
    r[:, 6] = rng.random(B) < term_frac
    r[:, 4:6] = np.where(r[:, 6:7] != 0, 0, rng.integers(0, 6000, (B, 2)) * np.float32(1e-3))
    if nstep:
        r[:, 3] = (rng.random(B) * 3).astype(np.float32)
        r[:, 7] = np.float32(GAMMA) ** rng.integers(1, 4, B)
    return r


@functools.lru_cache(maxsize=None)
def _flat(C):
    """FQE's critics (seed 12345) under a policy from another seed, targets equal to the critics."""
    flat = layout.init_state(C, 12345)
    flat[:layout.NET_STRIDE] = layout.init_state(1, 7)[:layout.NET_STRIDE]
    return flat


def _engine(precision, C, B, nstep=False, prep=False, interval=100, lr=LR):
    eng = CqlEngine(CqlHyperParams(batch_size=B, n_critics=C, n_action_samples=1, precision=precision, gamma=GAMMA,
                                   critic_lr=lr, n_steps=3 if nstep else 1))
    eng.set_state(_flat(C))
    if prep:
        eng.set_preprocessing(**PREP)
    eng.fqe_enable(interval)
    return eng


def _slots(flat, C):
    n = layout.NET_STRIDE
    return (flat[:n], flat[n:(1 + C) * n], flat[(2 + C) * n:(2 + 2 * C) * n])     # actor, critics, target critics


def _compare_update(eng, precision, C, rows, st_before, nstep, prep, interval, tag):
    """eng has just run one update on `rows` from oracle state st_before (float32): check it against the oracle."""
    st32 = Q.cast(st_before, torch.float32)
    loss_ref, g_ref = Q.update(st32, rows, GAMMA, LR, interval, nstep=nstep, prep=prep)

    @functools.lru_cache(maxsize=1)
    def f64():                                       # the float64 twin of the same update, computed only when needed
        s = Q.cast(st_before, torch.float64)
        Q.update(s, rows, GAMMA, LR, interval, nstep=nstep, prep=prep)
        return s
    # The moments hold this step's gradient, so in the tensor-core precisions they take the gradient's max-norm gate (the
    # ReLU-flip note in tests/helpers.py), as in tests/test_gpu_update_shapes.py; fp32 keeps 1e-4.  The updated weights
    # keep 1e-4 except the measured entries of WEIGHT_LOOSER.
    mom_tol = Hp.TOL if precision == "fp32" else Hp.GRAD_MAX_TOL[precision]
    looser = WEIGHT_LOOSER.get(tag, {})
    flat = eng.get_state()
    m, v, step = eng.get_optimizer()
    budgeted = []
    for c in range(C):
        got = layout.unpack_state(flat, C)["critics"][c]
        gm = layout.unpack_state(m, C)["critics"][c]
        gv = layout.unpack_state(v, C)["critics"][c]
        for k in Q.NET_KEYS:
            Hp.check_f64_budget((tag, "w", c, k), got[k], st32["critics"][c][k].numpy(),
                                lambda: f64()["critics"][c][k].numpy(), budgeted, tol=looser.get((c, k), Hp.TOL))
            Hp.check_f64_budget((tag, "m", c, k), gm[k], st32["adam"][c][k]["m"].numpy(),
                                lambda: f64()["adam"][c][k]["m"].numpy(), budgeted, tol=mom_tol)
            Hp.check_f64_budget((tag, "v", c, k), gv[k], st32["adam"][c][k]["v"].numpy(),
                                lambda: f64()["adam"][c][k]["v"].numpy(), budgeted, tol=mom_tol)
    return loss_ref, g_ref, step, st32


def _check_grads(g_gpu, g_ref, precision, B, tag):
    mx, l2 = [], []
    for c in range(len(g_ref)):
        for k in Q.NET_KEYS:
            mx.append(Hp.rel_err(g_gpu[c][k], g_ref[c][k].numpy()))
            l2.append(Hp.rel_err_l2(g_gpu[c][k], g_ref[c][k].numpy()))
    assert max(mx) <= Hp.GRAD_MAX_TOL[precision], (tag, max(mx))
    assert max(l2) <= Hp.GRAD_L2_TOL[precision], (tag, max(l2))
    if precision != "fp32":
        # B = 1: every gradient tensor is one row's outer product, so the median is the one row's forward error --
        # measured 2.6e-5 in tf32x3 (C = 1), inside every per-tensor gate
        assert float(np.median(l2)) <= (3e-5 if B == 1 else Hp.GRAD_MEDIAN_TOL), (tag, float(np.median(l2)))


def _one_update(precision, C, B, kind, seed=0):
    nstep, prep = kind in ("nstep", "nstep+prep"), kind in ("prep", "nstep+prep")
    rows = rows_of(B, seed, term_frac=0.5 if kind == "terminal" else 0.1, nstep=nstep)
    eng = _engine(precision, C, B, nstep=nstep, prep=prep)
    try:
        st0 = Q.from_flat(_flat(C), C)
        loss, g = eng.fqe_update_rows(rows, want_grads=True)
        tag = (precision, C, B, kind)
        loss_ref, g_ref, step, _ = _compare_update(eng, precision, C, rows, st0, nstep, PREP if prep else None, 100, tag)
        assert step == 1
        assert abs(loss - loss_ref) <= Hp.TOL * max(1.0, abs(loss_ref)), (tag, loss, loss_ref)
        _check_grads(g, g_ref, precision, B, tag)
        actor, critics, targ = _slots(eng.get_state(), C)
        assert np.array_equal(actor, _flat(C)[:layout.NET_STRIDE])          # the policy never changes
        assert np.array_equal(targ, critics)                                # update 1 synchronises the target
    finally:
        eng.close()


@pytest.mark.parametrize("B", [1, 37, 100, 1024, 8192])
@pytest.mark.parametrize("C", [1, 2, 10])
@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_one_update_against_oracle(precision, C, B):
    _one_update(precision, C, B, "plain")


@pytest.mark.parametrize("B", [37, 1024])
@pytest.mark.parametrize("kind", ["terminal", "nstep", "prep", "nstep+prep"])
@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_one_update_rows_kinds_against_oracle(precision, kind, B):
    _one_update(precision, 2, B, kind, seed=3)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_sampled_updates_restarted_oracle_and_target_bits(precision):
    """I = 2 over five sampled updates: each from the GPU's own state against the oracle on the rows cql_sample_rows
    returns for that step's positions; the target is a bit copy after updates 1, 3, 5 and bit-unchanged after 2, 4."""
    C, B, I = 2, 64, 2
    eng = _engine(precision, C, B, prep=True, interval=I)
    try:
        eng.set_table_rows(rows_of(3000, 9))
        prev_targ = None
        for k in range(5):
            flat = eng.get_state()
            m, v, step = eng.get_optimizer()
            assert step == k
            st = Q.from_flat(flat, C, m, v, step)
            rows = eng.sample_rows(B, pos=k * B).cpu().numpy()
            loss = eng.fqe_update(1)
            loss_ref, _, _, _ = _compare_update(eng, precision, C, rows, st, False, PREP, I, (precision, "sampled", k))
            assert abs(loss - loss_ref) <= Hp.TOL * max(1.0, abs(loss_ref)), (k, loss, loss_ref)
            actor, critics, targ = _slots(eng.get_state(), C)
            assert np.array_equal(actor, _flat(C)[:layout.NET_STRIDE])
            if k % I == 0:
                assert np.array_equal(targ, critics), k
            else:
                assert not np.array_equal(targ, critics) and np.array_equal(targ, prev_targ), k
            prev_targ = targ.copy()
        before = eng.launch_count
        eng.fqe_update(9)
        assert eng.launch_count - before == 9 * LAUNCHES[precision]
    finally:
        eng.close()


def test_runs_and_streams_give_the_same_bits():
    outs = []
    for stream in (None, None, "side"):
        eng = _engine("f16x3", 3, 256, interval=3)
        try:
            eng.set_table_rows(rows_of(20000, 4))
            side = torch.cuda.Stream() if stream else None
            loss = eng.fqe_update(11, stream=side.cuda_stream if side else None)
            if side:
                side.synchronize()
            outs.append((eng.get_state(), eng.get_optimizer(), loss))
        finally:
            eng.close()
    for s, (m, v, k), loss in outs[1:]:
        assert np.array_equal(s, outs[0][0]) and np.array_equal(m, outs[0][1][0]) and np.array_equal(v, outs[0][1][1])
        assert k == outs[0][1][2] == 11 and loss == outs[0][2]


def _model(**kw):
    m = CQL(top_k=3, batch_size=64, seed=11, n_steps_per_epoch=5, **kw)
    m.fit(make_log("tiny", seed=2))
    return m


def _learner(m):
    return m.engine.get_state(), m.engine.get_optimizer()


def test_fit_continues_exactly_and_leaves_the_model_alone():
    a, b = _model(scaler="min_max"), _model(scaler="min_max")
    f1 = FQE(a, n_critics=2, batch_size=32, target_update_interval=3)
    f1.fit(n_steps=5)
    f1.fit(n_steps=8)
    f2 = FQE(b, n_critics=2, batch_size=32, target_update_interval=3)
    f2.fit(n_steps=13)
    assert np.array_equal(f1.engine.get_state(), f2.engine.get_state())
    assert f1.last_loss == f2.last_loss
    _, _, k = f1.engine.get_optimizer()
    assert k == 13
    f1.offline_metrics()
    f1.predict_value([0, 1], [2, 3])
    f1.close()
    f2.close()
    a.resume(n_steps=7)                              # cql.fit -> FQE(cql).fit -> cql.resume == cql.fit -> cql.resume
    c = _model(scaler="min_max")
    c.resume(n_steps=7)
    (sa, (ma, va, ka)), (sc, (mc, vc, kc)) = _learner(a), _learner(c)
    assert np.array_equal(sa, sc) and np.array_equal(ma, mc) and np.array_equal(va, vc) and ka == kc
    assert a.last_metrics == c.last_metrics


def test_fqe_handle_refuses_cql_updates_and_needs_the_right_table():
    from replay_cql_b200 import _lib
    m = _model()
    f = FQE(m, batch_size=16)
    with pytest.raises(_lib.CqlArgumentError, match="FQE mode"):
        f.engine.update(1)
    with pytest.raises(_lib.CqlArgumentError, match="FQE mode"):
        f.engine.step_phase(0)
    f2 = FQE(m, n_steps=2)
    try:
        with pytest.raises(ValueError, match="n_steps"):
            f2.fit(n_steps=1)
    finally:
        f2.close()
    f.fit(make_log("tiny", seed=2), n_steps=3)        # its own table from the log, by the same builder
    assert f.engine.n_transitions == m.engine.n_transitions
    assert np.array_equal(f.engine.export_transitions(), m.engine.export_transitions())
    f.close()


def test_n_step_rows_are_discounted_with_fqe_gamma():
    """FQE(gamma=0.9, n_steps=3) of a model trained with gamma 0.99 and n_steps 3: the model's table, discounted with
    0.99, is refused without a log; a log is built into rows whose discounts are FQE's 0.9^k (the builder's float64
    product of the float32 gamma), with the same transitions, horizons k and one-step returns as the model's rows."""
    log = make_log("tiny", seed=2)
    m = _model(n_steps=3)
    f = FQE(m, gamma=0.9, n_steps=3, batch_size=16)
    try:
        with pytest.raises(ValueError, match="gamma"):
            f.fit(n_steps=1)
        f.fit(log, n_steps=1)
        rows, model_rows = f.engine.export_transitions(), m.engine.export_transitions()
        def discounts(gamma):                           # k = 1, 2, 3: g *= gamma in float64, then rounded to float32
            g, out = 1.0, []
            for _ in range(3):
                g = g * np.float64(np.float32(gamma))
                out.append(np.float32(g))
            return out
        mine, theirs = discounts(0.9), discounts(GAMMA)
        k_fqe = np.array([mine.index(x) if x in mine else -1 for x in rows[:, 7]])
        k_model = np.array([theirs.index(x) if x in theirs else -1 for x in model_rows[:, 7]])
        assert (k_fqe >= 0).all() and (k_fqe == 2).any(), np.unique(rows[:, 7])
        assert np.array_equal(k_fqe, k_model)
        assert np.array_equal(rows[:, [0, 1, 2, 4, 5, 6]], model_rows[:, [0, 1, 2, 4, 5, 6]])
        one = k_fqe == 0
        assert np.array_equal(rows[one, 3], model_rows[one, 3])
    finally:
        f.close()


BEHAVIOUR_GAMMA = 0.8


def _behaviour_table(kind, n=2000, seed=0):
    rng = np.random.default_rng(seed)
    r = np.zeros((n, 8), np.float32)
    r[:, 0:2] = rng.random((n, 2))
    r[:, 2] = rng.uniform(-1, 1, n)
    if kind == "const":                    # every row its own one-step episode, reward 0.5
        r[:, 3] = 0.5
        r[:, 6] = 1
    else:                                  # two-step episodes s0 -> s1, reward 1 at the terminal s1; s0 in [0, 0.5)^2 and
        r[0::2, 0:2] *= 0.5                # s1 in [0.5, 1)^2, so the critic can tell them apart
        r[1::2, 0:2] = 0.5 + 0.5 * r[1::2, 0:2]
        r[1::2, 3] = 1
        r[1::2, 6] = 1
        r[0::2, 4:6] = r[1::2, 0:2]
    return r


@pytest.mark.parametrize("kind,want,steps", [("const", 0.5, 3000), ("two_step", BEHAVIOUR_GAMMA, 4000)])
@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_value_converges(precision, kind, want, steps):
    """gamma 0.8, learning_rate 1e-3, batch 100, target_update_interval 50: initial_state_value_estimation within 0.03
    of the exact policy value after `steps` updates (two-step episodes: V(s0) = gamma, 0.2 from the undiscounted 1)."""
    m = _model()
    m.engine.set_table_rows(_behaviour_table(kind))
    f = FQE(m, gamma=BEHAVIOUR_GAMMA, learning_rate=1e-3, target_update_interval=50, precision=precision)
    f.fit(n_steps=steps)
    got = f.offline_metrics()["initial_state_value_estimation"]
    f.close()
    assert abs(got - want) <= 0.03, (precision, kind, got)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
def test_offline_metrics_and_predict_value_against_oracles(precision):
    m = _model(scaler="standard")
    f = FQE(m, n_critics=3, batch_size=64, target_update_interval=4, precision=precision, gamma=0.95)
    f.fit(n_steps=20)
    flat = f.engine.get_state()
    st = Hp.flat_to_oracle_state(flat, O.OracleConfig(n_critics=3))
    rows = f.engine.export_transitions()
    prep = f.engine.get_preprocessing()
    want = OM.evaluate(st, rows, 0.95, prep=prep, return_threshold=1.0)
    got = f.offline_metrics(return_threshold=1.0)
    w = offline_scores(want, True)
    from tests import scaler_oracle as S
    obs = S.obs_fwd(prep.get("scaler"), torch.from_numpy(rows[:, 0:2].copy()))
    with torch.no_grad():
        qmax = max(1.0, float(O.q_ensemble(st["critics"], obs, O.predict_action(st, obs)).abs().max()))
    scale = {"td_error": qmax * qmax, "continuous_action_diff": 36.0, "discounted_sum_of_advantage": qmax / (1 - 0.95)}
    for k, v in w.items():
        if np.isnan(v):
            assert np.isnan(got[k]), k
        else:
            assert abs(got[k] - v) <= 1e-5 * scale.get(k, qmax), (precision, k, got[k], v)
    users = np.array([0, 3, 7, 11, 19], np.int32)
    items = np.array([1, 2, 40, 5, 9], np.int32)
    pv = f.predict_value(users, items)
    x = S.obs_fwd(prep.get("scaler"), torch.from_numpy(np.stack([users, items], 1).astype(np.float32)))
    ref = O.relevance(st, x, "q").numpy()
    assert np.max(np.abs(pv - ref)) <= 1e-5 * max(1.0, float(np.max(np.abs(ref)))), (precision, pv, ref)
    f.close()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_give_identical_bits():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29543", "tests/_fqe_dp_check.py"],
                         cwd=ROOT, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    res = {int(l.split()[1]): json.loads(l.split(" result ", 1)[1]) for l in out.stdout.splitlines() if " result " in l}
    assert set(res) == {0, 1}
    assert res[0] == res[1]
