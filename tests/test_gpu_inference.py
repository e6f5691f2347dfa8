"""GPU: d3rlpy's per-observation inference (``predict_value`` with explicit actions and ``with_std``,
``predict_action``, ``sample_action``) against the CPU oracle and a host reference of the sampling noise.

Gates: the scorer gate of ``test_gpu_scoring.py`` (1e-5 * max(1, max|ref|)) for values, standard deviations and actions,
against the float32 and the float64 oracle.  bf16 runs and its error is printed, not gated.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import cql_oracle as O
from replay_cql_b200 import _lib, layout
from replay_cql_b200.models import CQL
from replay_cql_b200.ope import FQE
from replay_cql_b200.synthetic import make_log
from tests import helpers as Hp
from tests import sampling_oracle as SO
from tests import scaler_oracle as S

pytestmark = pytest.mark.gpu
TOL = 1e-5
CHUNK = 1 << 18                                      # INF_CHUNK: pairs per forward chunk (csrc/infer.cuh)
SAMPLE_SEED_XOR = 0xE7037ED1A0B428DB                 # cql_sample_action's Philox key: seed ^ this
PREP = {"scaler": {"type": "min_max", "minimum": [0.0, 0.0], "maximum": [6039.0, 3705.0]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]}}
FP_GRADE = ("fp32", "tf32x3", "f16x3")


def _gate(got, ref):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = float(np.max(np.abs(got - ref))) if ref.size else 0.0
    return err, TOL * max(1.0, float(np.max(np.abs(ref))) if ref.size else 1.0)


def _assert_gate(got, ref, tag):
    err, lim = _gate(got, ref)
    assert err <= lim, (tag, err, lim)


def _engine(engine_factory, precision, C, prep, seed=11, state_seed=None):
    eng = engine_factory(batch_size=64, n_critics=C, precision=precision, seed=seed)
    flat = layout.init_state(C, 31 if state_seed is None else state_seed)
    eng.set_state(flat)
    if prep:
        eng.set_preprocessing(**prep)
    return eng, flat


def _pairs(n, seed, n_users=6040, n_items=3706, lo=0):
    rng = np.random.default_rng(seed)
    u = rng.integers(lo, lo + n_users, n).astype(np.int32)
    i = rng.integers(lo, lo + n_items, n).astype(np.int32)
    a = rng.uniform(1.0, 5.0, n).astype(np.float32)          # ratings
    return u, i, a


def _obs(u, i, prep, dtype):
    """observations as the network sees them; ``prep``: explicit scaler parameters ({scaler, action_scaler}) or None"""
    obs = torch.from_numpy(np.stack([u, i], 1).astype(np.float32))
    if prep:
        obs = S.obs_fwd(prep["scaler"], obs)
    return obs.to(dtype)


def _ref_q(flat, C, u, i, actions, prep, dtype):
    """per-critic Q [C, n] of the oracle at the explicit (raw) actions or the greedy action"""
    st = Hp.flat_to_oracle_state(flat, O.OracleConfig(n_critics=C), dtype=dtype)
    obs = _obs(u, i, prep, dtype)
    if actions is None:
        a = O.predict_action(st, obs)
    else:
        a = torch.from_numpy(np.asarray(actions, dtype=np.float32))[:, None]
        a = (S.act_fwd(prep["action_scaler"], a) if prep else a).to(dtype)
    with torch.no_grad():
        return O.q_ensemble(st["critics"], obs, a).double().numpy()


def _ref_sample(flat, u, i, prep, seed, call, rows, dtype=torch.float64):
    """host reference of sample_action for the given rows of a call"""
    st = Hp.flat_to_oracle_state(flat, O.OracleConfig(n_critics=1), dtype=dtype)
    obs = _obs(u[rows], i[rows], prep, dtype)
    r = SO.philox4x32_10(int(seed) ^ SAMPLE_SEED_XOR, call, np.asarray(rows, dtype=np.int64))
    eps = torch.from_numpy(SO.box_muller(r[0], r[1])).to(dtype)[:, None]
    with torch.no_grad():
        mu, ls = O.actor_forward(st["actor"], obs)
        a, _ = O.policy_sample(mu, ls, eps)
    if prep:
        a = S.act_rev(prep["action_scaler"], a)
    return a[:, 0].double().numpy()


def _ref_greedy_action(flat, u, i, prep, dtype):
    st = Hp.flat_to_oracle_state(flat, O.OracleConfig(n_critics=1), dtype=dtype)
    a = O.predict_action(st, _obs(u, i, prep, dtype))
    if prep:
        a = S.act_rev(prep["action_scaler"], a)
    return a[:, 0].double().numpy()


PREPS = {"raw": None, "mm": PREP}
CASES = [pytest.param(p, C, kind, prep, id=f"{p}-C{C}-{kind}-{name}")
         for p in FP_GRADE for C in (1, 2, 10) for kind in ("explicit", "greedy") for name, prep in PREPS.items()]


@pytest.mark.parametrize("precision,C,kind,prep", CASES)
def test_predict_value_and_std_against_oracle(engine_factory, precision, C, kind, prep):
    eng, flat = _engine(engine_factory, precision, C, prep)
    u, i, a = _pairs(3001, seed=C * 10 + (prep is not None))
    acts = a if kind == "explicit" else None
    mean, std = eng.predict_value(u, i, acts, with_std=True)
    assert mean.dtype == np.float32 and std.dtype == np.float32 and mean.shape == std.shape == (u.size,)
    assert np.array_equal(eng.predict_value(u, i, acts), mean)           # the std costs nothing of the mean's bits
    for dtype in (torch.float32, torch.float64):
        q = _ref_q(flat, C, u, i, acts, prep, dtype)
        _assert_gate(mean, q.mean(axis=0), (dtype, "mean"))
        _assert_gate(std, q.std(axis=0), (dtype, "std"))
    if C == 1:
        assert not std.any()                                               # exactly 0.0
    else:
        assert (std > 0).mean() > 0.99


@pytest.mark.parametrize("kind", ["explicit", "greedy"])
def test_bf16_runs(engine_factory, kind):
    eng, flat = _engine(engine_factory, "bf16", 2, PREP)
    u, i, a = _pairs(2000, seed=5)
    acts = a if kind == "explicit" else None
    mean, std = eng.predict_value(u, i, acts, with_std=True)
    assert np.isfinite(mean).all() and np.isfinite(std).all()
    q = _ref_q(flat, 2, u, i, acts, PREP, torch.float64)
    print(f"bf16 {kind}: max |mean - oracle| = {_gate(mean, q.mean(0))[0]:.3g}, "
          f"max |std - oracle| = {_gate(std, q.std(0))[0]:.3g} (max |Q| {np.abs(q).max():.3g})")
    print(f"bf16 sample_action finite: {np.isfinite(eng.sample_action(u, i)).all()}")


@pytest.mark.parametrize("precision", FP_GRADE)
@pytest.mark.parametrize("prep", PREPS.values(), ids=PREPS.keys())
@pytest.mark.parametrize("C", [2, 10])
def test_greedy_calls_agree_with_the_pair_scorer(engine_factory, precision, prep, C):
    eng, flat = _engine(engine_factory, precision, C, prep)
    u, i, _ = _pairs(5000, seed=7)
    _assert_gate(eng.predict_value(u, i), eng.score_pairs(u, i, mode="q"), "q")
    pa = eng.predict_action(u, i)
    _assert_gate(pa, eng.score_pairs(u, i, mode="policy"), "policy")
    _assert_gate(pa, _ref_greedy_action(flat, u, i, prep, torch.float64), "policy oracle")


@pytest.mark.parametrize("precision", FP_GRADE)
@pytest.mark.parametrize("prep", PREPS.values(), ids=PREPS.keys())
def test_sample_action_against_host_reference(engine_factory, precision, prep):
    seed = 987654321
    eng, flat = _engine(engine_factory, precision, 2, prep, seed=seed)
    u, i, _ = _pairs(4000, seed=9)
    rows = np.arange(u.size)
    first = eng.sample_action(u, i)
    second = eng.sample_action(u, i)
    refs = [_ref_sample(flat, u, i, prep, seed, call, rows) for call in (0, 1)]
    for call, got in ((0, first), (1, second)):
        _assert_gate(got, refs[call], ("call", call))
        _assert_gate(got, _ref_sample(flat, u, i, prep, seed, call, rows, torch.float32), ("call f32", call))
    # consecutive calls draw new noise (the raw ids saturate tanh for most rows: there both draws give +-1)
    moved = np.abs(refs[0] - refs[1]) > 1e-4
    assert moved.mean() > (0.9 if prep else 0.0) and (first[moved] != second[moved]).all()
    eng.predict_action(u, i)                                                 # greedy: draws nothing, counts nothing
    _assert_gate(eng.sample_action(u, i), _ref_sample(flat, u, i, prep, seed, 2, rows), "call 2")
    fresh, _ = _engine(engine_factory, precision, 2, prep, seed=seed)
    assert np.array_equal(fresh.sample_action(u, i), first)                 # a fresh handle repeats the first call
    other, _ = _engine(engine_factory, precision, 2, prep, seed=seed + 1)
    other_ref = _ref_sample(flat, u, i, prep, seed + 1, 0, rows)
    _assert_gate(other.sample_action(u, i), other_ref, "seed + 1")           # the seed keys the stream


def _fitted(**kw):
    m = CQL(top_k=3, batch_size=64, seed=11, n_steps_per_epoch=5, n_critics=3, scaler="min_max",
            action_scaler="min_max", **kw)
    m.fit(make_log("tiny", seed=2))
    return m


def _learner(m):
    s = m.engine.get_state()
    mm, vv, k = m.engine.get_optimizer()
    return s, mm, vv, k


def test_inference_leaves_the_model_alone():
    """fit -> predict_value / predict_action / sample_action -> resume equals fit -> resume, bit for bit"""
    a, b = _fitted(), _fitted()
    before = _learner(a)
    table = a.engine.export_transitions()
    u, i, r = _pairs(1000, seed=3)
    a.predict_value(u, i, r, with_std=True)
    a.predict_value(u, i)
    a.predict_action(u, i)
    a.sample_action(u, i)
    a.sample_action(u, i)
    after = _learner(a)
    assert all(np.array_equal(x, y) for x, y in zip(before[:3], after[:3])) and before[3] == after[3]
    assert np.array_equal(a.engine.export_transitions(), table)
    a.resume(n_steps=7)
    b.resume(n_steps=7)
    (sa, ma, va, ka), (sb, mb, vb, kb) = _learner(a), _learner(b)
    assert np.array_equal(sa, sb) and np.array_equal(ma, mb) and np.array_equal(va, vb) and ka == kb == 12
    assert a.last_metrics == b.last_metrics


def test_public_calls_match_the_engine_and_the_oracle():
    m = _fitted()
    flat = m.engine.get_state()
    prep = m.engine.get_preprocessing()
    u, i, r = _pairs(777, seed=4, n_users=50, n_items=60)
    mean, std = m.predict_value(u, i, r[:, None], with_std=True)           # d3rlpy's [n, 1] action column
    st = Hp.flat_to_oracle_state(flat, O.OracleConfig(n_critics=3), dtype=torch.float64)
    obs = S.obs_fwd(prep["scaler"], torch.from_numpy(np.stack([u, i], 1).astype(np.float32))).double()
    act = S.act_fwd(prep["action_scaler"], torch.from_numpy(r)[:, None]).double()
    q = O.q_ensemble(st["critics"], obs, act).numpy()
    _assert_gate(mean, q.mean(0), "mean")
    _assert_gate(std, q.std(0), "std")
    assert np.array_equal(m.predict_action(u, i), m.engine.predict_action(u, i))
    pol = S.act_rev(prep["action_scaler"], O.predict_action(st, obs))[:, 0].numpy()
    _assert_gate(m.predict_action(u, i), pol, "predict_action")
    s = m.sample_action(u, i)
    assert s.shape == (u.size,) and np.isfinite(s).all()


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_fqe_predict_value(precision):
    m = _fitted()
    f = FQE(m, n_critics=3, batch_size=32, target_update_interval=3, precision=precision)
    try:
        f.fit(n_steps=6)
        flat, prep = f.engine.get_state(), m.engine.get_preprocessing()
        u, i, r = _pairs(1500, seed=6, n_users=50, n_items=60)
        two = f.predict_value(u, i)
        assert np.array_equal(two, f.engine.score_pairs(u, i, mode="q"))   # the two-argument call is unchanged
        mean, std = f.predict_value(u, i, with_std=True)
        _assert_gate(mean, two, "greedy vs pair scorer")
        q = _ref_q(flat, 3, u, i, None, prep, torch.float64)
        _assert_gate(mean, q.mean(0), "greedy mean")
        _assert_gate(std, q.std(0), "greedy std")
        me = f.predict_value(u, i, r)
        _assert_gate(me, _ref_q(flat, 3, u, i, r, prep, torch.float64).mean(0), "explicit mean")
        # the FQE handle's policy is the model's actor: the same greedy actions
        _assert_gate(f.engine.predict_action(u, i), m.predict_action(u, i), "policy")
    finally:
        f.close()


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
@pytest.mark.parametrize("n", [1, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK + 3])
def test_chunk_edges(engine_factory, precision, n):
    """rows on both sides of every chunk boundary (and the first and last rows) against the oracle"""
    eng, flat = _engine(engine_factory, precision, 2, PREP)
    u, i, a = _pairs(n, seed=n)
    mean, std = eng.predict_value(u, i, a, with_std=True)
    greedy = eng.predict_value(u, i)
    samp = eng.sample_action(u, i)
    edges = sorted({r for b in range(0, n + CHUNK, CHUNK) for r in range(b - 3, b + 3) if 0 <= r < n} | {n - 1})
    rows = np.asarray(edges)
    q = _ref_q(flat, 2, u[rows], i[rows], a[rows], PREP, torch.float64)
    _assert_gate(mean[rows], q.mean(0), "mean")
    _assert_gate(std[rows], q.std(0), "std")
    _assert_gate(greedy[rows], _ref_q(flat, 2, u[rows], i[rows], None, PREP, torch.float64).mean(0), "greedy")
    _assert_gate(samp[rows], _ref_sample(flat, u, i, PREP, 11, 0, rows), "sample")
    assert np.isfinite(mean).all() and np.isfinite(samp).all()


@pytest.mark.parametrize("precision", ["tf32x3", "f16x3"])
def test_stress_scale_ids(engine_factory, precision):
    """ids just below 2^24: hidden activations far outside the fp16 range; reference = the float64 oracle"""
    eng, flat = _engine(engine_factory, precision, 2, None)
    u, i, a = _pairs(3000, seed=8, n_users=4000, n_items=4000, lo=2 ** 24 - 4000)
    mean, std = eng.predict_value(u, i, a, with_std=True)
    q = _ref_q(flat, 2, u, i, a, None, torch.float64)
    _assert_gate(mean, q.mean(0), "mean")
    _assert_gate(std, q.std(0), "std")
    _assert_gate(eng.predict_value(u, i), _ref_q(flat, 2, u, i, None, None, torch.float64).mean(0), "greedy")
    _assert_gate(eng.sample_action(u, i), _ref_sample(flat, u, i, None, 11, 0, np.arange(u.size)), "sample")


def test_empty_inputs_and_rejections(engine_factory):
    eng, flat = _engine(engine_factory, "f16x3", 2, None)
    assert eng.predict_value([], []).shape == (0,)
    m0, s0 = eng.predict_value([], [], [], with_std=True)
    assert m0.shape == s0.shape == (0,)
    assert eng.predict_action([], []).shape == (0,) and eng.sample_action([], []).shape == (0,)
    u, i, a = _pairs(10, seed=1)
    bad_a = a.copy()
    bad_a[3] = np.nan
    for args in (([1, 2], [1]), ([1, 2 ** 24], [1, 2]), ([-1], [0]), ([0], [2 ** 24]), ([0.5], [1])):
        with pytest.raises(ValueError):
            eng.predict_value(*args)
        with pytest.raises(ValueError):
            eng.sample_action(*args)
    with pytest.raises(ValueError):
        eng.predict_value(u, i, bad_a)
    with pytest.raises(ValueError):
        eng.predict_value(u, i, a[:5])
    # the C ABI itself: return code 3, nothing computed, the sampling counter untouched
    lib, h = eng._lib, eng._h
    p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
    out, sd = np.zeros(10, np.float32), np.zeros(10, np.float32)
    big = u.copy()
    big[7] = 2 ** 24
    neg = i.copy()
    neg[0] = -5
    assert lib.cql_predict_value(h, p(u), p(i), None, -1, p(out), None, None) == 3
    assert lib.cql_predict_value(h, p(big), p(i), None, 10, p(out), p(sd), None) == 3
    assert lib.cql_predict_value(h, p(u), p(neg), p(a), 10, p(out), None, None) == 3
    assert lib.cql_predict_value(h, p(u), p(i), p(bad_a), 10, p(out), None, None) == 3
    assert lib.cql_predict_value(h, p(u), p(i), p(a), 10, None, None, None) == 3
    assert lib.cql_sample_action(h, p(u), p(i), -3, 0, p(out), None) == 3
    assert lib.cql_sample_action(h, p(big), p(i), 10, 0, p(out), None) == 3
    assert lib.cql_sample_action(h, p(u), p(neg), 10, 1, p(out), None) == 3
    assert lib.cql_sample_action(h, p(u), p(i), 10, 2, p(out), None) == 3
    assert not out.any() and not sd.any()
    assert lib.cql_predict_value(h, p(u), p(i), None, 0, None, None, None) == 0
    assert lib.cql_sample_action(h, None, None, 0, 0, None, None) == 0
    _assert_gate(eng.sample_action(u, i), _ref_sample(flat, u, i, None, 11, 0, np.arange(10)), "first draw")
