"""GPU: the update's inputs -- minibatch rows and Philox noise -- against the host reference (tests/sampling_oracle.py),
and the sampled update (``cql_update``, the product path) against the oracle.

The parity tests elsewhere feed the GPU host noise through ``update_batch(..., noise)``, so the device draws were only
ever compared with themselves.  Here ``CQL_BUF_BATCH`` / ``CQL_BUF_NOISE`` expose what an update consumed:

* rows: the gathered minibatch, bit for bit, equals the host rows at ``sampled_indices`` (scalers applied by
  ``scaler_oracle.transform_rows``) over batch sizes, action-sample counts, table sizes around the batch and
  data-parallel chunk, ranks of replicated and sharded tables, step counters past 2^32 and epoch boundaries;
  ``sample_rows`` against ``stream_index`` with chunk B;
* noise: the draws of ``k_step_head`` (``update``, the phase split) and ``k_noise`` (``update_batch`` and
  ``update_batches`` with Philox noise) against ``update_noise``: uniform blocks bit-exact, Gaussian blocks within
  GAUSS_ULPS float32 ulps of the float64 value (CUDA's documented bounds: ``logf`` 1 ulp, ``cospif`` 1 ulp, ``sqrtf``
  and the product correctly rounded; the tests print the largest distance seen);
* the read-back noise given back as provided noise takes the bit-identical step, so both paths read one layout;
* ``update(1)`` from the oracle's state (non-trivial Adam moments) against ``O.update`` on the host-indexed rows and the
  read-back noise, at the update tests' 1e-4 gates;
* the MDP builder's seeded action noise against ``mdp_action_noise`` on every row;
* ``cql_create`` refuses world_size > 256 (8 rank bits in the noise stream).
"""
import numpy as np
import pandas as pd
import pytest
import torch

from oracle import cql_oracle as O
from replay_cql_b200 import _lib, mdp
from replay_cql_b200.engine import CqlEngine, CqlHyperParams
from tests import helpers as Hp
from tests import sampling_oracle as S
from tests import scaler_oracle as SO

pytestmark = pytest.mark.gpu
GAUSS_ULPS = 4
BIG = 2 ** 33 + 3                      # a step counter past 2^32
PREP = {"scaler": {"type": "standard", "mean": [3000.5, 1850.25], "std": [1740.0, 1070.0]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
        "reward_scaler": {"type": "standard", "mean": [0.3], "std": [0.45]}}


@pytest.fixture
def make():
    """CqlEngine(hp, device 0, rank, world_size) without dp_attach: a local update on rank r's rows and Philox stream."""
    made = []

    def mk(B, n, W=1, r=0, seed=12345, C=2, precision="f16x3"):
        hp = CqlHyperParams(batch_size=B, n_critics=C, n_action_samples=n, seed=seed, precision=precision)
        made.append(CqlEngine(hp, device=0, rank=r, world_size=W))
        return made[-1]

    yield mk
    for e in made:
        e.close()


def _read(eng, which):
    torch.cuda.synchronize()
    return eng.grad_tensor(which).cpu().numpy().copy()


def _set_step(eng, step):
    m, v, _ = eng.get_optimizer()
    eng.set_optimizer(m, v, step)


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _index_rows(N):
    """Rows that encode their index exactly: obs = (i mod 2^16, i div 2^16), distinct act / rew, s' = row i + 1's obs."""
    i = np.arange(N, dtype=np.int64)
    rows = np.zeros((N, 8), np.float32)
    rows[:, 0], rows[:, 1] = i % 65536, i // 65536
    rows[:, 2] = 1.0 + (i % 4093) / 1024.0
    rows[:, 3] = (i % 3) * 0.5
    rows[:, 4], rows[:, 5] = (i + 1) % 65536, (i + 1) // 65536
    rows[:, 6] = (i % 11 == 10)
    return rows


def _batch_rows(B, N, seed, scale):
    b = Hp.batch_to_numpy(Hp.make_batch(N, seed=seed, scale=scale))
    return np.ascontiguousarray(np.concatenate([b["obs"], b["act"], b["rew"], b["next_obs"], b["term"],
                                                np.zeros((N, 1), np.float32)], 1))


# ---------------------------------------------------------------- minibatch rows
def _table_size(kind, B, W):
    return {"1": 1, "B-1": B - 1, "B": B, "BW-1": B * W - 1, "BW": B * W, "2BW+17": 2 * B * W + 17,
            "2^24+5": 2 ** 24 + 5}[kind]


# (B, n, table size, W, r, sharded, start step): every value of every axis appears
ROW_CELLS = [
    (1, 1, "1", 1, 0, False, 0),
    (1, 32, "BW", 8, 0, True, BIG),
    (37, 7, "B-1", 2, 1, False, 1),
    (37, 7, "BW-1", 8, 7, True, BIG),
    (37, 1, "2BW+17", 8, 7, False, 1),
    (300, 32, "B", 8, 0, False, BIG),
    (300, 7, "2BW+17", 2, 1, True, 0),
    (300, 1, "BW-1", 2, 1, False, 0),
    (4737, 1, "2^24+5", 8, 7, False, BIG),
    (4737, 32, "BW", 1, 0, True, 1),
    (4737, 7, "2BW+17", 2, 1, False, 2),
]


@pytest.mark.parametrize("B,n,N,W,r,sharded,start", ROW_CELLS,
                         ids=[f"B{c[0]}-n{c[1]}-N{c[2]}-W{c[3]}r{c[4]}-{'shard' if c[5] else 'repl'}-s{c[6]}"
                              for c in ROW_CELLS])
def test_sampled_rows_are_the_stream_rows(make, B, n, N, W, r, sharded, start):
    """Three consecutive update(1): each gathered minibatch is the host table's rows at sampled_indices(step)."""
    N = _table_size(N, B, W)
    seed = 9
    rows = _index_rows(N)
    eng = make(B, n, W, r, seed=seed)
    eng.set_table_rows(rows)
    eng.set_table_sharded(sharded)
    _set_step(eng, start)
    chunk = B if sharded else B * W
    n_eff = N - N % chunk or N
    epochs = set()
    for k in range(3):
        eng.update(1, want_metrics=False)
        got = _read(eng, _lib.BUF_BATCH).reshape(B, 8)
        idx = S.sampled_indices(start + k, B, r, W, sharded, N, seed)
        assert _same_bits(got, rows[idx]), (k, int(np.sum(np.any(got != rows[idx], axis=1))))
        p0 = (start + k) * B if sharded else ((start + k) * W + r) * B
        epochs |= {p0 // n_eff, (p0 + B - 1) // n_eff}
    assert eng.get_optimizer()[2] == start + 3
    print(f"\n[rows B={B} N={N} W={W} r={r} sharded={sharded} start={start}] epochs touched: {len(epochs)}")


def test_sampled_rows_with_scalers(make):
    """With scalers on, the minibatch the update trained on is transform_rows of the stream rows."""
    B, n, W, r, seed = 37, 7, 2, 1, 9
    N = 2 * B * W + 17
    rows = _batch_rows(B, N, seed=4, scale=1.0)
    eng = make(B, n, W, r, seed=seed)
    eng.set_table_rows(rows)
    prep = eng.set_preprocessing(**PREP)
    _set_step(eng, 1)
    for k in range(3):
        eng.update(1, want_metrics=False)
        idx = S.sampled_indices(1 + k, B, r, W, False, N, seed)
        assert _same_bits(_read(eng, _lib.BUF_BATCH).reshape(B, 8), SO.transform_rows(prep, rows[idx])), k


@pytest.mark.parametrize("B,N", [(37, 100), (37, 7), (1, 5), (300, 2 * 300 + 17)])
def test_sample_rows_follow_the_stream(make, B, N):
    """cql_sample_rows: positions pos + j of the stream with chunk B (across epoch boundaries, and far out), and
    explicit indices."""
    seed = 2 ** 40 + 3
    rows = _index_rows(N)
    eng = make(B, 1, seed=seed)
    eng.set_table_rows(rows)
    for pos, count in ((0, 3 * N + 1), (N // 2, 2 * N + 3), (2 ** 40 + 7, N + 5)):
        got = eng.sample_rows(count, pos=pos).cpu().numpy()
        idx = S.stream_index(pos + np.arange(count), N, B, seed)
        assert _same_bits(got, rows[idx]), pos
    idx = np.random.default_rng(N).integers(0, N, 999)
    assert _same_bits(eng.sample_rows(idx.size, idx=idx).cpu().numpy(), rows[idx])


# ---------------------------------------------------------------- noise
_ULPS = []


def _check_noise(got, seed, done, rank, B, n, tag):
    ref = S.update_noise_packed(seed, done, rank, B, n)
    assert got.shape == ref.shape, tag
    uni = S.uniform_mask(B, n)
    assert _same_bits(got[uni], ref[uni].astype(np.float32)), (tag, "uniform", int(np.sum(got[uni] != ref[uni])))
    g, rg = got[~uni].astype(np.float64), ref[~uni]
    ulps = np.abs(g - rg) / np.spacing(np.abs(rg).astype(np.float32)).astype(np.float64)
    worst = float(ulps.max())
    _ULPS.append(worst)
    assert worst <= GAUSS_ULPS, (tag, "gaussian", worst, int(np.argmax(ulps)))
    return worst


# (seed, W, r, B, n, start)
NOISE_CELLS = [
    (0, 1, 0, 37, 7, 0),
    (9, 2, 1, 300, 10, 1),
    (2 ** 40 + 3, 8, 7, 37, 7, BIG),
    (9, 8, 0, 1, 1, 5),
    (0, 8, 7, 4737, 3, BIG),
    (2 ** 40 + 3, 1, 0, 300, 32, 1),
    (9, 8, 7, 37, 1, 0),
    (0, 2, 1, 1, 32, BIG),
]


@pytest.mark.parametrize("seed,W,r,B,n,start", NOISE_CELLS,
                         ids=[f"seed{c[0]}-W{c[1]}r{c[2]}-B{c[3]}-n{c[4]}-s{c[5]}" for c in NOISE_CELLS])
def test_update_noise_matches_reference(make, seed, W, r, B, n, start):
    """One engine through the four Philox paths, each with its own step counter: update(1) and the phase split
    (k_step_head), update_batch without noise and the last step of update_batches (k_noise)."""
    eng = make(B, n, W, r, seed=seed)
    eng.set_table_rows(_batch_rows(B, 2 * B + 17, seed=3, scale=1e-3))
    _set_step(eng, start)
    worst = []
    eng.update(1, want_metrics=False)
    worst.append(_check_noise(_read(eng, _lib.BUF_NOISE), seed, start, r, B, n, "update"))
    eng.update_data_parallel(lambda buf: None)
    worst.append(_check_noise(_read(eng, _lib.BUF_NOISE), seed, start + 1, r, B, n, "phase split"))
    batches = [Hp.batch_to_numpy(Hp.make_batch(B, seed=50 + i, scale=1e-3)) for i in range(3)]
    eng.update_batch(batches[0])
    worst.append(_check_noise(_read(eng, _lib.BUF_NOISE), seed, start + 2, r, B, n, "update_batch"))
    eng.update_batches(batches[1:])
    worst.append(_check_noise(_read(eng, _lib.BUF_NOISE), seed, start + 4, r, B, n, "update_batches"))
    assert eng.get_optimizer()[2] == start + 5
    print(f"\n[noise seed={seed} W={W} r={r} B={B} n={n}] largest Gaussian distance (float32 ulps) per path "
          f"{worst}; over the file so far {max(_ULPS)}")


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_read_back_noise_as_provided_noise_takes_the_same_step(make, precision):
    B, C, n = 37, 3, 7
    a, b = make(B, n, 8, 7, seed=9, C=C, precision=precision), make(B, n, 8, 7, seed=9, C=C, precision=precision)
    batch = Hp.batch_to_numpy(Hp.make_batch(B, seed=21, scale=1e-3))
    for e in (a, b):
        _set_step(e, 4)
    ma, _ = a.update_batch(batch)
    flat = _read(a, _lib.BUF_NOISE)
    mb, _ = b.update_batch(batch, noise=S.unpack_noise(flat, B, n))
    assert _same_bits(_read(b, _lib.BUF_NOISE), flat)
    assert ma == mb
    assert _same_bits(a.get_state(), b.get_state())
    for x, y in zip(a.get_optimizer(), b.get_optimizer()):
        assert np.array_equal(x, y)


# ---------------------------------------------------------------- the sampled update against the oracle
def _scalar_err(a, b):
    return abs(float(a) - float(b)) / max(1.0, abs(float(b)))


def _as64(d):
    return {k: v.double() for k, v in d.items()}


ORACLE_CASES = [
    ((37, 3, 7), "fp32", 1, 0, False),
    ((37, 3, 7), "f16x3", 1, 0, False),
    ((300, 4, 10), "fp32", 1, 0, False),
    ((300, 4, 10), "f16x3", 1, 0, False),
    ((37, 3, 7), "f16x3", 8, 7, False),
    ((37, 3, 7), "f16x3", 1, 0, True),
]


@pytest.mark.parametrize("case,precision,W,r,scaled", ORACLE_CASES,
                         ids=[f"B{c[0][0]}-C{c[0][1]}-n{c[0][2]}-{c[1]}-W{c[2]}r{c[3]}{'-scaled' if c[4] else ''}"
                              for c in ORACLE_CASES])
def test_sampled_update_matches_oracle(make, case, precision, W, r, scaled):
    """update(1) -- on-device gather and Philox noise in one graph -- from the oracle's state with non-trivial Adam
    moments equals O.update on the rows at sampled_indices and the noise the update drew: the six metrics and every
    updated tensor within 1e-4 (the float64 budget rule of the update tests)."""
    B, C, n = case
    seed = 9
    cfg = O.OracleConfig(n_critics=C, n_action_samples=n)
    st = O.init_state(cfg, seed=7)
    O.update(cfg, st, Hp.make_batch(64, seed=17, scale=1e-3), O.make_noise(64, n, seed=18))   # Adam warm-up
    st0 = O.cast_state(st, torch.float32)
    N = 2 * B * W + 17
    rows = _batch_rows(B, N, seed=1000 + B, scale=1.0 if scaled else 1e-3)
    eng = make(B, n, W, r, seed=seed, C=C, precision=precision)
    eng.set_table_rows(rows)
    prep = eng.set_preprocessing(**PREP) if scaled else None
    eng.set_state(Hp.oracle_state_to_flat(st0))
    eng.set_optimizer(*Hp.oracle_adam_to_flat(st0))
    done = int(st0["step"])
    mg = eng.update(1)
    want = rows[S.sampled_indices(done, B, r, W, False, N, seed)]
    if scaled:
        want = SO.transform_rows(prep, want)
    assert _same_bits(_read(eng, _lib.BUF_BATCH).reshape(B, 8), want)
    flat_noise = _read(eng, _lib.BUF_NOISE)
    _check_noise(flat_noise, seed, done, r, B, n, "oracle case")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    batch = {"obs": t(want[:, 0:2]), "act": t(want[:, 2:3]), "rew": t(want[:, 3:4]), "next_obs": t(want[:, 4:6]),
             "term": t(want[:, 6:7])}
    noise = {k: t(v) for k, v in S.unpack_noise(flat_noise, B, n).items()}
    m32, _ = O.update(cfg, st, batch, noise)
    flat32 = Hp.oracle_state_to_flat(st)
    r64 = {}

    def ref64():
        if not r64:
            s64 = O.cast_state(st0, torch.float64)
            r64["m"], _ = O.update(cfg, s64, _as64(batch), _as64(noise))
            r64["flat"] = Hp.oracle_state_to_flat(O.cast_state(s64, torch.float32))
        return r64

    budgeted = []
    for name in Hp.METRIC_NAMES:
        Hp.check_f64_budget((name,), mg[name], m32[name], lambda name=name: ref64()["m"][name], budgeted, err=_scalar_err)
    g_t, r32 = Hp.state_tensors(eng.get_state(), C), Hp.state_tensors(flat32, C)
    for k in r32:
        Hp.check_f64_budget(("state",) + k, g_t[k], r32[k], lambda k=k: Hp.state_tensors(ref64()["flat"], C)[k], budgeted)
    assert eng.get_optimizer()[2] == done + 1
    print(f"\n[sampled update {case} {precision} W={W} r={r} scaled={scaled}] float64-budgeted comparisons: {budgeted}")


# ---------------------------------------------------------------- MDP builder action noise
def _mdp_log(n, seed=0):
    rng = np.random.default_rng(seed)
    return pd.DataFrame({"user_idx": rng.integers(0, max(2, n // 40), n), "item_idx": rng.integers(0, 5000, n),
                         "timestamp": rng.integers(0, n // 4 + 2, n),
                         "relevance": rng.integers(1, 6, n).astype(np.float64) + rng.random(n)})


@pytest.mark.parametrize("scale", [1e-3, 1.0])
def test_mdp_seeded_action_noise_matches_reference(make, scale):
    """Every row's action from the one-call builder and from chunked ingestion against (float)((double)(float)rel +
    mdp_action_noise): within 1 float32 ulp of the action at the default scale 1e-3; at scale 1 the noise's own error
    (GAUSS_ULPS of the noise) is added to that."""
    n, seed = 200_003, 3
    log = _mdp_log(n)
    eng = make(64, 1, seed=seed)
    rel = log["relevance"].to_numpy()
    want = S.mdp_actions(seed, rel, scale)
    nz = S.mdp_action_noise(seed, np.arange(n), scale)
    gate = np.spacing(np.abs(want)) + GAUSS_ULPS * np.spacing(np.abs(nz).astype(np.float32)) * (scale != 1e-3)
    for entry in ("one_call", "chunked"):
        if entry == "one_call":
            outs = eng.build_mdp_on_device(log["user_idx"].to_numpy(), log["item_idx"].to_numpy(), log["timestamp"],
                                           rel, top_k=10, action_randomization_scale=scale, action_noise=None,
                                           want_outputs=True)
        else:
            outs = mdp.ingest_log(eng, log, top_k=10, action_randomization_scale=scale, action_noise=None,
                                  want_outputs=True)
        act, order = outs[1], outs[4]
        w = want[order]
        err = np.abs(act.astype(np.float64) - w.astype(np.float64))
        bad = err > gate[order]
        assert not bad.any(), (entry, int(bad.sum()), float(err.max()))
        print(f"\n[mdp noise scale={scale} {entry}] bit-exact rows {int(np.sum(act == w))} of {n}; "
              f"largest error / gate {float(np.max(err / gate[order])):.2f}")


# ---------------------------------------------------------------- world size
def test_world_size_above_256_is_rejected():
    """The noise stream holds 8 rank bits: rank 256 would draw rank 0's noise.  257 ranks are refused with code 3 and a
    message; 256 ranks (the last one 255) are accepted."""
    hp = CqlHyperParams(batch_size=8, n_critics=1, n_action_samples=1)
    for rank in (0, 256):
        with pytest.raises(_lib.CqlArgumentError, match="world_size must be <= 256"):
            CqlEngine(hp, device=0, rank=rank, world_size=257)
    e = CqlEngine(hp, device=0, rank=255, world_size=256)
    e.close()
