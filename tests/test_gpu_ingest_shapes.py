"""GPU: the log ingestion path against the oracle at every size, column type and chunking the API accepts.

Covers the one-call builder (``cql_build_mdp``), chunked ingestion (``cql_mdp_begin`` / ``cql_mdp_append`` /
``cql_mdp_finish``) and the seen-items CSR (``cql_seen_csr``).  Every builder output is compared bit for bit: the
episode-ordered (obs, act, rew, term, order), the replay table itself, and the table statistics, which must equal
the bits ``cql_load_transitions`` gives for the reference arrays ("same bits from every producer", cql_b200.h).

References: the loop oracle (``oracle/mdp_oracle.py``) where it is affordable (few users, up to 65 537 rows), else
the vectorised host builder ``mdp.build_mdp``, which tests/test_mdp.py and the small cases here pin to the oracle.
The seen CSR is checked against a dict of sorted sets written below.
"""
import numpy as np
import pandas as pd
import pyarrow as pa
import pytest

from oracle import mdp_oracle
from replay_cql_b200 import mdp

pytestmark = pytest.mark.gpu

I64_MIN, I64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max
SLOT_VALUES_8B = (16 << 20) // 8          # MdpSession::SLOT_BYTES / 8: int64 / float64 values per pinned-ring slot
ORACLE_MAX_ROWS, ORACLE_MAX_USERS = 65_537, 5_000
LARGE_N = 9_000_001                       # 8-byte columns: five ring slots (the 4-slot ring wraps); 4-byte: three


# ----------------------------------------------------------------------------- fixtures and helpers
@pytest.fixture(scope="module")
def eng(engine_factory):
    return engine_factory(batch_size=64)


@pytest.fixture(scope="module")
def ref_eng(engine_factory):
    """Loads the reference arrays through cql_load_transitions: its table_stats are the bits every producer must give."""
    return engine_factory(batch_size=64)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(-1), a.shape, a.dtype


def _same_bits(a, b):
    (x, sa, da), (y, sb, db) = _bits(a), _bits(b)
    return sa == sb and da == db and np.array_equal(x, y)


def _reference(log: pd.DataFrame, top_k: int, noise) -> mdp.MdpArrays:
    """Host builder's arrays; pinned to the loop oracle wherever the oracle is affordable."""
    ref = mdp.build_mdp(log, top_k=top_k, action_noise=noise)
    if len(log) <= ORACLE_MAX_ROWS and log["user_idx"].nunique() <= ORACLE_MAX_USERS:
        want = mdp_oracle.build_mdp(log, top_k=top_k, action_noise=noise)
        got = mdp.to_transitions(ref)
        for k in want:
            assert _same_bits(got[k], want[k]), f"host builder != oracle in {k}"
    return ref


def _table_rows(ref: mdp.MdpArrays) -> np.ndarray:
    tr = mdp.to_transitions(ref)
    n = len(ref)
    return np.concatenate([tr["obs"], tr["act"], tr["rew"], tr["next_obs"], tr["term"], np.zeros((n, 1), np.float32)], 1)


def _check_build(eng, ref_eng, outs, ref: mdp.MdpArrays, table=True):
    obs, act, rew, term, order = outs
    n = len(ref)
    assert eng.n_transitions == n
    for name, got, want in (("obs", obs, ref.obs), ("act", act, ref.act), ("rew", rew, ref.rew), ("term", term, ref.term)):
        assert _same_bits(got, want), f"{name}: {int((got != want).sum())} of {want.size} values differ"
    assert np.array_equal(order, ref.order)
    if table:
        rows = eng.export_transitions()
        assert _same_bits(rows, _table_rows(ref))
        idx = np.unique(np.r_[0, n - 1, np.linspace(0, n - 1, 17).astype(np.int64)])
        assert _same_bits(eng.sample_rows(idx.size, idx=idx).cpu().numpy(), rows[idx])
    ref_eng.load_transitions(ref.obs, ref.act, ref.rew, ref.term)
    got_st, want_st = eng.table_stats(), ref_eng.table_stats()
    for k in want_st:
        assert _same_bits(np.asarray(got_st[k]), np.asarray(want_st[k])), f"table_stats {k}"


def _one_call(eng, log, top_k, noise, scale=1e-3):
    return eng.build_mdp_on_device(log["user_idx"].to_numpy(), log["item_idx"].to_numpy(), log["timestamp"],
                                   log["relevance"].to_numpy(), top_k=top_k, action_randomization_scale=scale,
                                   action_noise=noise, want_outputs=True)


def _chunked(eng, src, top_k, noise, scale=1e-3):
    return mdp.ingest_log(eng, src, top_k=top_k, action_randomization_scale=scale, action_noise=noise, want_outputs=True)


def _arrow(log: pd.DataFrame, cuts=None, n_chunks=3) -> pa.Table:
    """``log`` as a pyarrow Table cut into chunks at ``cuts`` (row positions), the same cuts for every column."""
    t = pa.Table.from_pandas(log, preserve_index=False)
    if cuts is None:
        cuts = np.linspace(0, t.num_rows, n_chunks + 1).astype(int)
    cuts = np.unique(np.r_[0, np.asarray(cuts, dtype=np.int64), t.num_rows])
    return pa.concat_tables([t.slice(a, b - a) for a, b in zip(cuts[:-1], cuts[1:])])


def _users(rng, n, episodes):
    if episodes == "one_row_each":
        return rng.permutation(n).astype(np.int64)
    if episodes == "one_user":
        return np.full(n, 7, dtype=np.int64)
    if episodes == "zipf":
        return (rng.zipf(1.4, n) - 1) % max(1, n // 6 + 1)
    ids = rng.choice(2 ** 24, size=max(2, n // 5), replace=False)        # sparse ids up to 2**24 - 1
    ids[:2] = (0, 2 ** 24 - 1)
    return ids[rng.integers(0, ids.size, n)]


def _log(n, episodes="zipf", seed=0):
    rng = np.random.default_rng(seed)
    items = rng.integers(0, 2 ** 24, n) if episodes == "sparse" else rng.integers(0, 5000, n)
    if episodes == "sparse" and n >= 2:
        items[:2] = (0, 2 ** 24 - 1)
    return pd.DataFrame({"user_idx": _users(rng, n, episodes), "item_idx": items,
                         "timestamp": rng.integers(0, max(2, n // 4), n),           # ties
                         "relevance": rng.integers(1, 6, n).astype(np.float64)})


def _noise(n, seed=1):
    return np.random.default_rng(seed).standard_normal(n) * 1e-3


# ----------------------------------------------------------------------------- sizes x episodes x entry point
_REF_CACHE = {}


@pytest.mark.parametrize("entry", ["one_call", "chunked_arrow"])
@pytest.mark.parametrize("episodes", ["one_row_each", "one_user", "zipf", "sparse"])
@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 4097, 65_537, 1_048_579])
def test_sizes_and_episodes(eng, ref_eng, n, episodes, entry):
    key = (n, episodes)
    if key not in _REF_CACHE:
        _REF_CACHE.clear()
        log = _log(n, episodes, seed=n)
        _REF_CACHE[key] = (log, _noise(n), _reference(log, 3, _noise(n)))
    log, noise, ref = _REF_CACHE[key]
    if entry == "one_call":
        outs = _one_call(eng, log, 3, noise)
    else:
        outs = _chunked(eng, _arrow(log, n_chunks=min(n, 5)), 3, noise)
    _check_build(eng, ref_eng, outs, ref)


# ----------------------------------------------------------------------------- timestamp and relevance types
def _ts_column(kind, rng, n):
    """-> (pandas column or None, arrow array or None): None means 'derive from the other'."""
    small = rng.integers(0, 12, n)                                   # heavy ties
    if kind == "int64_ties":
        return small.astype(np.int64), None
    if kind == "int64_extreme":
        pool = np.array([I64_MIN, I64_MIN + 1, I64_MIN + 2, -(2 ** 62), -7, -1, 0, 1, 2 ** 62, I64_MAX - 1, I64_MAX], np.int64)
        return pool[rng.integers(0, pool.size, n)], None
    if kind == "int32":
        return (small - 6).astype(np.int32) * 100_000_000, None
    if kind == "datetime64_pre1970":
        return pd.Series(pd.to_datetime((small - 9) * 86_400_000_123, unit="ms")), None
    if kind.startswith("float"):
        x = (rng.integers(-20, 20, n) * 0.25).astype(np.float32 if kind.startswith("float32") else np.float64)
        x[::11] = -0.0
        return x, None
    if kind == "date32":
        return None, pa.array((small - 6).astype(np.int32) * 4000, type=pa.int32()).cast(pa.date32())
    unit, tz = kind.split("_")[1], ("Europe/Berlin" if kind.endswith("_tz") else None)
    step = {"s": 1, "ms": 10 ** 3, "us": 10 ** 6, "ns": 10 ** 9}[unit]
    vals = (small - 6).astype(np.int64) * 7_777_777 * step           # both sides of 1970
    return None, pa.array(vals, type=pa.int64()).cast(pa.timestamp(unit, tz=tz))


TS_KINDS = ["int64_ties", "int64_extreme", "int32", "datetime64_pre1970", "float64", "float32", "date32",
            "arrow_s", "arrow_ms", "arrow_us", "arrow_ns", "arrow_s_tz", "arrow_ns_tz"]


@pytest.mark.parametrize("kind", TS_KINDS)
def test_timestamp_types(eng, ref_eng, kind):
    """Every timestamp type through the one-call form, chunked Arrow (uneven chunks) and chunked pandas.  Float
    timestamps with fractional ties and negative values failed here: the Arrow path truncated them on the device."""
    n = 4097
    rng = np.random.default_rng(11)
    base = _log(n, "zipf", seed=3)
    base["user_idx"] %= 40
    pdcol, arcol = _ts_column(kind, rng, n)
    if arcol is not None:
        table = _arrow(base.drop(columns="timestamp"), cuts=[1, 700, 701, 3000])
        table = table.append_column("timestamp", pa.chunked_array([arcol.slice(0, 1), arcol.slice(1, 2000), arcol.slice(2001)]))
        log = table.to_pandas()
    else:
        log = base.assign(timestamp=pdcol)
        table = _arrow(log, cuts=[1, 700, 701, 3000])
    noise = _noise(n, seed=5)
    for top_k in (1, 3):
        ref = _reference(log, top_k, noise)
        _check_build(eng, ref_eng, _one_call(eng, log, top_k, noise), ref)
        _check_build(eng, ref_eng, _chunked(eng, table, top_k, noise), ref)
        _check_build(eng, ref_eng, _chunked(eng, log, top_k, noise), ref, table=False)


def test_float_timestamp_arrow_equals_pandas_path(eng):
    """The same float-timestamp log through Arrow and pandas chunks builds the same table (it did not: the Arrow
    chunks were truncated to integers on the device, -0.5 == 0.5 and 0.5 == 0.9)."""
    log = pd.DataFrame({"user_idx": [0, 0, 0, 0, 1, 1, 1], "item_idx": [1, 2, 3, 4, 5, 6, 7],
                        "timestamp": [0.9, 0.5, -0.5, 0.5, 0.25, -0.25, 0.0], "relevance": [1.0, 1.0, 1.0, 2.0, 3.0, 3.0, 3.0]})
    noise = np.zeros(len(log))
    ref = _reference(log, 1, noise)
    a = _chunked(eng, pa.Table.from_pandas(log, preserve_index=False), 1, noise)
    b = _chunked(eng, log, 1, noise)
    for x, y, z in zip(a, b, (ref.obs, ref.act, ref.rew, ref.term, ref.order)):
        assert np.array_equal(x, z) and np.array_equal(y, z)


def test_nan_timestamp_rejected(eng):
    log = pd.DataFrame({"user_idx": [0, 0], "item_idx": [1, 2], "timestamp": [0.5, np.nan], "relevance": [1.0, 2.0]})
    table = pa.table({c: pa.array(log[c].to_numpy()) for c in log.columns})       # NaN stays NaN, not a null
    for src in (log, table):
        with pytest.raises(ValueError, match="NaN"):
            mdp.ingest_log(eng, src, top_k=1)
    with pytest.raises(ValueError, match="NaN"):
        _one_call(eng, log, 1, None)


REL_KINDS = ["int64_1to5", "int32_1to5", "fractional", "negative", "signed_zero", "float32"]


@pytest.mark.parametrize("kind", REL_KINDS)
def test_relevance_types(eng, ref_eng, kind):
    n = 4097
    rng = np.random.default_rng(21)
    log = _log(n, "zipf", seed=4)
    log["user_idx"] %= 30
    if kind == "int64_1to5":
        rel = rng.integers(1, 6, n).astype(np.int64)
    elif kind == "int32_1to5":
        rel = rng.integers(1, 6, n).astype(np.int32)
    elif kind == "fractional":
        rel = rng.integers(0, 9, n) * 0.375 + 1 / 3
    elif kind == "negative":
        rel = -rng.integers(0, 9, n) * 0.5 - 1e-9
    elif kind == "signed_zero":           # -0.0 next to +0.0 in one user: one relevance (CUB and numpy agree)
        rel = np.where(rng.integers(0, 2, n) == 0, -0.0, 0.0)
        rel[::5] = 1.0
    else:
        rel = (rng.integers(0, 9, n) * 0.3).astype(np.float32)
    log["relevance"] = rel
    noise = _noise(n, seed=6)
    for top_k in (1, 4):
        ref = _reference(log, top_k, noise)
        _check_build(eng, ref_eng, _one_call(eng, log, top_k, noise), ref)
        _check_build(eng, ref_eng, _chunked(eng, _arrow(log, cuts=[5, 2049]), top_k, noise), ref)


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
@pytest.mark.parametrize("entry", ["one_call", "chunked_arrow", "chunked_pandas"])
def test_non_finite_relevance_rejected_on_device(eng, ref_eng, entry, bad):
    """A NaN action would make every critic gradient NaN: the device flags it where it reads relevance, the build
    fails, no table is left, and the handle builds correctly afterwards."""
    log = _log(3000, "zipf", seed=8)
    log.loc[2999 if np.isnan(bad) else 1234, "relevance"] = bad
    src = log
    if entry == "chunked_arrow":             # (from_pandas would turn NaN into a null, which ingestion rejects earlier)
        src = _arrow(log)
        src = src.set_column(src.schema.get_field_index("relevance"), "relevance",
                             pa.chunked_array([pa.array(log["relevance"].to_numpy()[:1500]),
                                               pa.array(log["relevance"].to_numpy()[1500:])]))
        assert src.column("relevance").null_count == 0
    with pytest.raises(ValueError, match="non-finite"):
        if entry == "one_call":
            _one_call(eng, log, 2, None)
        else:
            _chunked(eng, src, 2, None)
    assert eng.n_transitions == 0
    good = _log(500, "zipf", seed=9)
    noise = _noise(500)
    _check_build(eng, ref_eng, _one_call(eng, good, 2, noise), _reference(good, 2, noise))


def test_top_k_edges(eng, ref_eng):
    """0, 1, 3, the longest episode -1 / +0 / +1, 2**31 - 1 and negatives: top_k <= 0 rewards nothing in both
    builders, a top_k past every episode rewards everything."""
    log = _log(2049, "zipf", seed=12)
    log["user_idx"] %= 25
    longest = int(log["user_idx"].value_counts().max())
    noise = _noise(len(log))
    for top_k in (0, 1, 3, longest - 1, longest, longest + 1, 2 ** 31 - 1, -1, -(2 ** 31)):
        ref = mdp.build_mdp(log, top_k=top_k, action_noise=noise)
        if top_k >= 0:
            ref = _reference(log, top_k, noise)
        if top_k <= 0:
            assert not ref.rew.any()
        if top_k >= longest:
            assert ref.rew.all()
        _check_build(eng, ref_eng, _one_call(eng, log, top_k, noise), ref, table=top_k in (0, 3))
        _check_build(eng, ref_eng, _chunked(eng, _arrow(log), top_k, noise), ref, table=False)


# ----------------------------------------------------------------------------- chunkings of the chunked API
_COLS = ("user_idx", "item_idx", "timestamp", "relevance", "action_noise")


def _columns(log, noise):
    c = {k: np.ascontiguousarray(log[k].to_numpy()) for k in _COLS[:4]}
    c["timestamp"] = np.ascontiguousarray(c["timestamp"].astype(np.int64))
    c["user_idx"], c["item_idx"] = c["user_idx"].astype(np.int32), c["item_idx"].astype(np.int32)
    c["relevance"] = c["relevance"].astype(np.float64)
    if noise is not None:
        c["action_noise"] = np.ascontiguousarray(noise, dtype=np.float64)
    return c


def _feed(eng, cols, plan, n, top_k=3):
    """plan: [(column, lo, hi)] appended in that order (each column's own dtype)."""
    eng.mdp_begin(n)
    keep = []
    for col, lo, hi in plan:
        a = np.ascontiguousarray(cols[col][lo:hi])
        keep.append(a)
        eng.mdp_append(col, a.ctypes.data if a.size else 0, a.dtype, hi - lo)
    return eng.mdp_finish(top_k, 1e-3, want_outputs=True, n_rows=n)


def _plan(kind, names, n, rng):
    if kind == "one_per_column":
        return [(c, 0, n) for c in names]
    if kind == "single_rows":
        return [(c, i, i + 1) for c in names for i in range(n)]
    if kind == "interleaved":
        cuts = np.unique(np.r_[0, rng.integers(0, n, 9), n])
        return [(c, a, b) for a, b in zip(cuts[:-1], cuts[1:]) for c in names]
    if kind == "zero_counts":
        out = []
        for c in names:
            out += [(c, 0, 0), (c, 0, n // 3), (c, n // 3, n // 3), (c, n // 3, n), (c, n, n)]
        return out
    raise AssertionError(kind)


@pytest.mark.parametrize("order", ["ts_first", "ts_last", "reversed", "noise_first"])
@pytest.mark.parametrize("kind,n", [("one_per_column", 4097), ("single_rows", 257), ("interleaved", 4097),
                                    ("zero_counts", 4097)])
def test_chunkings(eng, ref_eng, kind, n, order):
    names = {"ts_first": ["timestamp", "user_idx", "item_idx", "relevance", "action_noise"],
             "ts_last": ["user_idx", "item_idx", "relevance", "action_noise", "timestamp"],
             "reversed": ["action_noise", "relevance", "timestamp", "item_idx", "user_idx"],
             "noise_first": ["action_noise", "item_idx", "timestamp", "relevance", "user_idx"]}[order]
    log = _log(n, "zipf", seed=n + 1)
    noise = _noise(n, seed=2)
    ref = _reference(log, 3, noise)
    outs = _feed(eng, _columns(log, noise), _plan(kind, names, n, np.random.default_rng(0)), n)
    _check_build(eng, ref_eng, outs, ref)


def test_uneven_arrow_chunks_per_column(eng, ref_eng):
    """Each column cut at its own points, none on a slot boundary, one chunk larger than a ring slot."""
    n = SLOT_VALUES_8B + 4099
    log = _log(n, "zipf", seed=31)
    noise = _noise(n, seed=3)
    rng = np.random.default_rng(4)
    arrays = {}
    for c in _COLS[:4]:
        a = pa.Array.from_pandas(log[c])
        cuts = np.unique(np.r_[0, rng.integers(1, n, 5), n]) if c != "timestamp" else np.array([0, 1, n - 3, n])
        arrays[c] = pa.chunked_array([a.slice(lo, hi - lo) for lo, hi in zip(cuts[:-1], cuts[1:])])
    table = pa.table(arrays)
    assert table.column("timestamp").chunk(1).nbytes > 16 << 20
    _check_build(eng, ref_eng, _chunked(eng, table, 3, noise), _reference(log, 3, noise))


DTYPE_CASES = [(c, d) for c in _COLS for d in (np.int32, np.int64, np.float32, np.float64)]


@pytest.mark.parametrize("col,dtype", DTYPE_CASES, ids=[f"{c}-{np.dtype(d).name}" for c, d in DTYPE_CASES])
def test_column_dtypes(eng, ref_eng, col, dtype):
    """Every CQL_DT_* for every column; a float timestamp chunk is rejected, not truncated."""
    n = 3001
    log = _log(n, "zipf", seed=41)
    log["timestamp"] -= n // 8                                  # negative keys as well
    noise = (np.random.default_rng(5).integers(-40, 40, n) * 2.0 ** -12)      # exact in every dtype when col == noise
    cols = _columns(log, noise)
    if col == "action_noise" and np.dtype(dtype).kind == "i":
        noise = np.random.default_rng(5).integers(-2, 3, n).astype(np.float64)
        cols["action_noise"] = noise
    cols[col] = cols[col].astype(dtype)
    plan = _plan("interleaved", list(_COLS), n, np.random.default_rng(1))
    if col == "timestamp" and np.dtype(dtype).kind == "f":
        with pytest.raises(ValueError, match="timestamps must be int32 or int64"):
            _feed(eng, cols, plan, n)
        good = _columns(log, noise)
        _check_build(eng, ref_eng, _feed(eng, good, plan, n), _reference(log, 3, noise))
        return
    _check_build(eng, ref_eng, _feed(eng, cols, plan, n), _reference(log, 3, noise))


# ----------------------------------------------------------------------------- session handling
def test_back_to_back_builds_do_not_leak(eng, ref_eng):
    big, small = _log(70_001, "zipf", seed=51), _log(3001, "one_user", seed=52)
    nb, ns = _noise(len(big), 1), _noise(len(small), 2)
    _check_build(eng, ref_eng, _one_call(eng, big, 3, nb), mdp.build_mdp(big, top_k=3, action_noise=nb))
    _check_build(eng, ref_eng, _chunked(eng, _arrow(small), 3, ns), _reference(small, 3, ns))
    _check_build(eng, ref_eng, _chunked(eng, big, 3, nb), mdp.build_mdp(big, top_k=3, action_noise=nb))
    _check_build(eng, ref_eng, _one_call(eng, small, 3, ns), _reference(small, 3, ns))


def test_begin_while_open_drops_the_old_session(eng, ref_eng):
    old, log = _log(5000, "zipf", seed=53), _log(1500, "zipf", seed=54)
    noise = _noise(len(log))
    c = _columns(old, _noise(len(old)))
    _feed_partial = [("timestamp", 0, 5000), ("user_idx", 0, 2000), ("action_noise", 0, 100)]
    eng.mdp_begin(5000)
    for col, lo, hi in _feed_partial:
        eng.mdp_append(col, c[col][lo:hi].ctypes.data, c[col].dtype, hi - lo)
    outs = _feed(eng, _columns(log, noise), _plan("one_per_column", list(_COLS), len(log), None), len(log))
    _check_build(eng, ref_eng, outs, _reference(log, 3, noise))


def _raw_append(eng, col, dtype_code, arr, count):
    eng._check(eng._lib.cql_mdp_append(eng._h, col, dtype_code, arr.ctypes.data, count), "cql_mdp_append")


@pytest.mark.parametrize("case", ["append_past_n", "finish_incomplete_column", "partial_noise", "bad_column",
                                  "bad_dtype", "float_timestamp", "finish_without_begin", "append_without_begin"])
def test_error_paths_raise_and_leave_the_handle_usable(eng, ref_eng, case):
    n = 1000
    log = _log(n, "zipf", seed=61)
    noise = _noise(n)
    c = _columns(log, noise)
    with pytest.raises(ValueError):
        if case in ("finish_without_begin", "append_without_begin"):
            _feed(eng, c, [(k, 0, n) for k in _COLS[:4]], n)            # a complete session: closed by its finish
            if case == "finish_without_begin":
                eng.mdp_finish(3, 1e-3)
            else:
                eng.mdp_append("user_idx", c["user_idx"].ctypes.data, np.int32, n)
        else:
            eng.mdp_begin(n)
            for k in _COLS[:4]:
                if case == "finish_incomplete_column" and k == "item_idx":
                    eng.mdp_append(k, c[k].ctypes.data, c[k].dtype, n - 1)
                else:
                    eng.mdp_append(k, c[k].ctypes.data, c[k].dtype, n)
            if case == "append_past_n":
                eng.mdp_append("user_idx", c["user_idx"].ctypes.data, np.int32, 1)
            elif case == "partial_noise":
                eng.mdp_append("action_noise", c["action_noise"].ctypes.data, np.float64, n - 10)
            elif case == "bad_column":
                _raw_append(eng, 5, 3, c["relevance"], n)
            elif case == "bad_dtype":
                _raw_append(eng, 3, 4, c["relevance"], n)
            elif case == "float_timestamp":
                _raw_append(eng, 2, 3, c["relevance"], 1)
            eng.mdp_finish(3, 1e-3)
    _check_build(eng, ref_eng, _feed(eng, c, _plan("one_per_column", list(_COLS), n, None), n), _reference(log, 3, noise))


# ----------------------------------------------------------------------------- the large case
@pytest.fixture(scope="module")
def large():
    """~9 M rows: one column chunk spans several ring slots and the ring wraps inside one column; sorts and the
    max-scan span many tiles; Zipf-like episodes over 300 k users, items up to 2**24 - 1."""
    n = LARGE_N
    rng = np.random.default_rng(2024)
    users = ((rng.zipf(1.2, n) - 1) % 300_000).astype(np.int32)
    users[: n // 50] = 123_457                                      # one long episode
    log = pd.DataFrame({"user_idx": users, "item_idx": rng.integers(0, 2 ** 24, n).astype(np.int32),
                        "timestamp": rng.integers(-(10 ** 6), 10 ** 6, n) * 1_000_003,
                        "relevance": rng.integers(1, 6, n).astype(np.float64)})
    noise = _noise(n, seed=7)
    ref = mdp.build_mdp(log, top_k=10, action_noise=noise)
    return log, noise, ref


def _in_row_order(outs):
    act, order = outs[1], outs[4]
    out = np.empty_like(act)
    out[order] = act
    return out


def test_large_parity(eng, ref_eng, large):
    log, noise, ref = large
    n = len(log)
    assert n * 8 > 4 * (16 << 20)                                  # 8-byte columns wrap the 4-slot ring
    _check_build(eng, ref_eng, _one_call(eng, log, 10, noise), ref)
    table = _arrow(log.assign(relevance=log["relevance"].astype(np.float32)), cuts=[3, 5_000_000, 5_000_001, 7_777_777])
    _check_build(eng, ref_eng, _chunked(eng, table, 10, noise), ref, table=False)
    _check_build(eng, ref_eng, _chunked(eng, log, 10, noise), ref, table=False)


def test_large_seeded_device_noise(engine_factory, eng, large):
    """The device's own noise is a function of (handle seed, original row): the same bits through every entry point
    and chunking, for a prefix of the log on its own, different under another seed; scale 0 adds nothing; and it
    is N(0, scale^2)."""
    from scipy import stats
    log, _, _ = large
    n = len(log)
    rel32 = log["relevance"].to_numpy().astype(np.float32)
    base = _in_row_order(_one_call(eng, log, 10, None))
    variants = [_chunked(eng, _arrow(log, cuts=[1, 2 * SLOT_VALUES_8B + 5, 6_000_000]), 10, None),
                _chunked(eng, _arrow(log, n_chunks=97), 10, None),
                _chunked(eng, log, 10, None)]
    for outs in variants:
        assert _same_bits(_in_row_order(outs), base)
    m = 1_048_579
    assert _same_bits(_in_row_order(_one_call(eng, log.iloc[:m], 10, None)), base[:m])
    other = engine_factory(batch_size=64, seed=777)
    diff = _in_row_order(_one_call(other, log, 10, None)) != base
    assert diff.mean() > 0.99
    other.close()
    zero = _in_row_order(_one_call(eng, log, 10, None, scale=0.0))
    assert _same_bits(zero, rel32)
    # the distribution, at scale 1 (float32 rounding of the action is ~1e-6 of a standard deviation there)
    z = _in_row_order(_one_call(eng, log, 10, None, scale=1.0)).astype(np.float64) - rel32
    mean, sd = z.mean(), z.std()
    assert abs(mean) < 5.0 / np.sqrt(n), mean
    assert abs(sd - 1.0) < 5.0 / np.sqrt(2 * n), sd
    assert stats.kstest(z, "norm").pvalue > 1e-4


# ----------------------------------------------------------------------------- seen-items CSR
def _seen_reference(users, items, n_users_dim, wanted=None):
    """Dict of sorted sets kept to the device's contract: users outside [0, n_users_dim), users whose `wanted` flag
    is zero or missing, and negative items are dropped; each user's items ascending and unique."""
    users, items = np.asarray(users, np.int64), np.asarray(items, np.int64)
    keep = (users >= 0) & (users < n_users_dim) & (items >= 0)
    if wanted is not None:
        w = np.zeros(n_users_dim, dtype=bool)
        w[: min(len(wanted), n_users_dim)] = np.asarray(wanted, dtype=bool)[:n_users_dim]
        keep &= w[np.clip(users, 0, n_users_dim - 1)]
    per_user = {}
    if keep.any():
        groups = pd.Series(items[keep]).groupby(users[keep]).unique()
        per_user = {int(u): sorted(set(v.tolist())) for u, v in groups.items()}
    counts = np.zeros(n_users_dim, dtype=np.int64)
    for u, s in per_user.items():
        counts[u] = len(s)
    indptr = np.zeros(n_users_dim + 1, dtype=np.int64)
    np.cumsum(counts, out=indptr[1:])
    seen = np.array([i for u in sorted(per_user) for i in per_user[u]], dtype=np.int32)
    return indptr, seen


def _check_seen(eng, users, items, n_users_dim, wanted=None):
    indptr_t, seen_t = eng.seen_csr_device(users, items, n_users_dim, wanted=wanted)
    want_ptr, want_seen = _seen_reference(users, items, n_users_dim, wanted)
    got_ptr, got_seen = indptr_t.cpu().numpy(), seen_t.cpu().numpy()
    assert np.array_equal(got_ptr, want_ptr)
    assert got_seen.size == want_seen.size == want_ptr[-1]              # n_seen
    assert np.array_equal(got_seen, want_seen)


def _seen_log(n, n_users_dim, seed):
    rng = np.random.default_rng(seed)
    users = rng.integers(-3, n_users_dim + 3, n)
    users[: n // 3] = rng.integers(0, min(n_users_dim, 40), n // 3)       # some users with many rows / duplicates
    items = rng.integers(0, 300, n)
    pick = rng.integers(0, 10, n)
    items[pick == 0] = 2 ** 31 - 1
    items[pick == 1] = 0
    items[pick == 2] = -rng.integers(1, 2 ** 31, int((pick == 2).sum()))
    return users.astype(np.int32), items.astype(np.int32)


@pytest.mark.parametrize("n_users_dim", [1, 2, 255, 256, 257, 2 ** 20, 2 ** 24])
def test_seen_csr_user_dims(eng, n_users_dim):
    users, items = _seen_log(50_000, n_users_dim, seed=n_users_dim)
    _check_seen(eng, users, items, n_users_dim)
    _check_seen(eng, users[:1], items[:1], n_users_dim)


def test_seen_csr_negative_items_are_dropped(eng):
    """Item -1 used to be filed after the user's positive items (an unsorted row for the scorer's binary search)."""
    users = np.array([2, 2, 2, 1, 3], np.int32)
    items = np.array([5, -1, 0, -2 ** 31, 2 ** 31 - 1], np.int32)
    indptr, seen = eng.seen_csr_device(users, items, 4)
    assert indptr.cpu().tolist() == [0, 0, 0, 2, 3] and seen.cpu().tolist() == [0, 5, 2 ** 31 - 1]
    assert mdp.seen_csr(pd.DataFrame({"user_idx": users, "item_idx": items}), 4)[1].tolist() == [0, 5, 2 ** 31 - 1]


@pytest.mark.parametrize("mask", ["all_zero", "all_one", "shorter", "random"])
@pytest.mark.parametrize("n_users_dim", [257, 2 ** 20])
def test_seen_csr_wanted_masks(eng, n_users_dim, mask):
    users, items = _seen_log(60_000, n_users_dim, seed=7)
    rng = np.random.default_rng(3)
    wanted = {"all_zero": np.zeros(n_users_dim, np.uint8), "all_one": np.ones(n_users_dim, np.uint8),
              "shorter": np.ones(n_users_dim // 3, np.uint8),
              "random": rng.integers(0, 2, n_users_dim).astype(bool)}[mask]
    _check_seen(eng, users, items, n_users_dim, wanted)


def test_seen_csr_every_row_dropped_and_empty(eng):
    _check_seen(eng, np.array([-1, 5, 9, 2], np.int32), np.array([1, 2, 3, -4], np.int32), 5)
    _check_seen(eng, np.zeros(0, np.int32), np.zeros(0, np.int32), 3)


def test_seen_csr_large(eng, large):
    log, _, _ = large
    users, items = log["user_idx"].to_numpy().copy(), log["item_idx"].to_numpy().copy()
    items[::1000] = -5
    users[7::1001] = 2 ** 20 + 3                                      # past n_users_dim: dropped
    _check_seen(eng, users, items, 2 ** 20)
    _check_seen(eng, users, items, 2 ** 20, wanted=(np.arange(2 ** 20) % 3 != 0))


# ----------------------------------------------------------------------------- model level
@pytest.mark.parametrize("kind", ["float_ties", "tz_datetime"])
def test_fit_arrow_equals_fit_pandas_for_timestamp_types(kind):
    """`CQL.fit(pyarrow.Table)` and `CQL.fit(pandas.DataFrame)` of one log land on the same model bit for bit."""
    from replay_cql_b200.models import CQL
    from replay_cql_b200.synthetic import make_log
    log = make_log("tiny")
    rng = np.random.default_rng(9)
    if kind == "float_ties":
        log["timestamp"] = rng.integers(-8, 8, len(log)) * 0.5
    else:
        log["timestamp"] = pd.to_datetime(log["timestamp"] % 50, unit="D").dt.tz_localize("UTC").dt.tz_convert("Asia/Kolkata")
    kw = dict(top_k=3, n_epochs=1, n_steps_per_epoch=12, batch_size=64, seed=3)
    a, b = CQL(**kw), CQL(**kw)
    a.fit(log)
    b.fit(_arrow(log, n_chunks=4))
    assert np.array_equal(a.engine.get_state(), b.engine.get_state())
    ref = mdp.build_mdp(log, top_k=3, action_noise=np.zeros(len(log)))
    outs = mdp.ingest_log(b.engine, _arrow(log, n_chunks=4), top_k=3, action_noise=np.zeros(len(log)), want_outputs=True)
    assert np.array_equal(outs[2], ref.rew) and np.array_equal(outs[4], ref.order)
    a.engine.close(); b.engine.close()
