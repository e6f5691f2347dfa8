"""MDP builder: interaction log -> episode-ordered (observation, action, reward, terminal).

Replaces the RePlay CQL wrapper's ``MdpDatasetBuilder.build`` ([EXT] upstream
``replay/experimental/models/cql.py``; SURVEY.md Appendix B) -- two Spark window
sorts, a global ``orderBy`` and ``toPandas()`` -- with vectorised sorts over the
Arrow/pandas columns, written straight into (pinned, when CUDA is up) host
buffers that ``cql_load_transitions`` uploads and expands on the GPU.

Semantics (one episode per user):
* global order (user_idx, timestamp) ascending; ties keep input order;
* reward = 1 for the user's ``top_k`` rows by (relevance desc, timestamp desc), else 0;
* terminal = 1 on the user's last row in that order;
* action = relevance + N(0,1) * ``action_randomization_scale``;
* observation = (user_idx, item_idx) as float32 (exact below 2**24).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Optional

import numpy as np
from pandas.api import types as pd_api

from .frames import to_pandas, timestamps_to_int64


@dataclass
class MdpArrays:
    obs: np.ndarray    # [n, 2] float32
    act: np.ndarray    # [n] float32
    rew: np.ndarray    # [n] float32
    term: np.ndarray   # [n] float32
    order: np.ndarray  # [n] int64: original row of each step

    def __len__(self) -> int:
        return int(self.obs.shape[0])


def alloc_host(shape, dtype=np.float32) -> np.ndarray:
    """Host buffer for H2D staging: pinned when a CUDA context can be created, else pageable."""
    try:
        import torch
        if torch.cuda.is_available():
            t = torch.empty(shape, dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
            return t.numpy()
    except Exception:  # pragma: no cover
        pass
    return np.empty(shape, dtype=dtype)


def build_mdp(log: Any, top_k: int = 10, action_randomization_scale: float = 1e-3,
              seed: Optional[int] = None, action_noise: Optional[np.ndarray] = None) -> MdpArrays:
    """``action_noise`` (per ORIGINAL row, already scaled) overrides the seeded draw (parity tests)."""
    pdf = to_pandas(log)
    for col in ("user_idx", "item_idx", "timestamp", "relevance"):
        if col not in pdf.columns:
            raise ValueError(f"log must have column {col}")
    n = len(pdf)
    user = pdf["user_idx"].to_numpy().astype(np.int64)
    item = pdf["item_idx"].to_numpy().astype(np.int64)
    if n and (user.max() >= 2 ** 24 or item.max() >= 2 ** 24):
        raise ValueError("user_idx/item_idx must be < 2**24 to be exact in float32 observations")
    ts = timestamps_to_int64(pdf["timestamp"])
    rel = pdf["relevance"].to_numpy().astype(np.float64)
    if not np.isfinite(rel).all():
        raise ValueError("relevance column has a non-finite value")
    row = np.arange(n, dtype=np.int64)

    order = np.lexsort((row, ts, user))                      # (user, timestamp, input order)
    u_sorted = user[order]
    term = np.ones(n, dtype=np.float32)
    if n > 1:
        term[:-1] = (u_sorted[1:] != u_sorted[:-1]).astype(np.float32)

    rank_order = np.lexsort((row, ~ts, -rel, user))          # (user, relevance desc, timestamp desc); ~ts = -ts - 1
                                                             # reverses every int64, INT64_MIN included
    ur = user[rank_order]
    starts = np.flatnonzero(np.r_[True, ur[1:] != ur[:-1]]) if n else np.zeros(0, dtype=np.int64)
    group_start = np.repeat(starts, np.diff(np.r_[starts, n])) if n else starts
    pos_in_user = np.arange(n, dtype=np.int64) - group_start
    rewarded = np.zeros(n, dtype=np.float32)
    rewarded[rank_order] = (pos_in_user < top_k).astype(np.float32)

    if action_noise is None:
        rng = np.random.default_rng(seed)
        action_noise = rng.standard_normal(n) * action_randomization_scale
    action = rel.astype(np.float32).astype(np.float64) + np.asarray(action_noise, dtype=np.float64)

    obs = alloc_host((n, 2))
    obs[:, 0] = u_sorted
    obs[:, 1] = item[order]
    act = alloc_host((n,)); act[:] = action[order]
    rew = alloc_host((n,)); rew[:] = rewarded[order]
    trm = alloc_host((n,)); trm[:] = term
    return MdpArrays(obs, act, rew, trm, order)


def to_transitions(mdp: MdpArrays) -> dict:
    """Host-side expansion into (s, a, r, s', done) -- what the GPU loader builds; for tests / e2e batches."""
    n = len(mdp)
    nxt = np.zeros((n, 2), dtype=np.float32)
    if n > 1:
        nxt[:-1] = mdp.obs[1:]
    nxt[mdp.term > 0] = 0.0
    return {"obs": mdp.obs, "act": mdp.act.reshape(-1, 1), "rew": mdp.rew.reshape(-1, 1),
            "next_obs": nxt, "term": mdp.term.reshape(-1, 1)}


def seen_csr(log: Any, n_users_dim: int):
    """Per-user sorted, de-duplicated seen items as CSR over user id (for the lazy seen filter).  Rows with a negative
    user or item are dropped (no candidate id is negative, so they filter nothing); a user at or past ``n_users_dim``
    widens the CSR."""
    pdf = to_pandas(log)
    user = pdf["user_idx"].to_numpy().astype(np.int64)
    item = pdf["item_idx"].to_numpy().astype(np.int64)
    keep = (user >= 0) & (item >= 0)
    if not keep.all():
        user, item = user[keep], item[keep]
    if user.size:
        n_users_dim = max(n_users_dim, int(user.max()) + 1)
    key = user * (2 ** 32) + item
    key.sort()                                  # (sort + neighbour mask: numpy's hash-based unique is ~4x slower on 1e6..2e7 keys)
    if key.size:
        key = key[np.concatenate(([True], key[1:] != key[:-1]))]
    u, i = key >> 32, (key & 0xFFFFFFFF).astype(np.int32)
    counts = np.bincount(u, minlength=n_users_dim)
    indptr = np.zeros(n_users_dim + 1, dtype=np.int64)
    np.cumsum(counts, out=indptr[1:])
    return indptr, i


# ----------------------------------------------------------------------------- ingestion without intermediate frames
def _column_chunks(log: Any, name: str):
    """Yield ``(address, numpy dtype, count, keepalive)`` for every chunk of column ``name`` -- WITHOUT materialising a
    frame: a pyarrow column is walked buffer by buffer (zero copy), a pandas column is one chunk of its own array."""
    from . import frames
    pa = frames.pa
    if pa is not None and isinstance(log, (pa.Table, pa.RecordBatch)):
        col = log.column(name)
        chunks = col.chunks if isinstance(col, pa.ChunkedArray) else [col]
        for ch in chunks:
            if len(ch) == 0:
                continue
            if ch.null_count:
                raise ValueError(f"column {name} has nulls")
            t = ch.type
            if pa.types.is_timestamp(t) or pa.types.is_date64(t) or pa.types.is_duration(t):
                ch, t = ch.view(pa.int64()), pa.int64()              # same buffer, order-preserving for one unit
            elif pa.types.is_date32(t):
                ch, t = ch.view(pa.int32()), pa.int32()              # days since the epoch
            if name == "timestamp" and pa.types.is_floating(t):      # float timestamps: the host's order-preserving key
                key = timestamps_to_int64(ch.to_numpy(zero_copy_only=False))
                yield key.ctypes.data, key.dtype, key.size, key
                continue
            if not (pa.types.is_integer(t) or pa.types.is_floating(t)) or t.bit_width not in (32, 64) or \
                    (pa.types.is_integer(t) and not pa.types.is_signed_integer(t)):
                ch = ch.cast(pa.float64() if pa.types.is_floating(t) or pa.types.is_decimal(t) else pa.int64())
                t = ch.type
            dt = np.dtype(t.to_pandas_dtype())
            buf = ch.buffers()[1]
            yield buf.address + ch.offset * dt.itemsize, dt, len(ch), ch
        return
    pdf = to_pandas(log)
    ser = pdf[name]
    if name == "timestamp" and not (pd_api.is_integer_dtype(ser.dtype) and ser.dtype.itemsize in (4, 8)):
        arr = timestamps_to_int64(ser)
    else:
        arr = ser.to_numpy()
        if arr.dtype not in (np.int32, np.int64, np.float32, np.float64):
            arr = arr.astype(np.float64 if np.issubdtype(arr.dtype, np.floating) else np.int64)
    arr = np.ascontiguousarray(arr)
    yield arr.ctypes.data, arr.dtype, arr.size, arr


def _n_rows(log: Any) -> int:
    return int(log.num_rows) if hasattr(log, "num_rows") else len(log)


def _check_ids(log: Any) -> None:
    from . import frames
    pa = frames.pa
    for name in ("user_idx", "item_idx"):
        if pa is not None and isinstance(log, (pa.Table, pa.RecordBatch)):
            import pyarrow.compute as pc
            mm = pc.min_max(log.column(name))
            lo, hi = mm["min"].as_py(), mm["max"].as_py()
        else:
            col = to_pandas(log)[name]
            lo, hi = col.min(), col.max()
        if lo < 0 or hi >= 2 ** 24:
            raise ValueError("user_idx/item_idx must be in [0, 2**24) to be exact in float32 observations")


def ingest_log(engine, log: Any, top_k: int = 10, action_randomization_scale: float = 1e-3,
               action_noise: Optional[np.ndarray] = None, want_outputs: bool = False):
    """Interaction log -> replay table in HBM, the Spark-free replacement of ``log.toPandas()`` + the window-sort MDP
    builder (SURVEY.md 8f-1; pattern being replaced: ``replay/models/neuromf.py:332``).  ``log``: ``pyarrow.Table`` /
    ``RecordBatch`` (e.g. ``pyarrow.parquet.read_table``: each column's chunks = the file's row groups), or a pandas
    frame.  No intermediate frame is built: every chunk's buffer goes host -> pinned ring -> device in its own dtype
    (``cql_mdp_append``), timestamps first so that their radix sorts overlap the other uploads."""
    n = _n_rows(log)
    if n == 0:
        raise ValueError("empty log")
    names = log.column_names if hasattr(log, "column_names") else list(log.columns)
    for col in ("user_idx", "item_idx", "timestamp", "relevance"):
        if col not in names:
            raise ValueError(f"log must have column {col}")
    _check_ids(log)
    engine.mdp_begin(n)
    for col in ("timestamp", "user_idx", "item_idx", "relevance"):
        for address, dt, count, _keep in _column_chunks(log, col):
            engine.mdp_append(col, address, dt, count)
    if action_noise is not None:
        nz = np.ascontiguousarray(action_noise, dtype=np.float64)
        if nz.size != n:
            raise ValueError("action_noise must have one value per log row")
        engine.mdp_append("action_noise", nz.ctypes.data, nz.dtype, n)
    return engine.mdp_finish(top_k, action_randomization_scale, want_outputs=want_outputs, n_rows=n)


def build_mdp_on_device(engine, log: Any, top_k: int = 10, action_randomization_scale: float = 1e-3,
                        action_noise: Optional[np.ndarray] = None, want_outputs: bool = False):
    """Same semantics as :func:`build_mdp`, but sorted and expanded on the GPU: the log columns go host -> device once
    (chunk by chunk through a pinned ring, :func:`ingest_log`) and the replay table never exists on the host."""
    return ingest_log(engine, log, top_k=top_k, action_randomization_scale=action_randomization_scale,
                      action_noise=action_noise, want_outputs=want_outputs)


# ----------------------------------------------------------------------------- data-parallel: the table sharded by user
def user_shard_bounds(user_counts: np.ndarray, world: int) -> np.ndarray:
    """Contiguous user-id ranges ``[bounds[r], bounds[r + 1])`` for ``world`` ranks, balanced by ROW count
    (``user_counts[u]`` = rows of user ``u``).  A user's episode is never split (SURVEY.md 8e: MDP build shards by user)."""
    if world < 1:
        raise ValueError("world must be >= 1")
    counts = np.asarray(user_counts, dtype=np.int64)
    csum = np.concatenate([[0], np.cumsum(counts)])
    total = int(csum[-1])
    targets = (np.arange(1, world, dtype=np.int64) * total) // world
    cuts = np.searchsorted(csum, targets, side="left")        # first user boundary at or past each target
    bounds = np.concatenate([[0], cuts, [counts.size]]).astype(np.int64)
    return np.maximum.accumulate(bounds)


def shard_log_by_user(log: Any, rank: int, world: int):
    """This rank's rows of ``log`` (all rows of the users in its range) -- pyarrow in, pyarrow out; pandas in, pandas out."""
    from . import frames
    pa = frames.pa
    if world == 1:
        return log
    if pa is not None and isinstance(log, pa.Table):
        import pyarrow.compute as pc
        user = log.column("user_idx").to_numpy()
    else:
        user = to_pandas(log)["user_idx"].to_numpy()
    counts = np.bincount(user, minlength=int(user.max()) + 1 if user.size else 1)
    b = user_shard_bounds(counts, world)
    mask = (user >= b[rank]) & (user < b[rank + 1])
    if pa is not None and isinstance(log, pa.Table):
        return log.filter(pa.array(mask))
    return to_pandas(log)[mask]
