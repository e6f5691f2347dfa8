"""d3rlpy's observation, action and reward scalers (``scaler``, ``action_scaler``, ``reward_scaler``) on the host side:
kind validation, the explicit-parameter (JSON) form, the mapping from the replay table's column statistics to
parameters, and the rank-order combination of per-shard statistics.  The transforms themselves run in the CUDA kernels
(``cql_set_preprocessing``; semantics in DESIGN.md section 1).

A scaler is ``None``, a kind name fitted on the table, or an explicit-parameter dict that round-trips through JSON:
``{"type": "min_max", "minimum": [..], "maximum": [..]}`` or ``{"type": "standard", "mean": [..], "std": [..]}``, one
value per column (observations: user, item; action and reward: one).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Union

import numpy as np

from . import _lib

KINDS = {"scaler": ("min_max", "standard"), "action_scaler": ("min_max",), "reward_scaler": ("min_max", "standard")}
COLUMNS = {"scaler": (0, 1), "action_scaler": (2,), "reward_scaler": (3,)}      # cql_table_stats.col indices
COLUMN_NAMES = ("obs.x (user_idx)", "obs.y (item_idx)", "act (relevance)", "rew")
PARAM_KEYS = {"min_max": ("minimum", "maximum"), "standard": ("mean", "std")}
STAT_KEYS = ("count", "min", "max", "mean", "m2")
_KIND_CODE = {None: _lib.SCALER_NONE, "min_max": _lib.SCALER_MIN_MAX, "standard": _lib.SCALER_STANDARD}

Spec = Union[None, str, dict]


def validate(arg: str, value: Spec) -> Spec:
    """``value`` of the ``CQL`` argument ``arg`` -> None, the kind name, or a normalised explicit-parameter dict
    (lists of floats).  Raises ``ValueError`` for anything else."""
    kinds = KINDS[arg]
    if value is None:
        return None
    if isinstance(value, str):
        if value not in kinds:
            raise ValueError(f"{arg}={value!r} is not supported: use None, one of {list(kinds)} or an explicit-parameter "
                             f"dict")
        return value
    if not isinstance(value, dict):
        raise ValueError(f"{arg} must be None, one of {list(kinds)} or an explicit-parameter dict")
    kind = value.get("type")
    if kind not in kinds:
        raise ValueError(f"{arg}: type {kind!r} is not supported, use one of {list(kinds)}")
    keys = PARAM_KEYS[kind]
    extra = set(value) - {"type", *keys}
    if extra:
        raise ValueError(f"{arg}: unknown keys {sorted(extra)} (a {kind} scaler takes {list(keys)})")
    out = {"type": kind}
    n_cols = len(COLUMNS[arg])
    for key in keys:
        if key not in value:
            raise ValueError(f"{arg}: a {kind} scaler needs {list(keys)}")
        v = np.asarray(value[key], dtype=np.float64).reshape(-1)
        if v.size != n_cols or not np.all(np.isfinite(v)):
            raise ValueError(f"{arg}: {key} must be {n_cols} finite value(s)")
        out[key] = [float(np.float32(x)) for x in v]        # the kernels' parameters are float32
    a, b = (np.asarray(out[k], dtype=np.float32) for k in keys)
    for j, c in enumerate(COLUMNS[arg]):
        if kind == "min_max" and not b[j] > a[j]:
            raise ValueError(f"{arg}: maximum must exceed minimum for column {COLUMN_NAMES[c]}")
        if kind == "standard" and b[j] < 0:
            raise ValueError(f"{arg}: std must be >= 0 for column {COLUMN_NAMES[c]}")
    return out


def params_from_stats(arg: str, kind: str, stats: dict) -> dict:
    """Fit: the table's column statistics -> explicit parameters.  min/max are column values; mean and the population
    std ``sqrt(M2 / n)`` are float64 statistics rounded once to float32."""
    cols = COLUMNS[arg]
    if arg == "reward_scaler" and not stats["rew_available"]:
        raise ValueError("reward_scaler: the table's reward statistics are unavailable (its rows were uploaded verbatim "
                         "with n_steps > 1, so the reward slot holds n-step returns); give reward_scaler as a dict")
    if any(int(stats["count"][c]) == 0 for c in cols):
        raise ValueError(f"{arg}: no replay table to fit on")
    if kind == "min_max":
        lo = [float(stats["min"][c]) for c in cols]
        hi = [float(stats["max"][c]) for c in cols]
        for c, a, b in zip(cols, lo, hi):
            if a == b:
                raise ValueError(f"{arg}='min_max': column {COLUMN_NAMES[c]} is constant ({a}), so max - min is 0")
        return {"type": "min_max", "minimum": lo, "maximum": hi}
    mean = [float(np.float32(stats["mean"][c])) for c in cols]
    std = [float(np.float32(np.sqrt(stats["m2"][c] / stats["count"][c]))) for c in cols]
    return {"type": "standard", "mean": mean, "std": std}


def resolve(specs: Dict[str, Spec], stats: Optional[dict]) -> Dict[str, Optional[dict]]:
    """{arg: validated spec} -> {arg: explicit dict or None}: names are fitted on ``stats``, dicts are kept as they are."""
    out = {}
    for arg in KINDS:
        spec = validate(arg, specs.get(arg))
        if isinstance(spec, str):
            if stats is None:
                raise ValueError(f"{arg}={spec!r} needs table statistics to fit on")
            spec = params_from_stats(arg, spec, stats)
        out[arg] = spec
    return out


def to_struct(params: Dict[str, Optional[dict]]) -> "_lib.Preprocessing":
    """Explicit parameters (``resolve`` output) -> ``struct cql_preprocessing``."""
    p = _lib.Preprocessing()
    for arg, prefix in (("scaler", "obs"), ("action_scaler", "act"), ("reward_scaler", "rew")):
        spec = validate(arg, params.get(arg))
        if isinstance(spec, str):
            raise ValueError(f"{arg}={spec!r} must be fitted first (see resolve)")
        kind = None if spec is None else spec["type"]
        setattr(p, f"{prefix}_kind", _KIND_CODE[kind])
        if spec is None:
            continue
        a, b = (spec[k] for k in PARAM_KEYS[kind])
        if prefix == "obs":
            p.obs_a[0], p.obs_a[1] = a
            p.obs_b[0], p.obs_b[1] = b
        else:
            setattr(p, f"{prefix}_a", a[0])
            setattr(p, f"{prefix}_b", b[0])
    return p


def from_struct(p: "_lib.Preprocessing") -> Dict[str, Optional[dict]]:
    """``struct cql_preprocessing`` -> {arg: explicit dict or None} (float32 values as Python floats)."""
    names = {v: k for k, v in _KIND_CODE.items()}
    out = {}
    for arg, prefix in (("scaler", "obs"), ("action_scaler", "act"), ("reward_scaler", "rew")):
        kind = names[int(getattr(p, f"{prefix}_kind"))]
        if kind is None:
            out[arg] = None
            continue
        if prefix == "obs":
            a, b = list(p.obs_a), list(p.obs_b)
        else:
            a, b = [getattr(p, f"{prefix}_a")], [getattr(p, f"{prefix}_b")]
        ka, kb = PARAM_KEYS[kind]
        out[arg] = {"type": kind, ka: [float(x) for x in a], kb: [float(x) for x in b]}
    return out


def stats_to_array(stats: dict) -> np.ndarray:
    """Statistics dict -> float64 [21] (count, min, max, mean, m2 per column, then rew_available), for all-gathers."""
    return np.concatenate([np.asarray(stats[k], dtype=np.float64) for k in STAT_KEYS] +
                          [np.array([1.0 if stats["rew_available"] else 0.0])])


def stats_from_array(a: np.ndarray) -> dict:
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    out = {k: a[4 * j: 4 * j + 4].copy() for j, k in enumerate(STAT_KEYS)}
    out["count"] = out["count"].astype(np.int64)
    out["rew_available"] = bool(a[20] != 0)
    return out


def combine(parts: List[dict]) -> dict:
    """Statistics of a table sharded over ranks, from the per-rank statistics in rank order: Chan's pairwise
    ``(n, mean, M2)`` merge and min/max, in float64 (the same order on every rank, hence the same bits)."""
    n = np.zeros(4)
    mean, m2 = np.zeros(4), np.zeros(4)
    lo, hi = np.full(4, np.inf), np.full(4, -np.inf)
    for p in parts:
        for c in range(4):
            nb = float(p["count"][c])
            if nb == 0:
                continue
            na = n[c]
            if na == 0:
                n[c], mean[c], m2[c] = nb, float(p["mean"][c]), float(p["m2"][c])
            else:
                tot = na + nb
                d = float(p["mean"][c]) - mean[c]
                mean[c] = mean[c] + d * (nb / tot)
                m2[c] = m2[c] + float(p["m2"][c]) + d * d * (na * nb / tot)
                n[c] = tot
            lo[c], hi[c] = min(lo[c], float(p["min"][c])), max(hi[c], float(p["max"][c]))
    return {"count": n.astype(np.int64), "min": lo, "max": hi, "mean": mean, "m2": m2,
            "rew_available": all(bool(p["rew_available"]) for p in parts)}
