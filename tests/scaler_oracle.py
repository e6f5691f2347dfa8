"""CPU restatement of d3rlpy's observation / action / reward scalers.  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED ([EXT-UNVERIFIED], DESIGN.md section 1): restated from d3rlpy 1.x ``preprocessing/scalers.py``,
``action_scalers.py`` and ``reward_scalers.py``.  ``fit`` runs over every step's one-step observation, action and
reward as slow per-episode loops in float64 (two passes for the standard scaler, like d3rlpy); the transforms are
separately rounded float32 torch ops.  Shares nothing with the CUDA statistics and transform kernels, nor with the
product's ``replay_cql_b200.scalers``.  The update oracle (``oracle.cql_oracle.update``) is fed transformed batches.
"""
from __future__ import annotations

import numpy as np
import torch


def _episodes(term):
    out, start, n = [], 0, len(term)
    for i in range(n):
        if term[i] != 0 or i == n - 1:
            out.append((start, i + 1))
            start = i + 1
    return out


def fit(obs, act, rew, term) -> dict:
    """Episode-ordered one-step steps -> per column (obs.x, obs.y, act, rew): count, min, max, mean, std (population)."""
    obs = np.asarray(obs, dtype=np.float32).reshape(-1, 2)
    cols = [obs[:, 0], obs[:, 1], np.asarray(act, np.float32).reshape(-1), np.asarray(rew, np.float32).reshape(-1)]
    eps = _episodes(np.asarray(term).reshape(-1))
    out = {k: [] for k in ("count", "min", "max", "mean", "std")}
    for x in cols:
        n, total, lo, hi = 0, 0.0, np.inf, -np.inf
        for a, b in eps:
            v = x[a:b].astype(np.float64)
            n += b - a
            total += float(np.sum(v))
            lo, hi = min(lo, float(np.min(v))), max(hi, float(np.max(v)))
        mean = total / n
        sq = 0.0
        for a, b in eps:
            sq += float(np.sum((x[a:b].astype(np.float64) - mean) ** 2))
        for k, v in zip(out, (n, lo, hi, mean, np.sqrt(sq / n))):
            out[k].append(v)
    return {k: np.asarray(v) for k, v in out.items()}


def params(kind: str, cols, stats) -> dict:
    """d3rlpy's fitted parameters of ``cols`` (indices into the fit's columns), float32-rounded as the kernels take them."""
    if kind == "min_max":
        return {"type": "min_max", "minimum": [float(np.float32(stats["min"][c])) for c in cols],
                "maximum": [float(np.float32(stats["max"][c])) for c in cols]}
    return {"type": "standard", "mean": [float(np.float32(stats["mean"][c])) for c in cols],
            "std": [float(np.float32(stats["std"][c])) for c in cols]}


def _affine(p):
    """(offset, denominator) float32 tensors: min_max (min, max - min), standard (mean, std + 1e-3), each rounded once."""
    if p["type"] == "min_max":
        a, b = np.float32(p["minimum"]), np.float32(p["maximum"])
        return torch.from_numpy(np.atleast_1d(a)), torch.from_numpy(np.atleast_1d(np.float32(b - a)))
    a, b = np.float32(p["mean"]), np.float32(p["std"])
    return torch.from_numpy(np.atleast_1d(a)), torch.from_numpy(np.atleast_1d(np.float32(b + np.float32(1e-3))))


def obs_fwd(p, x):
    """[..., 2] float32 observations -> scaled (``p`` None: unchanged)."""
    if p is None:
        return x
    off, den = _affine(p)
    return (x - off) / den


def rew_fwd(p, r):
    if p is None:
        return r
    off, den = _affine(p)
    return (r - off) / den


def act_fwd(p, a):
    if p is None:
        return a
    off, den = _affine(p)
    return ((a - off) / den) * 2.0 - 1.0


def act_rev(p, a):
    if p is None:
        return a
    off, den = _affine(p)
    return ((a + 1.0) / 2.0) * den + off


def transform_rows(prep: dict, rows) -> np.ndarray:
    """[n, 8] table rows (s.x s.y a r s'.x s'.y term discount) -> the rows the network sees: s, s' (a terminal row's
    (0, 0) included), a and r transformed; term and discount untouched.  ``prep``: {scaler, action_scaler,
    reward_scaler} -> explicit dict or None."""
    t = torch.from_numpy(np.array(rows, dtype=np.float32))
    out = t.clone()
    out[:, 0:2] = obs_fwd(prep.get("scaler"), t[:, 0:2])
    out[:, 4:6] = obs_fwd(prep.get("scaler"), t[:, 4:6])
    out[:, 2:3] = act_fwd(prep.get("action_scaler"), t[:, 2:3])
    out[:, 3:4] = rew_fwd(prep.get("reward_scaler"), t[:, 3:4])
    return out.numpy()


def transform_batch(prep: dict, batch: dict) -> dict:
    """Oracle minibatch (torch tensors obs [B,2], act, rew, next_obs, term, optional discount) -> transformed copy."""
    out = dict(batch)
    out["obs"] = obs_fwd(prep.get("scaler"), batch["obs"])
    out["next_obs"] = obs_fwd(prep.get("scaler"), batch["next_obs"])
    out["act"] = act_fwd(prep.get("action_scaler"), batch["act"])
    out["rew"] = rew_fwd(prep.get("reward_scaler"), batch["rew"])
    return out
