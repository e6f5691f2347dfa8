"""CPU: d3rlpy's scalers as the product restates them (``replay_cql_b200.scalers``) and as the test oracle does
(``tests/scaler_oracle.py``): hand-worked transforms, validation, the ``_init_args`` JSON round trip and the rank-order
combination of per-shard statistics."""
import json

import numpy as np
import pytest
import torch

from replay_cql_b200 import scalers
from replay_cql_b200.models import CQL
from tests import scaler_oracle as S

f32 = np.float32


def test_hand_worked_transforms():
    obs_mm = {"type": "min_max", "minimum": [2.0, 10.0], "maximum": [6.0, 30.0]}
    obs_sd = {"type": "standard", "mean": [1.0, 2.0], "std": [0.999, 4.999]}
    act_mm = {"type": "min_max", "minimum": [1.0], "maximum": [5.0]}
    rew_mm = {"type": "min_max", "minimum": [0.0], "maximum": [4.0]}
    rew_sd = {"type": "standard", "mean": [0.5], "std": [0.499]}
    x = torch.tensor([[4.0, 20.0], [2.0, 30.0]])
    assert S.obs_fwd(obs_mm, x).tolist() == [[0.5, 0.5], [0.0, 1.0]]
    # (x - mean) / (std + 1e-3), std + 1e-3 rounded once in float32
    want = [[(f32(4) - f32(1)) / (f32(0.999) + f32(1e-3)), (f32(20) - f32(2)) / (f32(4.999) + f32(1e-3))]]
    assert S.obs_fwd(obs_sd, x[:1]).numpy().tolist() == np.asarray(want, np.float32).tolist()
    a = torch.tensor([1.0, 3.0, 5.0, 4.0])
    assert S.act_fwd(act_mm, a).tolist() == [-1.0, 0.0, 1.0, 0.5]
    assert S.act_rev(act_mm, S.act_fwd(act_mm, a)).tolist() == a.tolist()
    assert S.act_rev(act_mm, torch.tensor([-1.0, 1.0, 0.0])).tolist() == [1.0, 5.0, 3.0]
    assert S.rew_fwd(rew_mm, torch.tensor([0.0, 1.0, 4.0])).tolist() == [0.0, 0.25, 1.0]
    assert S.rew_fwd(rew_sd, torch.tensor([0.5, 1.0])).tolist() == [0.0, 1.0]
    # a table row: s, a, r and s' transformed -- a terminal row's s' = (0, 0) too; term and discount untouched
    rows = np.array([[4, 20, 3, 1, 0, 0, 1, 0.5], [2, 10, 5, 0, 6, 30, 0, 0.25]], np.float32)
    t = S.transform_rows({"scaler": obs_mm, "action_scaler": act_mm, "reward_scaler": rew_mm}, rows)
    assert t.tolist() == [[0.5, 0.5, 0.0, 0.25, -0.5, -0.5, 1.0, 0.5], [0.0, 0.0, 1.0, 0.0, 1.0, 1.0, 0.0, 0.25]]
    assert np.array_equal(S.transform_rows({}, rows), rows)


def test_fit_matches_oracle_and_hand_values():
    obs = np.array([[0, 5], [0, 7], [1, 5], [2, 9]], np.float32)
    act = np.array([1, 2, 3, 4], np.float32)
    rew = np.array([0, 1, 0, 1], np.float32)
    term = np.array([0, 1, 0, 1], np.float32)
    o = S.fit(obs, act, rew, term)
    assert o["min"].tolist() == [0, 5, 1, 0] and o["max"].tolist() == [2, 9, 4, 1]
    assert o["mean"].tolist() == [0.75, 6.5, 2.5, 0.5]
    assert np.allclose(o["std"], np.sqrt([0.6875, 2.75, 1.25, 0.25]), rtol=1e-15)
    stats = {"count": np.full(4, 4), "min": o["min"], "max": o["max"], "mean": o["mean"],
             "m2": o["std"] ** 2 * 4, "rew_available": True}
    for arg, cols in scalers.COLUMNS.items():
        for kind in scalers.KINDS[arg]:
            assert scalers.params_from_stats(arg, kind, stats) == S.params(kind, cols, o)


def test_validation():
    for arg, bad in [("scaler", "pixel"), ("scaler", "clip"), ("reward_scaler", "multiply"), ("action_scaler", "standard"),
                     ("scaler", {"type": "min_max", "minimum": [0.0, 0.0], "maximum": [1.0, 0.0]}),
                     ("scaler", {"type": "standard", "mean": [0.0], "std": [1.0]}),
                     ("action_scaler", {"type": "min_max", "minimum": [1.0]}),
                     ("reward_scaler", {"type": "standard", "mean": [0.0], "std": [-1.0]}),
                     ("scaler", 3)]:
        with pytest.raises(ValueError):
            scalers.validate(arg, bad)
        with pytest.raises(ValueError):
            CQL(**{arg: bad})
    stats = {"count": np.full(4, 3), "min": np.array([0.0, 4.0, 1.0, 0.0]), "max": np.array([5.0, 4.0, 5.0, 0.0]),
             "mean": np.zeros(4), "m2": np.ones(4), "rew_available": True}
    with pytest.raises(ValueError, match="obs.y"):
        scalers.params_from_stats("scaler", "min_max", stats)          # a constant item column
    with pytest.raises(ValueError, match="rew"):
        scalers.params_from_stats("reward_scaler", "min_max", stats)
    assert scalers.params_from_stats("reward_scaler", "standard", stats)["std"] == [float(f32(np.sqrt(1 / 3)))]
    with pytest.raises(ValueError, match="unavailable"):
        scalers.params_from_stats("reward_scaler", "standard", dict(stats, rew_available=False))
    with pytest.raises(ValueError, match="soft_q_backup"):
        CQL(soft_q_backup=True, scaler="standard")


@pytest.mark.parametrize("spec", [
    dict(scaler="min_max", action_scaler="min_max", reward_scaler="standard"),
    dict(scaler="standard", action_scaler=None, reward_scaler="min_max"),
    dict(scaler={"type": "standard", "mean": [3000.5, 1800.25], "std": [1700.0, 1000.0]},
         action_scaler={"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
         reward_scaler={"type": "min_max", "minimum": 0.0, "maximum": [1.0]}),
])
def test_init_args_json_round_trip(spec):
    m = CQL(**spec)
    args = json.loads(json.dumps(m._init_args))
    for k in ("scaler", "action_scaler", "reward_scaler"):
        assert args[k] == getattr(m, k)
    again = CQL(**args)
    assert again._init_args == m._init_args
    p = scalers.from_struct(scalers.to_struct({k: v for k, v in args.items() if isinstance(v, dict)}))
    for k in ("scaler", "action_scaler", "reward_scaler"):
        assert p[k] == (args[k] if isinstance(args[k], dict) else None)


def _stats_of(obs, act, rew):
    cols = [obs[:, 0], obs[:, 1], act, rew]
    x = [np.asarray(c, np.float64) for c in cols]
    return {"count": np.array([v.size for v in x]), "min": np.array([v.min() for v in x]),
            "max": np.array([v.max() for v in x]), "mean": np.array([v.mean() for v in x]),
            "m2": np.array([np.sum((v - v.mean()) ** 2) for v in x]), "rew_available": True}


@pytest.mark.parametrize("seed", range(5))
def test_shard_combination_equals_whole_log(seed):
    """Per-shard statistics of a random split by user, combined in rank order, equal the whole log's within 1e-12."""
    rng = np.random.default_rng(seed)
    n = 5000
    users = np.sort(rng.integers(0, 300, n))
    obs = np.stack([users, rng.integers(0, 3706, n)], 1).astype(np.float32)
    act = (rng.integers(1, 6, n) + 1e-3 * rng.standard_normal(n)).astype(np.float32)
    rew = rng.integers(0, 2, n).astype(np.float32)
    cuts = np.sort(rng.choice(np.arange(1, 300), size=int(rng.integers(1, 6)), replace=False))
    bounds = [0] + [int(np.searchsorted(users, c)) for c in cuts] + [n]
    parts = [_stats_of(obs[a:b], act[a:b], rew[a:b]) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
    got, want = scalers.combine(parts), _stats_of(obs, act, rew)
    assert np.array_equal(got["count"], want["count"])
    assert np.array_equal(got["min"], want["min"]) and np.array_equal(got["max"], want["max"])
    assert np.allclose(got["mean"], want["mean"], rtol=1e-12, atol=0)
    assert np.allclose(got["m2"], want["m2"], rtol=1e-12, atol=0)
    back = scalers.stats_from_array(scalers.stats_to_array(got))
    assert all(np.array_equal(back[k], got[k]) for k in scalers.STAT_KEYS) and back["rew_available"]
