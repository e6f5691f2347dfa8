"""CPU: the vectorised MDP builder against the loop oracle; edge cases."""
import numpy as np
import pandas as pd
import pytest

from oracle import mdp_oracle
from replay_cql_b200.mdp import build_mdp, seen_csr, to_transitions
from replay_cql_b200.synthetic import make_log


def _check(log, top_k, seed=0):
    noise = np.random.default_rng(seed).standard_normal(len(log)) * 1e-3
    got = to_transitions(build_mdp(log, top_k=top_k, action_noise=noise))
    ref = mdp_oracle.build_mdp(log, top_k=top_k, action_noise=noise)
    for k in ref:
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)


@pytest.mark.parametrize("top_k", [0, 1, 3, 1000])
def test_random_log_with_ties(top_k):
    rng = np.random.default_rng(1)
    n = 500
    log = pd.DataFrame({"user_idx": rng.integers(0, 23, n), "item_idx": rng.integers(0, 50, n),
                        "timestamp": rng.integers(0, 40, n),        # many timestamp ties
                        "relevance": rng.integers(1, 6, n).astype(float)})
    _check(log, top_k)


def test_datetime_timestamps_and_shuffled_rows():
    log = make_log("tiny").sample(frac=1.0, random_state=3).reset_index(drop=True)
    log["timestamp"] = pd.to_datetime(log["timestamp"], unit="s")
    _check(log, 10)


def test_single_row_and_single_user():
    _check(pd.DataFrame({"user_idx": [7], "item_idx": [3], "timestamp": [1], "relevance": [5.0]}), 1)
    _check(pd.DataFrame({"user_idx": [2] * 5, "item_idx": [1, 2, 3, 4, 5], "timestamp": [5, 4, 3, 2, 1],
                         "relevance": [1.0, 5.0, 5.0, 2.0, 3.0]}), 2)


def test_empty_log():
    m = build_mdp(pd.DataFrame({"user_idx": [], "item_idx": [], "timestamp": [], "relevance": []}))
    assert len(m) == 0 and m.obs.shape == (0, 2)


def test_rejects_indices_not_exact_in_float32():
    with pytest.raises(ValueError):
        build_mdp(pd.DataFrame({"user_idx": [2 ** 24], "item_idx": [0], "timestamp": [0], "relevance": [1.0]}))
    with pytest.raises(ValueError):
        build_mdp(pd.DataFrame({"user_idx": [1], "item_idx": [0]}))


def test_seen_csr_sorted_unique():
    log = pd.DataFrame({"user_idx": [3, 1, 1, 3, 3], "item_idx": [9, 4, 4, 2, 9]})
    indptr, items = seen_csr(log, 5)
    assert indptr.tolist() == [0, 0, 1, 1, 3, 3]
    assert items.tolist() == [4, 2, 9]


def test_float_timestamps_with_ties():
    """Tied float timestamps are one key: the rank order breaks the tie by input order, as the oracle does."""
    rng = np.random.default_rng(0)
    n = 400
    log = pd.DataFrame({"user_idx": rng.integers(0, 7, n), "item_idx": rng.integers(0, 50, n),
                        "timestamp": rng.integers(-10, 10, n) * 0.5, "relevance": rng.integers(1, 4, n).astype(float)})
    for top_k in (1, 3):
        _check(log, top_k)
    log["timestamp"] = log["timestamp"].astype(np.float32)
    log.loc[::7, "timestamp"] = -0.0                       # -0.0 and +0.0 are one timestamp
    _check(log, 3)


def test_float_timestamp_key_preserves_order_and_ties():
    from replay_cql_b200.frames import timestamps_to_int64
    x = np.array([-np.inf, -1e300, -2.0, -1.0, -0.5, -5e-324, -0.0, 0.0, 5e-324, 0.5, 0.9, 1.0, 1e300, np.inf])
    k = timestamps_to_int64(x)
    assert k.dtype == np.int64 and np.all(np.diff(k[:6]) > 0) and np.all(np.diff(k[7:]) > 0)
    assert k[6] == k[7] and k[5] < k[6]
    x32 = np.array([-3.5, -0.0, 0.0, 0.25, 1e30], dtype=np.float32)
    assert np.array_equal(timestamps_to_int64(x32), timestamps_to_int64(x32.astype(np.float64)))
    with pytest.raises(ValueError):
        timestamps_to_int64(np.array([0.0, np.nan]))


@pytest.mark.parametrize("top_k", [1, 3])
def test_negative_and_extreme_int64_timestamps(top_k):
    lo, hi = np.iinfo(np.int64).min, np.iinfo(np.int64).max
    rng = np.random.default_rng(2)
    n = 300
    ts = rng.choice(np.array([lo, lo + 1, lo + 2, -(2 ** 62), -1, 0, 1, 2 ** 62, hi - 1, hi], dtype=np.int64), n)
    log = pd.DataFrame({"user_idx": rng.integers(0, 9, n), "item_idx": rng.integers(0, 40, n), "timestamp": ts,
                        "relevance": rng.integers(1, 3, n).astype(float)})
    _check(log, top_k)


def test_signed_zero_relevance_ties():
    """-0.0 and +0.0 relevance rank as equal: the tie falls to timestamp desc, then input order."""
    log = pd.DataFrame({"user_idx": [4] * 6, "item_idx": [1, 2, 3, 4, 5, 6], "timestamp": [1, 1, 2, 2, 0, 3],
                        "relevance": [-0.0, 0.0, 0.0, -0.0, -0.5, -1.0]})
    for top_k in (1, 2, 3, 4):
        _check(log, top_k)
    got = build_mdp(log, top_k=3, action_noise=np.zeros(6))
    pos = {int(r): i for i, r in enumerate(got.order)}
    assert [got.rew[pos[r]] for r in range(4)] == [1.0, 0.0, 1.0, 1.0]


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_non_finite_relevance_rejected(bad):
    log = pd.DataFrame({"user_idx": [0, 0, 1], "item_idx": [1, 2, 3], "timestamp": [0, 1, 2], "relevance": [1.0, bad, 2.0]})
    with pytest.raises(ValueError, match="non-finite"):
        build_mdp(log, top_k=1)


def test_nan_timestamp_rejected():
    log = pd.DataFrame({"user_idx": [0, 0], "item_idx": [1, 2], "timestamp": [0.5, np.nan], "relevance": [1.0, 2.0]})
    with pytest.raises(ValueError, match="NaN"):
        build_mdp(log, top_k=1)


@pytest.mark.parametrize("top_k", [0, -1, -(2 ** 31)])
def test_top_k_not_positive_rewards_nothing(top_k):
    log = make_log("tiny")
    assert not build_mdp(log, top_k=top_k, seed=0).rew.any()


def test_seen_csr_drops_negative_ids_and_widens_for_large_users():
    log = pd.DataFrame({"user_idx": [2, 2, 2, 1, -1, 6, 2], "item_idx": [-1, 5, 0, -7, 3, 2 ** 31 - 1, 5]})
    indptr, items = seen_csr(log, 4)
    assert indptr.tolist() == [0, 0, 0, 2, 2, 2, 2, 3]
    assert items.tolist() == [0, 5, 2 ** 31 - 1] and items.dtype == np.int32
    indptr, items = seen_csr(pd.DataFrame({"user_idx": [0, 1], "item_idx": [-1, -2]}), 3)
    assert indptr.tolist() == [0, 0, 0, 0] and items.size == 0


def test_synthetic_shapes():
    log = make_log("tiny")
    assert len(log) == 4000 and log["user_idx"].nunique() == 64
    assert log.groupby("user_idx")["timestamp"].apply(lambda s: (np.diff(s.to_numpy()) > 0).all()).all()
