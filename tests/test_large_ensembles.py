"""CPU: the ensemble limits of the public interface (n_critics 1..MAX_CRITICS = 10, n_action_samples
1..MAX_ACTION_SAMPLES = 32) and the oracle's second witness at the largest values."""
import json

import pytest

from oracle import cql_oracle as O
from replay_cql_b200 import _lib
from replay_cql_b200.engine import CqlHyperParams
from replay_cql_b200.models import CQL
from tests import test_oracle_second_witness as W


def test_limits_match_the_header():
    text = (W.__file__.rsplit("/tests/", 1)[0] + "/include/cql_b200.h")
    with open(text) as f:
        header = f.read()
    assert f"#define CQL_MAX_CRITICS {_lib.MAX_CRITICS} " in header
    assert f"#define CQL_MAX_ACTION_SAMPLES {_lib.MAX_ACTION_SAMPLES} " in header
    assert (_lib.MAX_CRITICS, _lib.MAX_ACTION_SAMPLES) == (10, 32)


@pytest.mark.parametrize("kw", [dict(n_critics=11), dict(n_critics=0), dict(n_action_samples=33),
                                dict(n_action_samples=0), dict(n_critics=2.5), dict(n_action_samples=-1)])
def test_out_of_range_ensembles_raise_at_construction(kw):
    with pytest.raises(ValueError, match="n_critics|n_action_samples"):
        CQL(**kw)
    with pytest.raises(ValueError, match="n_critics|n_action_samples"):
        CqlHyperParams(**kw)


@pytest.mark.parametrize("C,n", [(1, 1), (5, 11), (10, 32)])
def test_in_range_ensembles_construct(C, n):
    m = CQL(n_critics=C, n_action_samples=n)
    assert (m.n_critics, m.n_action_samples) == (C, n)
    hp = m._hyper_params()
    assert (hp.n_critics, hp.n_action_samples) == (C, n)


def test_largest_ensemble_round_trips_init_args_through_json():
    m = CQL(n_critics=10, n_action_samples=32, batch_size=256, seed=3)
    args = json.loads(json.dumps(m._init_args))
    assert args["n_critics"] == 10 and args["n_action_samples"] == 32
    assert CQL(**args)._init_args == m._init_args


def test_search_space_keeps_its_critic_range():
    """optimize() samples n_critics from 2..4 as before: the wider range is for users who ask for it."""
    assert CQL._search_space["n_critics"] == {"type": "int", "args": [2, 4]}


def test_one_update_equals_module_based_restatement_at_largest_ensemble(monkeypatch):
    """The module-based restatement of test_oracle_second_witness (nn.Linear critics, torch.distributions, torch.logsumexp
    over the 3n samples, torch.optim.Adam over all critics) at C = 10 and n = 32."""
    base = O.OracleConfig
    monkeypatch.setattr(O, "OracleConfig", lambda: base(n_critics=10, n_action_samples=32))
    assert O.OracleConfig().n_critics == 10 and O.OracleConfig().n_action_samples == 32
    W.test_one_update_equals_module_based_restatement()
