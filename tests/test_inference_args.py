"""CPU: argument checks of the per-observation inference calls (``predict_value``, ``predict_action``,
``sample_action``), their C ABI declarations and the sampling key -- no GPU needed."""
import re
from pathlib import Path

import numpy as np
import pytest

from replay_cql_b200 import _lib
from replay_cql_b200.engine import inference_inputs
from replay_cql_b200.models import CQL
from tests import sampling_oracle as SO

ROOT = Path(__file__).resolve().parent.parent
SAMPLE_SEED_XOR = 0xE7037ED1A0B428DB


def test_valid_inputs_are_converted():
    u, i, a = inference_inputs(np.array([0, 5, 2 ** 24 - 1], dtype=np.int64), [[1], [2], [3]], [1.5, 2, 3])
    assert u.dtype == i.dtype == np.int32 and a.dtype == np.float32
    assert u.flags.c_contiguous and i.flags.c_contiguous and a.flags.c_contiguous
    assert u.tolist() == [0, 5, 2 ** 24 - 1] and i.tolist() == [1, 2, 3] and a.tolist() == [1.5, 2.0, 3.0]
    u, i, a = inference_inputs(np.arange(4, dtype=np.uint16), np.arange(8, dtype=np.int32)[::2])
    assert a is None and i.tolist() == [0, 2, 4, 6]
    u, i, a = inference_inputs([], [], [])
    assert u.size == i.size == a.size == 0


@pytest.mark.parametrize("users,items", [
    ([1, 2], [1]),                                  # lengths differ
    ([-1], [0]),                                    # negative id
    ([0], [2 ** 24]),                               # not exact in float32
    (np.array([2 ** 32 + 1], dtype=np.int64), [0]), # would wrap to 1 as int32
    ([0.5], [1]),                                   # not an id
    ([True], [1]),
    (np.zeros((2, 2), dtype=np.int32), [1, 2]),     # not a column
])
def test_bad_ids_are_rejected(users, items):
    with pytest.raises(ValueError):
        inference_inputs(users, items)
    with pytest.raises(ValueError):
        inference_inputs(items, users)


@pytest.mark.parametrize("actions", [[1.0, np.nan], [np.inf, 1.0], [1.0], [1.0, 2.0, 3.0], [[1.0, 2.0], [3.0, 4.0]],
                                     [1e39, 1.0], ["a", "b"]])
def test_bad_actions_are_rejected(actions):
    with pytest.raises(ValueError):
        inference_inputs([0, 1], [2, 3], actions)


def test_public_calls_check_arguments_before_the_engine():
    m = CQL()
    with pytest.raises(ValueError):
        m.predict_value([0, 1], [2], None)
    with pytest.raises(ValueError):
        m.predict_value([0], [2], [np.nan])
    with pytest.raises(ValueError):
        m.predict_action([2 ** 24], [0])
    with pytest.raises(ValueError):
        m.sample_action([0], [-3])
    for call in (lambda: m.predict_value([0], [1]), lambda: m.predict_action([0], [1]), lambda: m.sample_action([0], [1])):
        with pytest.raises(AttributeError, match="not fitted"):
            call()


def _declaration(name):
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "cql_b200.h").read_text(), flags=re.S)
    m = re.search(name + r"\s*\(([^)]*)\)", text)
    assert m, name
    return [p.strip() for p in m.group(1).split(",")]


@pytest.mark.parametrize("name,n_args", [("cql_predict_value", 8), ("cql_sample_action", 7)])
def test_abi_declarations_match_the_binding(name, n_args):
    params = _declaration(name)
    assert len(params) == n_args and params[0].startswith("cql_handle*") and params[-1] == "void* stream"
    res, args = _lib.SIGNATURES[name]
    assert len(args) == n_args
    assert "int64_t n" in params and args[params.index("int64_t n")] is _lib.C.c_int64


def test_sampling_key_is_its_own():
    """cql_sample_action's Philox key differs from the update noise's and the MDP builder's, and the library, the header
    and the tests agree on it"""
    assert SAMPLE_SEED_XOR not in (SO.NOISE_SEED_XOR, SO.MDP_SEED_XOR)
    src = (ROOT / "replay_cql_b200" / "csrc" / "infer.cuh").read_text()
    assert re.search(r"INF_SEED_XOR\s*=\s*0x([0-9A-Fa-f]+)ull", src).group(1).upper() == f"{SAMPLE_SEED_XOR:016X}"
    assert f"0x{SAMPLE_SEED_XOR:016X}" in (ROOT / "include" / "cql_b200.h").read_text()


def test_sampling_reference_is_standard_normal():
    """the host reference of the sampling noise: seed ^ key, stream = call number, index = row"""
    seed = 12345
    r = SO.philox4x32_10(seed ^ SAMPLE_SEED_XOR, 0, np.arange(200_000))
    eps = SO.box_muller(r[0], r[1])
    assert abs(eps.mean()) < 0.01 and abs(eps.std() - 1.0) < 0.01
    r1 = SO.philox4x32_10(seed ^ SAMPLE_SEED_XOR, 1, np.arange(200_000))
    assert abs(np.corrcoef(eps, SO.box_muller(r1[0], r1[1]))[0, 1]) < 0.01       # the next call is a new stream
    ru = SO.philox4x32_10(seed ^ SO.NOISE_SEED_XOR, 0, np.arange(200_000))
    assert abs(np.corrcoef(eps, SO.box_muller(ru[0], ru[1]))[0, 1]) < 0.01       # not the first update's noise
