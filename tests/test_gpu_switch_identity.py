"""The update schedule's A/B switches that change only how the launches are made leave the results bit-identical.

CQL_NO_FOLD=1 puts the separate gradient-reduction launches back in place of k_adam_pack summing the backward's partials
(the same additions in the same order, DESIGN.md section 3); CQL_NO_PDL=1 launches every kernel without programmatic
dependent launch.  The switches are read once per process, so every arm runs in a fresh one: same seed, same synthetic
table, 20 sampled updates in f16x3 at batch 1024.  The learner state, both Adam moments and the metrics must be equal
bit for bit across the arms.
"""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

CHILD = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from replay_cql_b200.engine import CqlEngine, CqlHyperParams
eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=777, precision="f16x3"), device=0)
eng.synth_table(1_000_003, 6040, 3706, seed=777)
eng.update(20, want_metrics=False)
m, v, step = eng.get_optimizer()
np.savez(sys.argv[2], state=eng.get_state(), adam_m=m, adam_v=v, step=np.int64(step),
         metrics=np.array(list(eng.read_metrics().values()), dtype=np.float32))
eng.close()
"""

ARMS = {"default": {}, "no_fold": {"CQL_NO_FOLD": "1"}, "no_pdl": {"CQL_NO_PDL": "1"}}


def test_switches_leave_the_update_bit_identical(tmp_path):
    out = {}
    for arm, extra in ARMS.items():
        env = {k: v for k, v in os.environ.items() if not k.startswith("CQL_")}
        env.update(extra)
        path = tmp_path / f"{arm}.npz"
        p = subprocess.run([sys.executable, "-c", CHILD, str(ROOT), str(path)], cwd=ROOT, env=env, capture_output=True,
                           text=True, timeout=600)
        assert p.returncode == 0, f"{arm}:\n{p.stdout}\n{p.stderr}"
        out[arm] = np.load(path)
    ref = out["default"]
    assert int(ref["step"]) == 20
    for arm in ("no_fold", "no_pdl"):
        for key in ref.files:
            assert np.array_equal(ref[key], out[arm][key]), f"{arm}: {key} differs from the default schedule"
