"""Throughput of ``cql_offline_eval`` (d3rlpy's offline scorers, DESIGN.md section 1) on the ML-20M synthetic replay
table, with the card's name and power limit read in the same run.

    python profiles/offline_eval_bench.py [--rows N] [--reps R] [--out FILE]

The JSON result line is printed; --out also writes it to FILE.

Per precision: one warm-up call, then R calls timed with CUDA events (the call synchronises, so the span is R whole
evaluations).  FLOP are the algorithmic count -- (1 actor + 2 C critic) rows x 133 120 FLOP per table row -- over the
measured time; the update's critic-forward rate (``timed_update``: B (6 n + 2) rows x C networks per forward) is the
reference the ratio is taken against.  The CPU oracle (tests/offline_metrics_oracle.py) is timed on a 100 k-row slice of
the same table and extrapolated linearly to the whole table (labelled as such).
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np
import torch

from replay_cql_b200.engine import CqlEngine, CqlHyperParams

FLOP_PER_ROW = 133_120          # one 3-layer MLP row: 2 x (in x 256 + 256 x 256 + 256 x out) + activations


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=20_000_263)
    ap.add_argument("--users", type=int, default=138_493)
    ap.add_argument("--items", type=int, default=26_744)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-rows", type=int, default=100_000)
    ap.add_argument("--out", default=None, help="also write the result to this JSON file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("offline_eval_bench needs a GPU")
    res = {"card": card(), "rows": a.rows, "users": a.users, "reps": a.reps}
    for precision in ("f16x3", "fp32"):
        C = 2
        eng = CqlEngine(CqlHyperParams(precision=precision, n_critics=C))
        eng.synth_table(a.rows, a.users, a.items, seed=7)
        eng.offline_metrics(5.0)                                       # warm-up: module load, pool growth
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = eng.launch_count
        t0.record()
        for _ in range(a.reps):
            sums = eng.offline_metrics(5.0)
        t1.record()
        t1.synchronize()
        ms = t0.elapsed_time(t1) / a.reps
        per_call_launches = (eng.launch_count - launches) // a.reps
        fwd = [eng.timed_update()["critic_fwd"] for _ in range(5)]
        hp = eng.hp
        upd_rows = hp.batch_size * (6 * hp.n_action_samples + 2) * C
        upd_rate = upd_rows / (float(np.median(fwd)) * 1e-3)
        eval_critic_rate = a.rows * 2 * C / (ms * 1e-3)
        res[precision] = {
            "ms_per_call": ms, "rows_per_s": a.rows / (ms * 1e-3),
            "tflop_per_s": a.rows * (1 + 2 * C) * FLOP_PER_ROW / (ms * 1e-3) / 1e12,
            "critic_rows_per_s": eval_critic_rate, "update_critic_fwd_rows_per_s": upd_rate,
            "ratio_to_update_critic_fwd": eval_critic_rate / upd_rate, "launches_per_call": per_call_launches,
            "n_episodes": sums["n_episodes"],
        }
        if precision == "fp32":
            from oracle import cql_oracle as O
            from tests import helpers as Hp
            from tests import offline_metrics_oracle as OM
            idx = torch.arange(a.oracle_rows, dtype=torch.int64, device="cuda")
            rows = eng.sample_rows(a.oracle_rows, idx=idx).cpu().numpy()
            st = Hp.flat_to_oracle_state(eng.get_state(), O.OracleConfig(n_critics=C))
            t = time.perf_counter()
            OM.evaluate(st, rows, hp.gamma, return_threshold=5.0)
            dt = time.perf_counter() - t
            res["cpu_oracle"] = {"rows": a.oracle_rows, "s": dt,
                                 "extrapolated_s_for_table (not measured)": dt * a.rows / a.oracle_rows}
        eng.close()
    res["card_after"] = card()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
