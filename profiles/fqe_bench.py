"""Throughput of fitted Q evaluation (``cql_fqe_update``, ``replay_cql_b200.ope.FQE``; DESIGN.md section 1 "FQE") on
the ML-20M synthetic replay table, with the card's name and power limit read in the same run.

    python profiles/fqe_bench.py [--rows N] [--steps K] [--fit-steps F] [--out FILE]

The JSON result line is printed; --out also writes it to FILE.

Per precision (f16x3, fp32) and batch size (100, d3rlpy FQE's default, and 1024), one critic: the FQE handle is warmed
up (graph capture, first replays), then K updates are timed with CUDA events.  ``fit_s`` is the host wall time of one
``FQE.fit(n_steps=F)`` from construction-complete to return (table copy, graph capture and F updates; default
batch size, f16x3), taken on a CQL model whose engine holds the synthetic table.  The CPU oracle (tests/fqe_oracle.py)
is timed over 20 updates at each batch size after one warm-up update (measured, not extrapolated).
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

import torch

from replay_cql_b200 import layout
from replay_cql_b200.engine import CqlEngine, CqlHyperParams


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def fqe_engine(precision, B, table_eng):
    eng = CqlEngine(CqlHyperParams(batch_size=B, n_critics=1, n_action_samples=1, precision=precision, critic_lr=1e-4))
    flat = layout.init_state(1, 12345)
    flat[:layout.NET_STRIDE] = table_eng.get_state()[:layout.NET_STRIDE]
    eng.set_state(flat)
    eng.fqe_enable(100)
    eng.copy_table_from(table_eng)
    return eng


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=20_000_263)
    ap.add_argument("--users", type=int, default=138_493)
    ap.add_argument("--items", type=int, default=26_744)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--fit-steps", type=int, default=10_000)
    ap.add_argument("--oracle-steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the result to this JSON file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fqe_bench needs a GPU")
    res = {"card": card(), "rows": a.rows, "users": a.users, "steps": a.steps, "n_critics": 1}
    model_eng = CqlEngine(CqlHyperParams(precision="f16x3"))            # the CQL model: its actor is the policy
    model_eng.synth_table(a.rows, a.users, a.items, seed=7)
    for precision in ("f16x3", "fp32"):
        for B in (100, 1024):
            eng = fqe_engine(precision, B, model_eng)
            eng.fqe_update(a.warmup)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            launches = eng.launch_count
            t0.record()
            loss = eng.fqe_update(a.steps)
            t1.record()
            t1.synchronize()
            ms = t0.elapsed_time(t1)
            res[f"{precision}_B{B}"] = {"updates_per_s": a.steps / (ms * 1e-3), "us_per_update": ms * 1e3 / a.steps,
                                        "launches_per_update": (eng.launch_count - launches) / a.steps,
                                        "last_loss": loss}
            eng.close()
    from replay_cql_b200.models import CQL
    from replay_cql_b200.ope import FQE
    model = CQL(precision="f16x3")
    model.engine = model_eng
    fqe = FQE(model)
    t = time.perf_counter()
    fqe.fit(n_steps=a.fit_steps)
    res["fit"] = {"n_steps": a.fit_steps, "batch_size": fqe.batch_size, "precision": fqe.precision,
                  "fit_s": time.perf_counter() - t, "last_loss": fqe.last_loss}
    t = time.perf_counter()
    est = fqe.offline_metrics()["initial_state_value_estimation"]
    res["fit"]["offline_metrics_s"] = time.perf_counter() - t
    res["fit"]["initial_state_value_estimation"] = est
    fqe.close()
    from tests import fqe_oracle as Q
    res["cpu_oracle"] = {}
    for B in (100, 1024):
        rows = model_eng.sample_rows(B * (a.oracle_steps + 1), pos=0).cpu().numpy()
        st = Q.from_flat(layout.init_state(1, 12345), 1)
        Q.update(st, rows[:B], 0.99, 1e-4, 100)                          # warm-up, not timed
        t = time.perf_counter()
        for k in range(1, a.oracle_steps + 1):
            Q.update(st, rows[k * B:(k + 1) * B], 0.99, 1e-4, 100)
        dt = time.perf_counter() - t
        res["cpu_oracle"][f"B{B}"] = {"updates": a.oracle_steps, "s": dt, "updates_per_s (measured)": a.oracle_steps / dt,
                                      "threads": torch.get_num_threads()}
    model_eng.close()
    res["card_after"] = card()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
