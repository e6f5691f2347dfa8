"""Cost of larger critic ensembles and action-sample counts: f16x3 updates/s at batch 1024 for several (n_critics,
n_action_samples), and users scored to top-10 per second at n_critics 2 and 10, on the ML-20M shape, with the card's name
and power limit read in the same run.

    python profiles/ensemble_bench.py [--steps K] [--warmup W] [--out FILE]

The JSON result line is printed; --out also writes it to FILE.

Updates: the replay table is the on-device synthetic ML-20M table (20 000 263 rows, 138 493 users, 26 744 items); after W
warm-up updates (graph capture, module load), K sampled updates (one CUDA-graph replay) are timed with CUDA events on one
stream.  Scoring: every one of the 138 493 users against all 26 744 items, top-10, no seen filter (the scorer's work grows
with C; the filter's does not), one warm-up call on 4 096 users, then one timed call.  The score matrix (3.7 G pairs) and
the update's working set are far larger than the 126 MB L2.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np
import torch

from replay_cql_b200.engine import CqlEngine, CqlHyperParams

ROWS, USERS, ITEMS = 20_000_263, 138_493, 26_744
UPDATE_SHAPES = [(2, 10), (4, 10), (10, 10), (2, 32), (10, 32)]
SCORE_CRITICS = [2, 10]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def updates_per_s(C, n, steps, warmup):
    eng = CqlEngine(CqlHyperParams(batch_size=1024, n_critics=C, n_action_samples=n, precision="f16x3", seed=7), device=0)
    try:
        eng.synth_table(ROWS, USERS, ITEMS, seed=7)
        st = torch.cuda.Stream()
        eng.update(warmup, want_metrics=False, stream=st.cuda_stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        eng.update(steps, want_metrics=False, stream=st.cuda_stream)
        e1.record(st)
        st.synchronize()
        ms = e0.elapsed_time(e1)
        m = eng.read_metrics()
        assert all(np.isfinite(v) for v in m.values()), m
        return {"C": C, "n": n, "updates_per_s": round(steps / (ms / 1e3), 1), "us_per_update": round(ms * 1e3 / steps, 1)}
    finally:
        eng.close()


def users_per_s(C):
    eng = CqlEngine(CqlHyperParams(batch_size=1024, n_critics=C, precision="f16x3", seed=7), device=0)
    try:
        dev = torch.device("cuda", 0)
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            users = torch.arange(USERS, dtype=torch.int32, device=dev)
            items = torch.arange(ITEMS, dtype=torch.int32, device=dev)
            oi = torch.empty((USERS, 10), dtype=torch.int32, device=dev)
            osc = torch.empty((USERS, 10), dtype=torch.float32, device=dev)
            eng.score_topk_device(users[:4096], items, 10, out_items=oi[:4096], out_scores=osc[:4096], stream=st.cuda_stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        with torch.cuda.stream(st):
            eng.score_topk_device(users, items, 10, out_items=oi, out_scores=osc, stream=st.cuda_stream)
        e1.record(st)
        st.synchronize()
        ms = e0.elapsed_time(e1)
        return {"C": C, "users_per_s": round(USERS / (ms / 1e3), 1), "ms": round(ms, 2)}
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--out", type=str, default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_bench needs a GPU")
    res = {"card": card(), "precision": "f16x3", "batch_size": 1024,
           "table": f"synthetic ML-20M shape: {ROWS} rows, {USERS} users, {ITEMS} items",
           "update": [updates_per_s(C, n, args.steps, args.warmup) for C, n in UPDATE_SHAPES],
           "score_top10": [users_per_s(C) for C in SCORE_CRITICS]}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
