"""Throughput of the per-observation inference calls against the pair scorer on an ML-20M-shaped model, with the
card's name and power limit read in the same run.

    python profiles/inference_bench.py [--pairs N] [--reps R] [--out FILE]

One f16x3 engine (n_critics 2, PyTorch-default initial weights) scores N random (user, item) pairs with user ids below
138 493 and item ids below 26 744 through
  - ``predict_value`` (tensor-core forward kernels, ``cql_predict_value``), without and with ``with_std``;
  - ``score_pairs(mode="q")`` (``k_score_pairs``, the FP32 CUDA-core pair scorer behind ``predict_pairs``);
  - ``sample_action`` (actor forward + Philox head).
Every call goes host arrays in, host arrays out and synchronises, so a host clock around it is the whole call: argument
checks, copies and kernels.  After one warm-up call of each, the calls alternate for R rounds; the median per call is
reported as pairs/s.  The greedy ``predict_value`` and ``score_pairs`` results of the measured pairs are compared
(max |difference| / max(1, max |Q|)).  The JSON result line is printed; --out also writes it to FILE.
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--users", type=int, default=138_493)
    ap.add_argument("--items", type=int, default=26_744)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the result to this JSON file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inference_bench needs a GPU")
    res = {"card": card(), "pairs": a.pairs, "users": a.users, "items": a.items, "reps": a.reps,
           "precision": "f16x3", "n_critics": 2}
    eng = CqlEngine(CqlHyperParams(precision="f16x3", n_critics=2))
    rng = np.random.default_rng(0)
    u = rng.integers(0, a.users, a.pairs).astype(np.int32)
    i = rng.integers(0, a.items, a.pairs).astype(np.int32)
    calls = {
        "predict_value": lambda: eng.predict_value(u, i),
        "predict_value_with_std": lambda: eng.predict_value(u, i, with_std=True),
        "score_pairs": lambda: eng.score_pairs(u, i, mode="q"),
        "sample_action": lambda: eng.sample_action(u, i),
    }
    out = {name: f() for name, f in calls.items()}                      # warm-up: module load, pool growth
    times = {name: [] for name in calls}
    launches = {}
    for _ in range(a.reps):
        for name, f in calls.items():
            l0 = eng.launch_count
            t = time.perf_counter()
            f()
            times[name].append(time.perf_counter() - t)
            launches[name] = eng.launch_count - l0
    for name in calls:
        s = float(np.median(times[name]))
        res[name] = {"s_per_call": s, "pairs_per_s": a.pairs / s, "min_s": float(np.min(times[name])),
                     "max_s": float(np.max(times[name])), "launches_per_call": launches[name]}
    res["speedup_predict_value_over_score_pairs"] = res["score_pairs"]["s_per_call"] / res["predict_value"]["s_per_call"]
    q, ref = out["predict_value"].astype(np.float64), out["score_pairs"].astype(np.float64)
    res["greedy_vs_score_pairs_rel_diff"] = float(np.max(np.abs(q - ref)) / max(1.0, float(np.max(np.abs(ref)))))
    res["with_std_mean_bit_equal"] = bool(np.array_equal(out["predict_value_with_std"][0], out["predict_value"]))
    res["card_after"] = card()
    eng.close()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
