"""CPU restatement of d3rlpy's offline scorers.  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED ([EXT-UNVERIFIED], DESIGN.md section 1): restated from d3rlpy 1.x ``metrics/scorer.py``
(``td_error_scorer``, ``discounted_sum_of_advantage_scorer``, ``average_value_estimation_scorer``,
``value_estimation_std_scorer``, ``initial_state_value_estimation_scorer``, ``soft_opc_scorer``,
``continuous_action_diff_scorer``) as per-episode loops over d3rlpy's 1024-transition windows (``_make_batches``): the
networks run as float32 torch ops (``oracle.cql_oracle``), every s' gets its own forward, the advantage recursion runs
backwards in Python floats inside each window, and the sums are float64.  Shares nothing with the CUDA kernels or with
``replay_cql_b200``.  Returns the SUMS and counts ``cql_offline_eval`` returns (``replay_cql_b200.engine.OFFLINE_SUM_KEYS``).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import cql_oracle as O
from tests import scaler_oracle as S

WINDOW = 1024


def episodes(term):
    """[(first, last + 1)] of every episode: it ends at a terminal row or at the end of the table."""
    out, start, n = [], 0, len(term)
    for i in range(n):
        if term[i] != 0 or i == n - 1:
            out.append((start, i + 1))
            start = i + 1
    return out


def evaluate(st, rows, gamma: float, prep: dict | None = None, return_threshold: float | None = None) -> dict:
    """Oracle state ``st`` (float32), one-step table rows [n, 8] -> float64 sums and int counts."""
    prep = prep or {}
    rows = np.asarray(rows, dtype=np.float32)
    g32 = torch.tensor(np.float32(gamma))
    g64 = float(np.float32(gamma))
    thr = None if return_threshold is None else float(np.float32(return_threshold))
    s = dict(td_error=0.0, discounted_advantage=0.0, value=0.0, value_std=0.0, initial_value=0.0, action_diff=0.0,
             success_q=0.0, all_q=0.0, n_rows=0, n_episodes=0, n_success_rows=0)
    with torch.no_grad():
        for a, b in episodes(rows[:, 6]):
            ret = 0.0
            for i in range(a, b):
                ret += float(rows[i, 3])
            success = thr is not None and ret >= thr
            for w0 in range(a, b, WINDOW):
                t = torch.from_numpy(rows[w0:min(b, w0 + WINDOW)].copy())
                obs = S.obs_fwd(prep.get("scaler"), t[:, 0:2])
                nobs = S.obs_fwd(prep.get("scaler"), t[:, 4:6])
                act = S.act_fwd(prep.get("action_scaler"), t[:, 2:3])
                rew = S.rew_fwd(prep.get("reward_scaler"), t[:, 3])
                q = O.predict_value(st, obs, act)
                pi = O.predict_action(st, obs)
                qs = O.q_ensemble(st["critics"], obs, pi)
                v = qs.mean(dim=0)
                sig = qs.std(dim=0, unbiased=False)
                vn = O.predict_value(st, nobs, O.predict_action(st, nobs))
                y = rew + g32 * vn * (1.0 - t[:, 6])
                td = (q - y) ** 2
                cad = (t[:, 2] - S.act_rev(prep.get("action_scaler"), pi)[:, 0]) ** 2
                adv = (q - v).tolist()
                A = adv[-1]
                sums = [A]
                for x in reversed(adv[:-1]):
                    A = x + g64 * A
                    sums.append(A)
                if w0 == a:
                    s["initial_value"] += float(v[0])
                s["td_error"] += float(np.sum(td.numpy().astype(np.float64)))
                s["discounted_advantage"] += float(np.sum(sums))
                s["value"] += float(np.sum(v.numpy().astype(np.float64)))
                s["value_std"] += float(np.sum(sig.numpy().astype(np.float64)))
                s["action_diff"] += float(np.sum(cad.numpy().astype(np.float64)))
                qsum = float(np.sum(q.numpy().astype(np.float64)))
                s["all_q"] += qsum
                if success:
                    s["success_q"] += qsum
                    s["n_success_rows"] += len(adv)
                s["n_rows"] += len(adv)
            s["n_episodes"] += 1
    return s
