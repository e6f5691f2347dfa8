"""CPU restatement of n-step replay rows and of the n-step TD target.  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED ([EXT-UNVERIFIED], DESIGN.md section 1): restated from d3rlpy 1.x, where a minibatch row carries the
n-step reward sum, the next observation and terminal flag of the step k steps later, and the critic loss uses
``gamma ** k`` (``ddpg_impl.compute_critic_loss``).  Written as slow per-episode Python loops; shares nothing with the
CUDA expansion kernel.  The update itself is ``oracle.cql_oracle.update`` unchanged: its only use of ``cfg.gamma`` is
the TD target ``y = r + gamma * q_targ * (1 - done)``, so a per-row discount [B, 1] in place of the scalar gamma
(:func:`discount_config`) is the n-step target.
"""
from __future__ import annotations

import dataclasses

import numpy as np


def n_step_transitions(obs, act, rew, term, n_steps: int, gamma: float) -> np.ndarray:
    """Episode-ordered one-step steps -> [n, 8] float32 n-step rows ``(s.x, s.y, a, R, s'.x, s'.y, term, discount)``.

    An episode is a run of steps ending at a terminal step or at the end of the input.  For step t with
    k = min(n_steps, steps from t to its episode's end, t included): R = sum_{j<k} gamma^j r[t+j] and
    discount = gamma^k, accumulated in float64 in the order ``R = R + g*r[t+j]; g = g*gamma`` (gamma = the float64
    value of the float32 ``gamma``), stored as float32; s' / term are those of step t+k-1 (its next step's
    observation, zeros when it is terminal or the last step).
    """
    obs = np.asarray(obs, dtype=np.float32).reshape(-1, 2)
    act, rew, term = (np.asarray(x, dtype=np.float32).reshape(-1) for x in (act, rew, term))
    n = obs.shape[0]
    g32 = float(np.float32(gamma))
    episodes, start = [], 0
    for i in range(n):
        if term[i] != 0 or i == n - 1:
            episodes.append((start, i + 1))
            start = i + 1
    out = np.zeros((n, 8), dtype=np.float32)
    for lo, hi in episodes:
        for t in range(lo, hi):
            k = min(n_steps, hi - t)
            R, g = 0.0, 1.0
            for j in range(k):
                R = R + g * float(rew[t + j])
                g = g * g32
            last = t + k - 1
            ends = term[last] != 0 or last == n - 1
            nx = (0.0, 0.0) if ends else (float(obs[last + 1, 0]), float(obs[last + 1, 1]))
            out[t] = (obs[t, 0], obs[t, 1], act[t], R, nx[0], nx[1], term[last], g)
    return out


def discount_config(cfg, discount):
    """``cfg`` whose TD discount is the per-row tensor ``discount`` [B, 1] (n-step rows: rew is the n-step return,
    next_obs / term those of the window's last step) -- the oracle update's TD target with each row's own gamma^k."""
    return dataclasses.replace(cfg, gamma=discount)
