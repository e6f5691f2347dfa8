"""CPU restatement of one fitted-Q-evaluation update (d3rlpy's FQE).  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED ([EXT-UNVERIFIED], DESIGN.md section 1 "FQE"): restated from d3rlpy 1.x ``ope/fqe.py`` and
``ope/torch/fqe_impl.py`` (``FQEImpl.update``, ``compute_target``, ``update_target``) on top of ``oracle.cql_oracle``'s
``mlp`` / ``actor_forward`` / ``q_ensemble`` / ``adam_step``, plain eager PyTorch with autograd for the backward.  Shares
nothing with the CUDA kernels or with ``replay_cql_b200``.  Works in float32 (the parity target) and float64.

State: {"actor": net (the frozen policy), "critics": [nets], "targ": [nets], "adam": [{key: {"m", "v"}}], "step": int}.
Rows: [B, 8] table rows ``s.x s.y a r s'.x s'.y term discount`` (raw; ``prep`` applies the scalers).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import cql_oracle as O
from replay_cql_b200 import layout
from tests import scaler_oracle as S

NET_KEYS = O.NET_KEYS
ADAM = O.OracleConfig(beta1=0.9, beta2=0.999, adam_eps=1e-8)


def _t(net, dtype):
    return {k: torch.from_numpy(np.array(v, dtype=np.float32)).to(dtype) for k, v in net.items()}


def from_flat(flat, n_critics: int, m=None, v=None, step: int = 0, dtype=torch.float32) -> dict:
    """Flat product-layout state (actor slot = the policy, critic / target-critic slots = FQE's networks) and optional
    flat Adam moments -> oracle state."""
    un = layout.unpack_state(np.asarray(flat, dtype=np.float32), n_critics)
    st = {"actor": _t(un["actor"], dtype), "critics": [_t(c, dtype) for c in un["critics"]],
          "targ": [_t(c, dtype) for c in un["targ_critics"]], "step": int(step)}
    mom = {}
    for key, buf in (("m", m), ("v", v)):
        mom[key] = (layout.unpack_state(np.asarray(buf, dtype=np.float32), n_critics)["critics"] if buf is not None
                    else [{k: np.zeros_like(x) for k, x in c.items()} for c in un["critics"]])
    st["adam"] = [{k: {"m": torch.from_numpy(np.array(mom["m"][c][k])).to(dtype),
                       "v": torch.from_numpy(np.array(mom["v"][c][k])).to(dtype)} for k in NET_KEYS}
                  for c in range(n_critics)]
    return st


def cast(st: dict, dtype) -> dict:
    c = lambda net: {k: x.detach().clone().to(dtype) for k, x in net.items()}
    return {"actor": c(st["actor"]), "critics": [c(n) for n in st["critics"]], "targ": [c(n) for n in st["targ"]],
            "adam": [{k: {"m": a[k]["m"].clone().to(dtype), "v": a[k]["v"].clone().to(dtype)} for k in NET_KEYS}
                     for a in st["adam"]], "step": st["step"]}


def minibatch(rows, dtype, prep=None):
    """-> (s, a, r, s', term, discount) in the networks' coordinates."""
    prep = prep or {}
    t = torch.from_numpy(np.array(rows, dtype=np.float32))
    s = S.obs_fwd(prep.get("scaler"), t[:, 0:2]).to(dtype)
    a = S.act_fwd(prep.get("action_scaler"), t[:, 2:3]).to(dtype)
    r = S.rew_fwd(prep.get("reward_scaler"), t[:, 3]).to(dtype)
    s1 = S.obs_fwd(prep.get("scaler"), t[:, 4:6]).to(dtype)
    return s, a, r, s1, t[:, 6].to(dtype), t[:, 7].to(dtype)


def td_target(st, rows, gamma: float, nstep: bool = False, prep=None):
    """``compute_target``: y = r + gamma_k * min_c Q_targ_c(s', tanh(mu(s'))) * (1 - term), gamma_k = the row's
    discount (slot 7) for n-step rows, else gamma."""
    dtype = st["actor"]["W1"].dtype
    _, _, r, s1, term, disc = minibatch(rows, dtype, prep)
    with torch.no_grad():
        mu1, _ = O.actor_forward(st["actor"], s1)
        q_t = O.q_ensemble(st["targ"], s1, torch.tanh(mu1)).min(dim=0).values
        g = disc if nstep else torch.tensor(gamma, dtype=dtype)
        return r + g * q_t * (1 - term)


def update(st, rows, gamma: float, lr: float, interval: int, nstep: bool = False, prep=None):
    """One ``FQEImpl.update`` then d3rlpy's ``if grad_step % target_update_interval == 0: update_target()`` with
    grad_step = the updates before this one.  Mutates ``st``.  -> (loss, [per-critic gradient dicts])."""
    dtype = st["actor"]["W1"].dtype
    s, a, _, _, _, _ = minibatch(rows, dtype, prep)
    y = td_target(st, rows, gamma, nstep, prep)
    leaf = [{k: x.detach().clone().requires_grad_(True) for k, x in c.items()} for c in st["critics"]]
    loss = 0.0
    for c in leaf:                                   # ensemble compute_error: sum over critics of the mean squared error
        loss = loss + ((O.critic_forward(c, s, a)[:, 0] - y) ** 2).mean()
    flat = [c[k] for c in leaf for k in NET_KEYS]
    gs = iter(torch.autograd.grad(loss, flat))
    grads_before = st["step"]
    st["step"] += 1
    grads = []
    for ci, c in enumerate(st["critics"]):
        gd = {}
        for k in NET_KEYS:
            g = next(gs)
            gd[k] = g.clone()
            O.adam_step(c[k], g, st["adam"][ci][k], lr, st["step"], ADAM)
        grads.append(gd)
    if grads_before % interval == 0:
        st["targ"] = [{k: x.clone() for k, x in c.items()} for c in st["critics"]]
    return float(loss.detach()), grads
