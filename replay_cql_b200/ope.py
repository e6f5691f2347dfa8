"""``FQE`` -- fitted Q evaluation of a trained ``CQL`` policy on the GPU (d3rlpy's ``d3rlpy.ope.FQE``).

Every offline scorer of a CQL model reads the model's own critics, which the conservative penalty pushes down on purpose,
so their values cannot be compared across checkpoints or hyperparameters.  FQE freezes the policy
``pi(x) = tanh(mu(x))``, trains fresh Q-networks on the logged transitions with a plain TD loss toward
``r + gamma * min_c Q_targ_c(s', pi(s')) * (1 - term)`` and reads the policy's value from them with the same scorers.
Semantics: DESIGN.md section 1, "FQE".
"""
from __future__ import annotations

import math
from typing import Any, Dict, Optional

import numpy as np

from . import _lib, layout
from .engine import PRECISIONS, CqlEngine, CqlHyperParams
from .mdp import build_mdp_on_device
from .models import evaluate_offline
from .parallel import dist_info


def _is_int(x) -> bool:
    return isinstance(x, (int, np.integer)) and not isinstance(x, bool)


class FQE:
    """Fitted Q evaluation of ``algo``'s policy.

    ``n_critics`` (1..10) fresh Q-networks ``(obs, act) -> q`` with PyTorch's default initialisation under ``seed``
    (``layout.init_state``) and hard-copied targets.  One update on a minibatch of ``batch_size`` logged transitions
    minimises ``sum_c mean_b (Q_c(s, a) - y)^2`` with Adam (``learning_rate``, betas (0.9, 0.999), eps 1e-8); the target
    becomes a copy of the critics after updates 1, 1 + I, 1 + 2I, ... (``I = target_update_interval``).  ``n_steps``
    (1..64) is the n-step TD horizon of the replay rows, as in ``CQL``.  The model's fitted scalers apply.
    ``precision`` defaults to the model's.

    The policy is a snapshot of the model's actor taken here; the model itself is never modified.  In a data-parallel
    job every rank trains the same replica from the same inputs.
    """

    def __init__(self, algo, n_critics: int = 1, learning_rate: float = 1e-4, batch_size: int = 100,
                 gamma: float = 0.99, n_steps: int = 1, target_update_interval: int = 100,
                 precision: Optional[str] = None, seed: int = 12345):
        if not _is_int(n_critics) or not 1 <= n_critics <= _lib.MAX_CRITICS:
            raise ValueError(f"n_critics must be an integer in 1..{_lib.MAX_CRITICS}")
        if not _is_int(batch_size) or batch_size < 1:
            raise ValueError("batch_size must be an integer >= 1")
        if not _is_int(target_update_interval) or target_update_interval < 1:
            raise ValueError("target_update_interval must be an integer >= 1")
        if not _is_int(n_steps) or not 1 <= n_steps <= _lib.MAX_N_STEPS:
            raise ValueError(f"n_steps (the n-step TD horizon) must be an integer in 1..{_lib.MAX_N_STEPS}")
        if isinstance(learning_rate, bool) or not isinstance(learning_rate, (int, float, np.integer, np.floating)) \
                or not math.isfinite(float(learning_rate)) or float(learning_rate) <= 0:
            raise ValueError("learning_rate must be a finite number > 0")
        if precision is not None and precision not in PRECISIONS:
            raise ValueError(f"precision must be None or one of {sorted(PRECISIONS)}")
        model = getattr(algo, "engine", None)
        if model is None:
            raise AttributeError("CQL model is not fitted or loaded")
        self.algo = algo
        self.n_critics, self.learning_rate, self.batch_size = int(n_critics), float(learning_rate), int(batch_size)
        self.gamma, self.n_steps, self.target_update_interval = float(gamma), int(n_steps), int(target_update_interval)
        self.precision = precision if precision is not None else model.hp.precision
        self.seed = int(seed)
        self.last_loss: Optional[float] = None
        hp = CqlHyperParams(batch_size=self.batch_size, n_critics=self.n_critics, n_action_samples=1, gamma=self.gamma,
                            critic_lr=self.learning_rate, beta1=0.9, beta2=0.999, adam_eps=1e-8,
                            precision=self.precision, squash=model.hp.squash, seed=self.seed, n_steps=self.n_steps)
        self.engine = CqlEngine(hp, device=model.device, rank=0, world_size=1)
        try:
            state = layout.init_state(self.n_critics, self.seed)           # FQE's critics, targets equal to them
            policy = model.get_state()[:layout.NET_STRIDE]                   # the model's actor slot (slot 0)
            state[:layout.NET_STRIDE] = policy
            ta = layout.slot_targ_actor(self.n_critics) * layout.NET_STRIDE
            state[ta:ta + layout.NET_STRIDE] = policy
            self.engine.set_state(state)
            prep = model.get_preprocessing()
            if any(v is not None for v in prep.values()):
                self.engine.set_preprocessing(**prep)
            self.engine.fqe_enable(self.target_update_interval)
        except BaseException:
            self.engine.close()
            raise

    def _load_table(self, log: Any) -> None:
        eng, model = self.engine, self.algo.engine
        if log is not None:
            n_log = int(log.num_rows) if hasattr(log, "num_rows") else len(log)
            if n_log == 0:
                raise ValueError("FQE.fit: empty log")
            # Built on a small builder engine: the model's seed draws the action noise (FQE trains on the rows the model's
            # fit built from this log), FQE's gamma and n_steps form the n-step returns and discounts.  Only the seed,
            # gamma and n_steps of a handle reach the builder, so it has the smallest shape the library accepts.
            hp = CqlHyperParams(batch_size=1, n_critics=1, n_action_samples=1, precision="fp32", gamma=self.gamma,
                                seed=model.hp.seed, n_steps=self.n_steps)
            tmp = CqlEngine(hp, device=model.device)
            try:
                build_mdp_on_device(tmp, log, top_k=self.algo.top_k,
                                    action_randomization_scale=self.algo.action_randomization_scale)
                eng.copy_table_from(tmp)
            finally:
                tmp.close()
            return
        if eng.n_transitions > 0:                      # a later fit continues on the table of the first
            return
        _, world, _ = dist_info()
        if model.n_transitions == 0:
            raise ValueError("FQE.fit: the model holds no replay table (e.g. loaded from a checkpoint saved without "
                             "save_replay_table) -- pass the log")
        if model.hp.n_steps != self.n_steps:
            raise ValueError(f"FQE.fit: the model's replay table holds n_steps={model.hp.n_steps} rows, FQE uses "
                             f"n_steps={self.n_steps} -- pass the log")
        if self.n_steps > 1 and np.float32(model.hp.gamma) != np.float32(self.gamma):
            raise ValueError(f"FQE.fit: the model's n-step replay table was discounted with gamma={model.hp.gamma}, FQE "
                             f"uses gamma={self.gamma} -- pass the log")
        if world > 1 and getattr(self.algo, "_table_sharded", False):
            raise ValueError("FQE.fit: the model's replay table is sharded over the ranks of this data-parallel job -- "
                             "pass the log")
        eng.copy_table_from(model)

    def fit(self, log: Any = None, n_steps: Optional[int] = None, n_epochs: Optional[int] = None,
            n_steps_per_epoch: Optional[int] = None) -> "FQE":
        """Train the FQE critics: ``n_steps`` updates, else ``n_epochs`` (default 1) epochs of ``n_steps_per_epoch``
        (default: table rows // batch_size) updates.  ``log=None`` trains on a device copy of the model's replay table
        (its ``n_steps`` must be FQE's and, for n-step rows, its ``gamma`` too: the discounts are part of the rows); a
        ``log`` (anything ``CQL.fit`` accepts) is built into FQE's own table by the same MDP builder with the model's
        seed and FQE's ``gamma`` and ``n_steps``.  Repeated calls
        continue exactly: ``fit(n_steps=N); fit(n_steps=M)`` equals ``fit(n_steps=N + M)``."""
        for name, v in (("n_steps", n_steps), ("n_epochs", n_epochs), ("n_steps_per_epoch", n_steps_per_epoch)):
            if v is not None and (not _is_int(v) or v < 0):
                raise ValueError(f"{name} must be an integer >= 0 or None")
        self._load_table(log)
        per_epoch = n_steps_per_epoch if n_steps_per_epoch is not None else self.engine.n_transitions // self.batch_size
        total = int(n_steps) if n_steps is not None else int(n_epochs if n_epochs is not None else 1) * int(per_epoch)
        if total > 0:
            self.last_loss = self.engine.fqe_update(total)
        return self

    def predict_value(self, users, items, actions=None, with_std: bool = False):
        """d3rlpy's ``FQE.predict_value(x, action, with_std)`` on the FQE critics for the pairs
        ``x = (users[i], items[i])``, float32: ``mean_c Q_fqe_c(x, a)`` and, with ``with_std``, ``(mean, std)`` with the
        population std over the FQE critics.  ``actions`` are in rating units (the model's action scaler applies); None
        evaluates the policy's own greedy action ``pi(x)``.  The two-argument call runs on the pair scorer
        (``score_pairs``), as it always has; explicit actions or ``with_std`` run on the forward kernels
        (``CQL.predict_value``), which agree with it within the 1e-5 Q-score gate.  Every rank of a data-parallel job computes its
        own inputs locally, with no collective."""
        if actions is None and not with_std:
            return self.engine.score_pairs(users, items, mode="q")
        return self.engine.predict_value(users, items, actions, with_std=with_std)

    def offline_metrics(self, log: Any = None, return_threshold: Optional[float] = None) -> Dict[str, float]:
        """d3rlpy's offline scorers on the FQE critics (same keys as ``CQL.offline_metrics``):
        ``initial_state_value_estimation`` and ``soft_opc`` are FQE's estimates of the policy's value.  ``log=None``
        evaluates FQE's own replay table (one-step rows only)."""
        return evaluate_offline(self.engine, log, return_threshold, self.algo.top_k,
                                self.algo.action_randomization_scale, False, mdp_seed=self.algo.engine.hp.seed)

    def close(self) -> None:
        if getattr(self, "engine", None) is not None:
            self.engine.close()
            self.engine = None
