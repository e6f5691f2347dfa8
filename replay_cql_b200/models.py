"""``CQL`` -- the drop-in recommender (the class a RePlay user imports as ``replay.models.CQL``).

Keeps the wrapper's public contract (SURVEY.md Appendix B, section 8b): ``fit(log)``,
``predict(log, k, users, items, filter_seen_items)``, ``predict_pairs``, ``fit_predict``,
``_init_args`` / ``_save_model`` / ``_load_model`` for ``save``/``load``.  Inside, d3rlpy's
``CQL.fit`` loop and the per-user scoring loop are replaced by ``engine.CqlEngine``.
"""
from __future__ import annotations

import dataclasses
import json
import os
from typing import Any, Dict, Optional

import numpy as np
import pandas as pd

from .engine import OFFLINE_SUM_KEYS, CqlEngine, CqlHyperParams, check_ensemble, offline_scores
from .engine import inference_inputs as _inference_inputs
from .mdp import build_mdp_on_device, seen_csr
from .parallel import GradAllReducer, dist_info, gather_rows, shard_range
from .recommender import Recommender, _rec_frame, get_top_k_recs


class CQL(Recommender):
    """Conservative Q-Learning recommender (Kumar et al. 2020) on RePlay's plug-in API.

    Observation = ``(user_idx, item_idx)``, action = ``relevance`` (one episode per user);
    relevance of a pair at predict time is ``mean_i Q_i(x, pi_greedy(x))`` (``score="q"``,
    d3rlpy ``predict_value(x, predict(x))``) or the greedy action itself (``score="policy"``).

    ``n_steps`` (d3rlpy's name, default 1) is the TD horizon: each replay row carries the discounted reward sum of up to
    ``n_steps`` steps of its user's episode and the TD target bootstraps from the state that many steps later with
    discount ``gamma ** k`` (``k`` shorter where the episode ends first).  It is unrelated to ``resume(n_steps=...)`` and
    ``engine.update(n_steps)``, which count update steps.

    ``scaler`` (observations: ``None``, ``"min_max"``, ``"standard"``), ``action_scaler`` (``None``, ``"min_max"``) and
    ``reward_scaler`` (``None``, ``"min_max"``, ``"standard"``) are d3rlpy's preprocessors, or explicit-parameter dicts
    (``replay_cql_b200.scalers``).  Names are fitted by ``fit`` on the replay table (all ranks' rows when it is
    sharded); ``resume`` and ``load`` keep the fitted parameters.  The minibatches and the scored observations are
    transformed, the replay table stays raw.  With ``score="q"`` the greedy action enters Q in the network's (scaled)
    action space, where d3rlpy's ``predict_value(x, predict(x))`` round-trips it through the reverse and forward action
    transforms -- a few ulps of the action apart; ``score="policy"`` returns the reverse-transformed action (rating
    units).
    """

    SHARD_ROWS = 200_000_000      # data-parallel fits shard the replay table by user range from this log size on
    _observation_shape = (2,)
    _action_size = 1
    can_predict_cold_users = False
    can_predict_cold_items = False
    accepts_arrow = True          # `_fit` ingests a pyarrow.Table chunk by chunk (mdp.ingest_log): no frame conversion
    _predict_filters_seen = True  # `_predict` returns at most k UNSEEN items per user: the template's generic pass is skipped

    _search_space = {
        "actor_learning_rate": {"type": "loguniform", "args": [1e-5, 1e-3]},
        "critic_learning_rate": {"type": "loguniform", "args": [3e-5, 3e-4]},
        "temp_learning_rate": {"type": "loguniform", "args": [1e-5, 1e-3]},
        "alpha_learning_rate": {"type": "loguniform", "args": [1e-5, 1e-3]},
        "gamma": {"type": "loguniform", "args": [0.9, 0.999]},
        "n_critics": {"type": "int", "args": [2, 4]},
    }

    # pylint: disable=too-many-arguments
    def __init__(
        self,
        top_k: int = 10,
        action_randomization_scale: float = 1e-3,
        n_epochs: int = 1,
        batch_size: int = 1024,
        actor_learning_rate: float = 1e-4,
        critic_learning_rate: float = 3e-4,
        temp_learning_rate: float = 1e-4,
        alpha_learning_rate: float = 1e-4,
        gamma: float = 0.99,
        tau: float = 0.005,
        n_critics: int = 2,
        initial_temperature: float = 1.0,
        initial_alpha: float = 1.0,
        alpha_threshold: float = 10.0,
        conservative_weight: float = 5.0,
        n_action_samples: int = 10,
        soft_q_backup: bool = False,
        use_gpu: bool = True,
        precision: str = "f16x3",
        score: str = "q",
        squash: str = "eps",
        seed: int = 12345,
        n_steps_per_epoch: Optional[int] = None,
        save_replay_table: bool = False,
        log_every: int = 1000,
        shard_table: Optional[bool] = None,
        n_steps: int = 1,
        scaler=None,
        action_scaler=None,
        reward_scaler=None,
    ):
        from . import _lib, scalers
        scaler = scalers.validate("scaler", scaler)
        action_scaler = scalers.validate("action_scaler", action_scaler)
        reward_scaler = scalers.validate("reward_scaler", reward_scaler)
        if not isinstance(n_steps, (int, np.integer)) or not 1 <= n_steps <= _lib.MAX_N_STEPS:
            raise ValueError(f"n_steps (the n-step TD horizon) must be an integer in 1..{_lib.MAX_N_STEPS}")
        check_ensemble(n_critics, n_action_samples)
        if soft_q_backup:
            raise ValueError("soft_q_backup=True is not supported (d3rlpy default False is restated)")
        if not use_gpu:
            raise ValueError("replay_cql_b200.CQL runs on a B200 only (use_gpu must be True); there is no CPU path")
        if score not in ("q", "policy"):
            raise ValueError("score must be 'q' or 'policy'")
        if top_k < 0 or n_epochs < 0 or batch_size < 1:
            raise ValueError("top_k, n_epochs must be >= 0 and batch_size >= 1")
        self.top_k = top_k
        self.action_randomization_scale = action_randomization_scale
        self.n_epochs = n_epochs
        self.batch_size = batch_size
        self.actor_learning_rate = actor_learning_rate
        self.critic_learning_rate = critic_learning_rate
        self.temp_learning_rate = temp_learning_rate
        self.alpha_learning_rate = alpha_learning_rate
        self.gamma = gamma
        self.tau = tau
        self.n_critics = n_critics
        self.initial_temperature = initial_temperature
        self.initial_alpha = initial_alpha
        self.alpha_threshold = alpha_threshold
        self.conservative_weight = conservative_weight
        self.n_action_samples = n_action_samples
        self.soft_q_backup = soft_q_backup
        self.use_gpu = use_gpu
        self.precision = precision
        self.score = score
        self.squash = squash
        self.seed = seed
        self.n_steps_per_epoch = n_steps_per_epoch
        self.save_replay_table = save_replay_table
        self.log_every = log_every
        self.shard_table = shard_table
        self.n_steps = int(n_steps)
        self.scaler, self.action_scaler, self.reward_scaler = scaler, action_scaler, reward_scaler
        self.engine: Optional[CqlEngine] = None
        self.last_metrics: Optional[Dict[str, float]] = None

    @property
    def _init_args(self) -> dict:
        return {
            "top_k": self.top_k,
            "action_randomization_scale": self.action_randomization_scale,
            "n_epochs": self.n_epochs,
            "batch_size": self.batch_size,
            "actor_learning_rate": self.actor_learning_rate,
            "critic_learning_rate": self.critic_learning_rate,
            "temp_learning_rate": self.temp_learning_rate,
            "alpha_learning_rate": self.alpha_learning_rate,
            "gamma": self.gamma,
            "tau": self.tau,
            "n_critics": self.n_critics,
            "initial_temperature": self.initial_temperature,
            "initial_alpha": self.initial_alpha,
            "alpha_threshold": self.alpha_threshold,
            "conservative_weight": self.conservative_weight,
            "n_action_samples": self.n_action_samples,
            "soft_q_backup": self.soft_q_backup,
            "use_gpu": self.use_gpu,
            "precision": self.precision,
            "score": self.score,
            "squash": self.squash,
            "seed": self.seed,
            "n_steps_per_epoch": self.n_steps_per_epoch,
            "save_replay_table": self.save_replay_table,
            "log_every": self.log_every,
            "shard_table": self.shard_table,
            "n_steps": self.n_steps,
            "scaler": self.scaler,
            "action_scaler": self.action_scaler,
            "reward_scaler": self.reward_scaler,
        }

    # ------------------------------------------------------------------ engine
    def _hyper_params(self) -> CqlHyperParams:
        return CqlHyperParams(
            batch_size=self.batch_size, n_critics=self.n_critics, n_action_samples=self.n_action_samples,
            gamma=self.gamma, tau=self.tau, actor_lr=self.actor_learning_rate, critic_lr=self.critic_learning_rate,
            temp_lr=self.temp_learning_rate, alpha_lr=self.alpha_learning_rate,
            initial_temperature=self.initial_temperature, initial_alpha=self.initial_alpha,
            alpha_threshold=self.alpha_threshold, conservative_weight=self.conservative_weight,
            precision=self.precision, squash=self.squash, seed=self.seed, n_steps=self.n_steps,
        )

    def _make_engine(self) -> CqlEngine:
        rank, world, local_rank = dist_info()
        if self.engine is not None:
            self.engine.close()
        self.engine = CqlEngine(self._hyper_params(), device=local_rank, rank=rank, world_size=world)
        return self.engine

    def _clear_cache(self) -> None:
        pass

    # ------------------------------------------------------------------ fit
    def _fit(self, log: pd.DataFrame, user_features=None, item_features=None) -> None:
        """MDP build -> HBM replay table -> ``n_epochs`` x (N // (B*world)) fused updates."""
        eng = self._make_engine()
        n_log = int(log.num_rows) if hasattr(log, "num_rows") else len(log)
        if n_log == 0:
            self.logger.warning("CQL.fit: empty log")
            return
        rank, world, _ = dist_info()
        # Data parallel: every rank holds the whole replay table, or -- for shapes that would not be worth replicating
        # (`shard_table=True`, default above SHARD_ROWS rows) -- only the episodes of ITS contiguous user range, balanced
        # by row count (SURVEY.md 8e "MDP build: by user"); it then walks its own epoch permutation.
        sharded = world > 1 and (self.shard_table if self.shard_table is not None else n_log >= self.SHARD_ROWS)
        if sharded:
            from .mdp import shard_log_by_user
            log = shard_log_by_user(log, rank, world)
        build_mdp_on_device(eng, log, top_k=self.top_k, action_randomization_scale=self.action_randomization_scale)
        eng.set_table_sharded(sharded)
        self._table_sharded = sharded
        self._fit_preprocessing(sharded)
        n_rows = eng.n_transitions
        per_epoch = self.n_steps_per_epoch
        if per_epoch is None:
            per_epoch = n_log // (self.batch_size * world)    # d3rlpy drops the last partial minibatch
        total = int(self.n_epochs) * int(per_epoch)
        if total == 0:
            self.logger.warning("CQL.fit: 0 update steps (log has %d rows, batch_size*world = %d)",
                                n_rows, self.batch_size * world)
            return
        self._run_steps(total, per_epoch)

    def _fit_preprocessing(self, sharded: bool) -> None:
        """Fit the scalers on the table just built (a sharded table: every rank's statistics, all-gathered and combined
        in rank order, so every rank applies the same parameter bits)."""
        from . import scalers
        specs = {"scaler": self.scaler, "action_scaler": self.action_scaler, "reward_scaler": self.reward_scaler}
        if all(v is None for v in specs.values()):
            return
        stats = self.engine.table_stats()
        if sharded:
            rows = gather_rows(scalers.stats_to_array(stats)[None, :])
            stats = scalers.combine([scalers.stats_from_array(r) for r in rows])
        self.engine.set_preprocessing(**specs, stats=stats)

    def _run_steps(self, total: int, per_epoch: Optional[int] = None) -> None:
        """``total`` updates on the engine's replay table, continuing from its step counter (which fixes the position
        in the epoch permutation and the Philox counters).  The six losses of d3rlpy's progress line (temp_loss, temp,
        alpha_loss, alpha, critic_loss, actor_loss) are logged at DEBUG every ``log_every`` steps on every world size,
        in the house style of ``replay/models/base_rec.py:639-646`` (``self.logger``)."""
        eng = self.engine
        rank, world, _ = dist_info()
        every = max(1, int(self.log_every or total))
        if per_epoch:
            every = min(every, max(1, int(per_epoch)))
        first = eng.get_optimizer()[2]
        stepper = exchange = None
        if world > 1:
            from .parallel import DataParallelStepper, PeerGradExchange, make_grad_exchange
            import torch
            torch.cuda.set_device(eng.device)
            exchange = getattr(self, "_exchange", None)
            if exchange is None or exchange.engine is not eng:
                exchange = self._exchange = make_grad_exchange(eng)     # NVLink peer memory if available, else NCCL
            fused = isinstance(exchange, PeerGradExchange) and exchange.fused
            if not fused:                                   # the step (phases + exchanges between them) as one CUDA graph
                stepper = DataParallelStepper(eng, reducer=exchange)
                stepper.stream.wait_stream(torch.cuda.current_stream())
            torch.distributed.barrier()                     # every rank's engine is attached before the first exchange
        done = 0
        while done < total:
            chunk = min(every, total - done)
            if stepper is None:
                # single GPU -- or data parallel with the exchange INSIDE the update kernels: the library's own graph
                self.last_metrics = eng.update(chunk)
                if exchange is not None:
                    exchange.check()                        # raises if a wait for a peer timed out
            else:
                stepper.run(chunk)                          # exactly `chunk` updates (eager warm-up steps included)
                stepper.finish()                            # raises if a gradient exchange timed out
                self.last_metrics = eng.read_metrics()
            done += chunk
            self.logger.debug("CQL step %d (rank %d/%d)%s %s", first + done, rank, world,
                              f" epoch {(done - 1) // per_epoch + 1}/{self.n_epochs}" if per_epoch else "",
                              " ".join(f"{k}={v:.6g}" for k, v in self.last_metrics.items()))
        if stepper is not None:
            assert stepper.steps_done == total
            stepper.graph = None

    def resume(self, log: Optional[pd.DataFrame] = None, n_steps: Optional[int] = None,
               n_epochs: Optional[int] = None) -> "CQL":
        """Continue training a fitted or loaded model EXACTLY where it stopped (SURVEY.md 8f-4): weights, targets, the
        Adam moments and the step counter come from the engine (``save``/``load`` persist them); the step counter fixes
        the position in the epoch permutation and the Philox counters, so ``fit(N) -> save -> load -> resume(M)`` is
        bit-identical to ``fit(N + M)``.  The replay table is taken from the checkpoint when it was saved with
        ``save_replay_table=True``; otherwise it is rebuilt from ``log`` (the MDP builder is deterministic: stable
        sorts + action noise seeded per original row)."""
        if self.engine is None:
            raise AttributeError("CQL model is not fitted or loaded")
        eng = self.engine
        if eng.n_transitions == 0:
            if log is None or len(log) == 0:
                raise ValueError("resume: the checkpoint holds no replay table (save_replay_table=False) -- pass the log")
            build_mdp_on_device(eng, log, top_k=self.top_k, action_randomization_scale=self.action_randomization_scale)
        _, world, _ = dist_info()
        per_epoch = self.n_steps_per_epoch or eng.n_transitions // (self.batch_size * world)
        total = int(n_steps) if n_steps is not None else int(n_epochs if n_epochs is not None else self.n_epochs) * per_epoch
        if total > 0:
            self._run_steps(total, per_epoch)
        return self

    # ------------------------------------------------------------------ predict
    def _predict(self, log: Optional[pd.DataFrame], k: int, users: pd.DataFrame, items: pd.DataFrame,
                 user_features=None, item_features=None, filter_seen_items: bool = True) -> pd.DataFrame:
        """Fused user x item scoring + seen filter + top-k on the GPU; users sharded over ranks."""
        if self.engine is None:
            raise AttributeError("CQL model is not fitted or loaded")
        u = np.sort(users["user_idx"].to_numpy().astype(np.int32))
        it = np.sort(items["item_idx"].to_numpy().astype(np.int32))
        if u.size == 0 or it.size == 0:
            return _rec_frame([], [], [])
        rank, world, _ = dist_info()
        lo, hi = shard_range(u.size, rank, world)
        u_local = u[lo:hi]
        indptr = seen = None
        kk = min(int(k), int(it.size))
        if kk <= 0:                                     # k = 0: nothing to recommend (the reference returns an empty frame)
            return _rec_frame([], [], [])
        from . import _lib
        on_device = kk <= _lib.MAX_TOPK and u_local.size > 0
        n_dim = int(u.max()) + 1
        if filter_seen_items and log is not None and len(log):
            wanted = np.zeros(n_dim, dtype=np.uint8)     # rows of the requested users: a table lookup, not isin()'s sort
            wanted[u_local] = 1
            if on_device:
                # the seen CSR is built on the GPU from the log's id columns (cql_seen_csr) and never exists on the host
                indptr, seen = self.engine.seen_csr_device(log["user_idx"].to_numpy(), log["item_idx"].to_numpy(), n_dim, wanted)
            else:
                lu = log["user_idx"].to_numpy()
                keep = (lu < n_dim) & (wanted[np.minimum(lu, n_dim - 1)] != 0)
                indptr, seen = seen_csr(log if keep.all() else log[keep], n_dim)
        if on_device:
            import torch
            dev = torch.device("cuda", self.engine.device)
            ti, ts = self.engine.score_topk_device(torch.from_numpy(u_local).to(dev), torch.from_numpy(it).to(dev), kk,
                                                   indptr, seen, mode=self.score)
            top_i, top_s = ti.cpu().numpy(), ts.cpu().numpy()
        else:
            top_i, top_s = self._score_topk_any_k(u_local, it, kk, indptr, seen, n_dim)
        rows_u = np.repeat(u_local, kk).reshape(-1, 1)
        packed = np.concatenate([rows_u.astype(np.float64), top_i.reshape(-1, 1).astype(np.float64),
                                 top_s.reshape(-1, 1).astype(np.float64)], axis=1)
        if world > 1:
            packed = gather_rows(packed)
        keep = packed[:, 1] >= 0
        return _rec_frame(packed[keep, 0], packed[keep, 1], packed[keep, 2])

    def _score_topk_any_k(self, u_local, items, k: int, indptr, seen, n_users_dim: int):
        """``engine.score_topk`` for any ``k`` (the reference's ``predict`` accepts any k, ``base_rec.py:466-539``): the
        kernel selects at most ``MAX_TOPK`` per pass, so a larger ``k`` runs in passes of ``MAX_TOPK``, each pass
        treating the items already selected as seen -- the concatenation is the descending top-``k`` (no CPU scoring)."""
        from . import _lib
        if k <= _lib.MAX_TOPK:
            return self.engine.score_topk(u_local, items, k, indptr, seen, mode=self.score)
        parts_i, parts_s = [], []
        if indptr is None:
            indptr, seen = np.zeros(n_users_dim + 1, dtype=np.int64), np.zeros(0, dtype=np.int32)
        left = k
        while left > 0:
            kk = min(left, _lib.MAX_TOPK)
            ti, ts = self.engine.score_topk(u_local, items, kk, indptr, seen, mode=self.score)
            parts_i.append(ti)
            parts_s.append(ts)
            left -= kk
            if left > 0:        # picked items join the seen lists of their users (sorted, de-duplicated CSR over user id)
                pu = np.repeat(u_local.astype(np.int64), kk)[(ti >= 0).reshape(-1)]
                pi = ti.reshape(-1)[(ti >= 0).reshape(-1)].astype(np.int64)
                su = np.repeat(np.arange(indptr.size - 1, dtype=np.int64), np.diff(indptr))
                key = np.unique(np.concatenate([su * (2 ** 32) + seen.astype(np.int64), pu * (2 ** 32) + pi]))
                counts = np.bincount(key >> 32, minlength=indptr.size - 1)
                indptr = np.zeros(indptr.size, dtype=np.int64)
                np.cumsum(counts, out=indptr[1:])
                seen = (key & 0xFFFFFFFF).astype(np.int32)
        return np.concatenate(parts_i, axis=1), np.concatenate(parts_s, axis=1)

    def _predict_pairs(self, pairs: pd.DataFrame, log: Optional[pd.DataFrame] = None) -> pd.DataFrame:
        """Native pair scoring instead of the generic fallback (``base_rec.py:784-823``)."""
        if self.engine is None:
            raise AttributeError("CQL model is not fitted or loaded")
        u = pairs["user_idx"].to_numpy().astype(np.int32)
        it = pairs["item_idx"].to_numpy().astype(np.int32)
        rel = self.engine.score_pairs(u, it, mode=self.score) if u.size else np.zeros(0, dtype=np.float32)
        return _rec_frame(u, it, rel)

    # ------------------------------------------------------------------ per-observation inference (d3rlpy's algo calls)
    def predict_value(self, users, items, actions=None, with_std: bool = False):
        """d3rlpy's ``predict_value(x, action, with_std)`` on observations ``x = (users[i], items[i])`` (DESIGN.md
        section 1, "Inference"): float32 ``mean_c Q_c(x, a)`` per pair and, with ``with_std``, ``(mean, std)`` with the
        population std over the critics (0 at ``n_critics = 1``).  ``actions`` are in rating units and pass through the
        fitted action scaler; None uses the greedy action ``tanh(mu(x))`` in network space (the value of
        ``score="q"``).  Ids must lie in [0, 2^24).  Data parallel: every rank computes its own inputs locally, with no
        collective.  The model is not modified."""
        u, i, a = _inference_inputs(users, items, actions)
        return self._fitted_engine().predict_value(u, i, a, with_std=with_std)

    def predict_action(self, users, items) -> np.ndarray:
        """d3rlpy's ``predict(x)``: the greedy action ``tanh(mu(x))`` per pair in rating units (the value of
        ``score="policy"``), float32.  Data parallel: every rank computes its own inputs locally."""
        u, i, _ = _inference_inputs(users, items)
        return self._fitted_engine().predict_action(u, i)

    def sample_action(self, users, items) -> np.ndarray:
        """d3rlpy's ``sample_action(x)``: one draw per pair from the squashed Gaussian policy, in rating units, float32.
        The noise comes from a Philox stream keyed by ``seed`` and numbered by this model's earlier ``sample_action``
        calls since its engine was created (``fit`` or ``load``): consecutive calls differ, and a model fitted or loaded
        the same way repeats them.  The counter is not saved and the update never reads it.  Data parallel: every rank
        computes its own inputs locally, with no collective (ranks asking for the same rows draw the same noise)."""
        u, i, _ = _inference_inputs(users, items)
        return self._fitted_engine().sample_action(u, i)

    def _fitted_engine(self) -> CqlEngine:
        if self.engine is None:
            raise AttributeError("CQL model is not fitted or loaded")
        return self.engine

    # ------------------------------------------------------------------ evaluation (the step right after predict)
    def evaluate(self, recs: pd.DataFrame, ground_truth: pd.DataFrame, k) -> dict:
        """Ranking metrics of a recommendation frame against ``ground_truth`` on the GPU:
        ``{metric: {k: value}}`` for NDCG, HitRate, MAP, MRR, Precision, Recall with the reference's definitions
        (``replay/metrics/*.py``; users = the ground-truth users, ``base_metric.py:102-140``).  Replaces the Spark
        joins + Python UDFs that ``optimize`` trials run after every ``predict`` (``optuna_objective.py:80-111``)."""
        if self.engine is None:
            raise AttributeError("CQL model is not fitted or loaded")
        ks = [int(x) for x in (k if hasattr(k, "__iter__") else [k])]
        gt = ground_truth[["user_idx", "item_idx"]].drop_duplicates()
        users = np.sort(gt["user_idx"].unique()).astype(np.int32)
        if users.size == 0:
            return {name: {kk: 0.0 for kk in ks} for name in self.engine.METRIC_NAMES}
        gt_ptr, gt_items = seen_csr(gt, int(users.max()) + 1)
        top = get_top_k_recs(recs, max(ks)) if len(recs) else recs
        top = top[top["user_idx"].isin(users)].sort_values(["user_idx", "relevance", "item_idx"],
                                                            ascending=[True, False, True], kind="stable")
        k_rec = max(1, max(ks))
        table = np.full((users.size, k_rec), -1, dtype=np.int32)
        if len(top):
            row = np.searchsorted(users, top["user_idx"].to_numpy())
            pos = top.groupby("user_idx").cumcount().to_numpy()
            table[row, pos] = top["item_idx"].to_numpy().astype(np.int32)
        return self.engine.rank_metrics(table, users, gt_ptr, gt_items, ks)

    def offline_metrics(self, log: Any = None, return_threshold: Optional[float] = None) -> Dict[str, float]:
        """d3rlpy's offline scorers (``d3rlpy.metrics.scorer``, DESIGN.md section 1) of the current networks on the GPU:
        ``td_error``, ``discounted_sum_of_advantage``, ``average_value_estimation``, ``value_estimation_std``,
        ``initial_state_value_estimation``, ``continuous_action_diff`` and, with ``return_threshold``, ``soft_opc``.

        ``log=None`` evaluates the fitted replay table (it must be one-step: ``n_steps = 1``, and present: a model loaded
        without ``save_replay_table`` has none).  With a ``log`` (anything ``fit`` accepts) the one-step rows are built
        by the same MDP builder (``top_k``, ``action_randomization_scale``) on a short-lived evaluation engine holding
        this model's networks and scalers.  Data parallel: each rank evaluates its own user range (of the log, or of a
        sharded table) and the sums are combined in rank order; a replicated table is evaluated whole on every rank.
        Nothing of the model changes: ``fit -> offline_metrics -> resume`` equals ``fit -> resume``."""
        if self.engine is None:
            raise AttributeError("CQL model is not fitted or loaded")
        return evaluate_offline(self.engine, log, return_threshold, self.top_k, self.action_randomization_scale,
                                getattr(self, "_table_sharded", False))

    def _default_criterion(self):
        """``optimize`` trials score NDCG@k on the GPU (``cql_rank_metrics``) instead of the pandas criterion."""
        return lambda recs, test, k: self.evaluate(recs, test, k)["NDCG"][int(k)]

    # ------------------------------------------------------------------ persistence (model_handler.py:38, :90)
    def _save_model(self, path: str) -> None:
        os.makedirs(path, exist_ok=True)
        if self.engine is None:
            with open(os.path.join(path, "meta.json"), "w") as f:
                json.dump({"fitted": False}, f)
            return
        m, v, step = self.engine.get_optimizer()
        np.savez(os.path.join(path, "state.npz"), state=self.engine.get_state(), adam_m=m, adam_v=v)
        n_rows = self.engine.n_transitions if self.save_replay_table else 0
        if n_rows:                                          # [n, 8] rows: obs.x obs.y act rew next.x next.y term discount
            np.save(os.path.join(path, "replay_table.npy"), self.engine.export_transitions())
        meta = {"fitted": True, "step": step, "format": 2, "replay_rows": int(n_rows)}
        prep = self.engine.get_preprocessing()
        if any(v is not None for v in prep.values()):
            meta["preprocessing"] = prep                    # the fitted parameters; absent = no preprocessing
        with open(os.path.join(path, "meta.json"), "w") as f:
            json.dump(meta, f)

    def _load_model(self, path: str) -> None:
        with open(os.path.join(path, "meta.json")) as f:
            meta = json.load(f)
        if not meta.get("fitted"):
            return
        data = np.load(os.path.join(path, "state.npz"))
        eng = self._make_engine()
        eng.set_state(data["state"])
        eng.set_optimizer(data["adam_m"], data["adam_v"], int(meta["step"]))
        if meta.get("preprocessing"):
            eng.set_preprocessing(**meta["preprocessing"])
        if meta.get("replay_rows"):
            # verbatim: n-step rows cannot be rebuilt from their columns, and one-step rows come back bit for bit
            eng.set_table_rows(np.load(os.path.join(path, "replay_table.npy")))


def evaluate_offline(eng: CqlEngine, log: Any, return_threshold: Optional[float], top_k: int,
                     action_randomization_scale: float, table_sharded: bool,
                     mdp_seed: Optional[int] = None) -> Dict[str, float]:
    """d3rlpy's offline scorers of ``eng``'s networks (``CQL.offline_metrics``, ``ope.FQE.offline_metrics``).

    ``log=None`` evaluates the engine's replay table (one-step, present; ``table_sharded``: in a data-parallel job it
    holds only this rank's users).  With a ``log`` the one-step rows are built by the MDP builder (``top_k``,
    ``action_randomization_scale``; ``mdp_seed``, default ``eng``'s seed, draws the action noise) on a short-lived
    evaluation engine holding ``eng``'s networks and scalers; in a data-parallel job each rank evaluates its own user range.  Sharded sums are combined in rank order."""
    if return_threshold is not None:
        if isinstance(return_threshold, bool) or not isinstance(return_threshold, (int, float, np.integer, np.floating)) \
                or not np.isfinite(float(return_threshold)):
            raise ValueError("return_threshold must be a finite number or None")
        return_threshold = float(return_threshold)
    rank, world, local_rank = dist_info()
    if log is None:
        if eng.hp.n_steps > 1:
            raise ValueError("offline_metrics: the replay table holds n-step rows (n_steps > 1) -- pass the log to "
                             "evaluate its one-step transitions")
        if eng.n_transitions == 0:
            raise ValueError("offline_metrics: the model holds no replay table (e.g. loaded from a checkpoint saved "
                             "without save_replay_table) -- pass the log")
        sums = eng.offline_metrics(return_threshold)
        sharded = world > 1 and table_sharded
    else:
        n_log = int(log.num_rows) if hasattr(log, "num_rows") else len(log)
        if n_log == 0:
            raise ValueError("offline_metrics: empty log")
        sharded = world > 1
        if sharded:
            from .mdp import shard_log_by_user
            log = shard_log_by_user(log, rank, world)
        n_local = int(log.num_rows) if hasattr(log, "num_rows") else len(log)
        sums = {k: 0 for k in OFFLINE_SUM_KEYS}
        if n_local:
            hp = dataclasses.replace(eng.hp, n_steps=1, seed=eng.hp.seed if mdp_seed is None else mdp_seed)
            ev = CqlEngine(hp, device=local_rank, rank=rank, world_size=world)
            try:
                ev.set_state(eng.get_state())
                prep = eng.get_preprocessing()
                if any(v is not None for v in prep.values()):
                    ev.set_preprocessing(**prep)
                build_mdp_on_device(ev, log, top_k=top_k, action_randomization_scale=action_randomization_scale)
                sums = ev.offline_metrics(return_threshold)
            finally:
                ev.close()
    if sharded:
        parts = gather_rows(np.array([[sums[k] for k in OFFLINE_SUM_KEYS]], dtype=np.float64))
        total = np.zeros(len(OFFLINE_SUM_KEYS), dtype=np.float64)
        for row in parts:                                   # rank order: every rank adds the same values in the same order
            total = total + row
        sums = {k: (int(v) if k.startswith("n_") else float(v)) for k, v in zip(OFFLINE_SUM_KEYS, total)}
    return offline_scores(sums, return_threshold is not None)
