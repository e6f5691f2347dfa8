"""Host driver of the CUDA library: one ``CqlEngine`` per GPU.

Mirrors the *role* of d3rlpy's ``CQLImpl`` for the RePlay wrapper ([EXT]
``d3rlpy/algos/torch/cql_impl.py``): owns the learner state, runs updates,
answers ``predict`` / ``predict_value`` -- but every number is produced by the
sm_100a kernels behind ``include/cql_b200.h``.  PyTorch appears only as
plumbing (``torch.distributed`` for the data-parallel gradient all-reduce and a
zero-copy view of the library's gradient buffer).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, asdict
from typing import Callable, Dict, Optional, Sequence

import numpy as np

from . import _lib, layout, scalers
from .frames import timestamps_to_int64

METRIC_NAMES = ("temp_loss", "temp", "alpha_loss", "alpha", "critic_loss", "actor_loss")
NOISE_KEYS = ("temp_eps", "alpha_eps_t", "alpha_eps_t1", "alpha_u",
              "critic_eps_t", "critic_eps_t1", "critic_u", "actor_eps")
PRECISIONS = {"fp32": _lib.PREC_FP32, "tf32x3": _lib.PREC_TF32X3, "bf16": _lib.PREC_BF16,
              "f16x3": _lib.PREC_F16X3}
SQUASH = {"eps": _lib.SQUASH_EPS, "softplus": _lib.SQUASH_SOFTPLUS}
SCORE_MODES = {"q": _lib.SCORE_Q, "policy": _lib.SCORE_POLICY}
OFFLINE_SUM_KEYS = tuple(name for name, _ in _lib.OfflineSums._fields_)


def offline_scores(sums: Dict[str, float], soft_opc: bool) -> Dict[str, float]:
    """Sums and counts of ``CqlEngine.offline_metrics`` (one table, or several shards added up) -> d3rlpy's offline
    scorer values (DESIGN.md section 1): means over rows, ``initial_state_value_estimation`` over episodes, ``soft_opc``
    (only when ``soft_opc``) NaN when no episode reached the return threshold.  Unlike d3rlpy's scorers, which negate the
    "smaller is better" ones, every value is the plain mean."""
    n, n_ep, n_ok = sums["n_rows"], sums["n_episodes"], sums["n_success_rows"]
    out = {
        "td_error": sums["td_error"] / n,
        "discounted_sum_of_advantage": sums["discounted_advantage"] / n,
        "average_value_estimation": sums["value"] / n,
        "value_estimation_std": sums["value_std"] / n,
        "initial_state_value_estimation": sums["initial_value"] / n_ep,
        "continuous_action_diff": sums["action_diff"] / n,
    }
    if soft_opc:
        out["soft_opc"] = sums["success_q"] / n_ok - sums["all_q"] / n if n_ok else float("nan")
    return out


@dataclass
class CqlHyperParams:
    """d3rlpy CQL defaults (SURVEY.md Appendix A); ``batch_size`` 1024 per BASELINE.json."""

    batch_size: int = 1024
    n_critics: int = 2
    n_action_samples: int = 10
    gamma: float = 0.99
    tau: float = 0.005
    actor_lr: float = 1e-4
    critic_lr: float = 3e-4
    temp_lr: float = 1e-4
    alpha_lr: float = 1e-4
    initial_temperature: float = 1.0
    initial_alpha: float = 1.0
    alpha_threshold: float = 10.0
    conservative_weight: float = 5.0
    beta1: float = 0.9
    beta2: float = 0.999
    adam_eps: float = 1e-8
    precision: str = "f16x3"   # tcgen05 fp16 hi/lo 3-term split, FP32-grade (1e-4 gates); "fp32" = CUDA-core FMA
    squash: str = "eps"
    seed: int = 12345
    n_steps: int = 1           # n-step TD horizon of the replay table and the TD target (d3rlpy ``n_steps``)

    def __post_init__(self):
        check_ensemble(self.n_critics, self.n_action_samples)


def check_ensemble(n_critics, n_action_samples) -> None:
    """``ValueError`` unless 1 <= n_critics <= ``MAX_CRITICS`` and 1 <= n_action_samples <= ``MAX_ACTION_SAMPLES``."""
    if not isinstance(n_critics, (int, np.integer)) or not 1 <= n_critics <= _lib.MAX_CRITICS:
        raise ValueError(f"n_critics must be an integer in 1..{_lib.MAX_CRITICS}")
    if not isinstance(n_action_samples, (int, np.integer)) or not 1 <= n_action_samples <= _lib.MAX_ACTION_SAMPLES:
        raise ValueError(f"n_action_samples must be an integer in 1..{_lib.MAX_ACTION_SAMPLES}")


MAX_ID = 2 ** 24                                     # ids are exact in float32 observations below this


def _column(x) -> np.ndarray:
    """1-D view of an array or an [n, 1] column (d3rlpy passes actions as [n, action_size])."""
    a = np.asarray(x)
    return a[:, 0] if a.ndim == 2 and a.shape[1] == 1 else a


def inference_inputs(users, items, actions=None):
    """Arguments of the per-observation inference calls -> (users int32, items int32, actions float32 or None), 1-D
    and contiguous.  ``ValueError`` unless users and items are integer ids in [0, 2^24) of one length and ``actions``
    (if given) holds one finite number per pair; the same checks the library makes (return code 3)."""
    out = []
    for name, ids in (("users", users), ("items", items)):
        a = _column(ids)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
            raise ValueError(f"{name} must be a 1-D array of integer ids")
        if a.size and (int(a.min()) < 0 or int(a.max()) >= MAX_ID):
            raise ValueError(f"{name}: ids must be in [0, 2**24) to be exact in float32 observations")
        out.append(np.ascontiguousarray(a, dtype=np.int32))
    u, i = out
    if u.size != i.size:
        raise ValueError("users and items must have the same length")
    if actions is None:
        return u, i, None
    a = _column(actions)
    if a.ndim != 1 or a.size != u.size:
        raise ValueError("actions must hold one action per (user, item) pair")
    if a.size and a.dtype.kind not in "iuf":
        raise ValueError("actions must be numbers")
    with np.errstate(over="ignore"):                  # a value beyond float32 becomes inf and is rejected below
        a = np.ascontiguousarray(a, dtype=np.float32)
    if not np.isfinite(a).all():
        raise ValueError("actions must be finite (as float32)")
    return u, i, a


def _ptr(arr: Optional[np.ndarray]):
    return None if arr is None else arr.ctypes.data_as(C.c_void_p)


def _f32(a, shape=None) -> np.ndarray:
    out = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None and out.shape != shape:
        raise ValueError(f"expected shape {shape}, got {out.shape}")
    return out


class _DevView:
    """Zero-copy ``__cuda_array_interface__`` view of a library-owned float buffer."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {
            "shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None,
        }


class CqlEngine:
    """Learner + scorer on one GPU."""

    def __init__(self, hp: CqlHyperParams | None = None, device: int = 0, rank: int = 0, world_size: int = 1):
        self.hp = hp or CqlHyperParams()
        if self.hp.precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
        if self.hp.squash not in SQUASH:
            raise ValueError(f"squash must be one of {sorted(SQUASH)}")
        self._lib = _lib.load()
        cfg = _lib.CqlConfig()
        cfg.struct_size = C.sizeof(cfg)
        cfg.device = device
        cfg.batch_size = self.hp.batch_size
        cfg.n_critics = self.hp.n_critics
        cfg.n_action_samples = self.hp.n_action_samples
        cfg.precision = PRECISIONS[self.hp.precision]
        cfg.squash = SQUASH[self.hp.squash]
        cfg.rank, cfg.world_size = rank, world_size
        for name in ("gamma", "tau", "actor_lr", "critic_lr", "temp_lr", "alpha_lr", "initial_temperature",
                     "initial_alpha", "alpha_threshold", "conservative_weight", "beta1", "beta2", "adam_eps"):
            setattr(cfg, name, float(getattr(self.hp, name)))
        cfg.seed = int(self.hp.seed) & (2**64 - 1)
        self._h = C.c_void_p()
        rc = self._lib.cql_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            msg = self._lib.cql_last_error(None)
            self._h = None
            err = _lib.CqlArgumentError if rc == 3 else _lib.CqlLibraryError
            raise err(f"cql_create failed: {msg.decode() if msg else rc}")
        self.device, self.rank, self.world_size = device, rank, world_size
        self.n_state = int(self._lib.cql_state_floats(self._h))
        assert self.n_state == layout.state_floats(self.hp.n_critics)
        if self.hp.n_steps != 1:
            self._check(self._lib.cql_set_n_steps(self._h, int(self.hp.n_steps)), "cql_set_n_steps")
        self.set_state(layout.init_state(self.hp.n_critics, self.hp.seed, self.hp.initial_temperature,
                                         self.hp.initial_alpha))

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.cql_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str) -> None:
        _lib.check(self._h, rc, what)

    def _torch_stream(self, stream):
        """Stream for calls that consume caller-owned cuda tensors: torch's current stream when it is a
        real (non-default) stream; otherwise drain torch's default stream and use the handle's own
        stream (NULL), which the library synchronises before returning."""
        if stream is not None:
            return C.c_void_p(stream)
        import torch
        cur = torch.cuda.current_stream(torch.device("cuda", self.device))
        if cur.cuda_stream != 0:
            return C.c_void_p(cur.cuda_stream)
        cur.synchronize()
        return None

    # ------------------------------------------------------------------ state
    def set_state(self, flat: np.ndarray) -> None:
        flat = _f32(flat, (self.n_state,))
        self._check(self._lib.cql_set_weights(self._h, _ptr(flat), flat.size), "cql_set_weights")

    def get_state(self) -> np.ndarray:
        flat = np.empty(self.n_state, dtype=np.float32)
        self._check(self._lib.cql_get_weights(self._h, _ptr(flat), flat.size), "cql_get_weights")
        return flat

    def set_optimizer(self, m: np.ndarray, v: np.ndarray, step: int) -> None:
        m, v = _f32(m, (self.n_state,)), _f32(v, (self.n_state,))
        self._check(self._lib.cql_set_optimizer(self._h, _ptr(m), _ptr(v), m.size, int(step)), "cql_set_optimizer")

    def get_optimizer(self):
        m = np.empty(self.n_state, dtype=np.float32)
        v = np.empty(self.n_state, dtype=np.float32)
        step = C.c_int64(0)
        self._check(self._lib.cql_get_optimizer(self._h, _ptr(m), _ptr(v), m.size, C.byref(step)), "cql_get_optimizer")
        return m, v, int(step.value)

    # ------------------------------------------------------------------ replay table
    def load_transitions(self, obs, act, rew, term) -> None:
        """Episode-ordered steps (MDP builder output) -> HBM-resident transition rows."""
        obs = _f32(obs)
        n = obs.shape[0]
        obs = _f32(obs, (n, 2))
        act, rew, term = (_f32(np.reshape(a, -1), (n,)) for a in (act, rew, term))
        self._check(self._lib.cql_load_transitions(self._h, _ptr(obs), _ptr(act), _ptr(rew), _ptr(term), n),
                    "cql_load_transitions")

    def set_table_rows(self, rows) -> None:
        """Replay table uploaded verbatim from [n, 8] rows in the table's own format (``export_transitions`` output,
        n-step rows included): no expansion."""
        rows = _f32(rows)
        if rows.ndim != 2 or rows.shape[1] != 8 or rows.shape[0] == 0:
            raise ValueError("rows must be a non-empty [n, 8] array")
        self._check(self._lib.cql_set_table_rows(self._h, _ptr(rows), rows.shape[0]), "cql_set_table_rows")

    def build_mdp_on_device(self, user_idx, item_idx, timestamp, relevance, top_k: int = 10,
                            action_randomization_scale: float = 1e-3, action_noise=None, want_outputs: bool = False):
        """GPU MDP builder (stable radix sorts on the device) -> replay table resident in HBM.

        Columns are in the log's input order.  ``action_noise`` (float64, per original row, already scaled)
        overrides the seeded device draw.  With ``want_outputs`` returns (obs, act, rew, term, order) as numpy
        arrays in episode order (for parity tests); otherwise None."""
        user = np.ascontiguousarray(user_idx, dtype=np.int32)
        item = np.ascontiguousarray(item_idx, dtype=np.int32)
        ts = np.ascontiguousarray(timestamps_to_int64(timestamp))
        rel = np.ascontiguousarray(relevance, dtype=np.float64)
        n = user.size
        if not (item.size == ts.size == rel.size == n):
            raise ValueError("log columns must have the same length")
        if n == 0:
            raise ValueError("empty log")
        if n and (user.max() >= 2 ** 24 or item.max() >= 2 ** 24 or user.min() < 0 or item.min() < 0):
            raise ValueError("user_idx/item_idx must be in [0, 2**24) to be exact in float32 observations")
        nz = None if action_noise is None else np.ascontiguousarray(action_noise, dtype=np.float64)
        outs = [None] * 5
        if want_outputs:
            outs = [np.empty((n, 2), np.float32), np.empty(n, np.float32), np.empty(n, np.float32),
                    np.empty(n, np.float32), np.empty(n, np.int64)]
        self._check(self._lib.cql_build_mdp(self._h, _ptr(user), _ptr(item), _ptr(ts), _ptr(rel), _ptr(nz), n, int(top_k),
                                            float(action_randomization_scale), *[_ptr(o) for o in outs]), "cql_build_mdp")
        return tuple(outs) if want_outputs else None

    # ---- chunked ingestion (Arrow record batches / Parquet row groups / pandas columns; see mdp.ingest_log)
    _COLS = {"user_idx": 0, "item_idx": 1, "timestamp": 2, "relevance": 3, "action_noise": 4}
    _DTS = {np.dtype(np.int32): _lib.DT_I32, np.dtype(np.int64): _lib.DT_I64,
            np.dtype(np.float32): _lib.DT_F32, np.dtype(np.float64): _lib.DT_F64}

    def mdp_begin(self, n_rows: int) -> None:
        self._check(self._lib.cql_mdp_begin(self._h, int(n_rows)), "cql_mdp_begin")

    def mdp_append(self, column: str, address: int, dtype, count: int) -> None:
        """Next ``count`` values of ``column`` from host memory at ``address`` (any of int32/int64/float32/float64)."""
        dt = self._DTS.get(np.dtype(dtype))
        if dt is None:
            raise ValueError(f"unsupported chunk dtype {dtype} for {column}")
        self._check(self._lib.cql_mdp_append(self._h, self._COLS[column], dt, C.c_void_p(int(address)), int(count)),
                    "cql_mdp_append")

    def mdp_finish(self, top_k: int = 10, action_randomization_scale: float = 1e-3, want_outputs: bool = False, n_rows: int = 0):
        outs = [None] * 5
        if want_outputs:
            n = int(n_rows)
            outs = [np.empty((n, 2), np.float32), np.empty(n, np.float32), np.empty(n, np.float32),
                    np.empty(n, np.float32), np.empty(n, np.int64)]
        self._check(self._lib.cql_mdp_finish(self._h, int(top_k), float(action_randomization_scale), *[_ptr(o) for o in outs]),
                    "cql_mdp_finish")
        return tuple(outs) if want_outputs else None

    def set_table_sharded(self, sharded: bool) -> None:
        """Data parallel: the table holds only this rank's user range -> sample this rank's own epoch permutation."""
        self._check(self._lib.cql_set_table_sharded(self._h, 1 if sharded else 0), "cql_set_table_sharded")

    def synth_table(self, n_rows: int, n_users: int, n_items: int, seed: int = 12345) -> None:
        """Fill the replay table with a seeded synthetic log of the given shape, generated on the device (stress shape)."""
        self._check(self._lib.cql_synth_table(self._h, int(n_rows), int(n_users), int(n_items), int(seed) & (2**64 - 1)),
                    "cql_synth_table")

    def table_stats(self) -> dict:
        """Column statistics of the loaded table's one-step rows (``cql_get_table_stats``): float64 arrays ``min``,
        ``max``, ``mean``, ``m2`` and int64 ``count`` over the columns (obs.x, obs.y, act, rew), and ``rew_available``."""
        st = _lib.TableStats()
        self._check(self._lib.cql_get_table_stats(self._h, C.byref(st)), "cql_get_table_stats")
        out = {k: np.array([getattr(st.col[c], k) for c in range(4)], dtype=np.int64 if k == "count" else np.float64)
               for k in scalers.STAT_KEYS}
        out["rew_available"] = bool(st.rew_available)
        return out

    def set_preprocessing(self, scaler=None, action_scaler=None, reward_scaler=None, stats: Optional[dict] = None) -> dict:
        """d3rlpy's scalers for every later update and scoring call (``cql_set_preprocessing``).  Each argument is None,
        a kind name fitted on ``stats`` (default: this engine's ``table_stats()``) or an explicit-parameter dict (see
        ``scalers``).  All None restores the unscaled path.  -> the explicit parameters applied."""
        specs = {"scaler": scaler, "action_scaler": action_scaler, "reward_scaler": reward_scaler}
        if stats is None and any(isinstance(v, str) for v in specs.values()):
            stats = self.table_stats()
        params = scalers.resolve(specs, stats)
        p = scalers.to_struct(params)
        self._check(self._lib.cql_set_preprocessing(self._h, C.byref(p)), "cql_set_preprocessing")
        return params

    def get_preprocessing(self) -> dict:
        """{"scaler", "action_scaler", "reward_scaler"} -> explicit-parameter dict or None."""
        p = _lib.Preprocessing()
        self._check(self._lib.cql_get_preprocessing(self._h, C.byref(p)), "cql_get_preprocessing")
        return scalers.from_struct(p)

    @property
    def n_transitions(self) -> int:
        return int(self._lib.cql_num_transitions(self._h))

    def sample_rows(self, count: int, idx=None, pos: int = 0, out=None, stream: int | None = None):
        """Stand-alone replay gather (K1).  ``idx``: explicit int64 indices (numpy or cuda tensor) or
        None for the epoch permutation stream starting at ``pos``.  -> cuda tensor [count, 8]
        rows ``(obs.x, obs.y, act, rew, next_obs.x, next_obs.y, term, discount)`` (discount 0 when n_steps = 1)."""
        import torch
        dev = f"cuda:{self.device}"
        if out is None:
            out = torch.empty((count, 8), dtype=torch.float32, device=dev)
        idx_ptr = None
        if idx is not None:
            if not isinstance(idx, torch.Tensor):
                idx = torch.as_tensor(np.ascontiguousarray(idx, dtype=np.int64), device=dev)
            if idx.dtype != torch.int64 or idx.numel() != count:
                raise ValueError("idx must be int64 with `count` elements")
            idx_ptr = C.c_void_p(idx.data_ptr())
        stream = self._torch_stream(stream)
        self._check(self._lib.cql_sample_rows(self._h, idx_ptr, int(pos), int(count), C.c_void_p(out.data_ptr()),
                                              stream), "cql_sample_rows")
        return out

    def export_transitions(self, chunk: int = 1 << 22) -> np.ndarray:
        """The replay table back on the host, [n, 8] float32 rows in table order (checkpointing)."""
        import torch
        n = self.n_transitions
        out = np.empty((n, 8), dtype=np.float32)
        for lo in range(0, n, chunk):
            hi = min(n, lo + chunk)
            idx = torch.arange(lo, hi, dtype=torch.int64, device=f"cuda:{self.device}")
            out[lo:hi] = self.sample_rows(hi - lo, idx=idx).cpu().numpy()
        return out

    # ------------------------------------------------------------------ updates
    def update(self, n_steps: int = 1, want_metrics: bool = True, stream: int | None = None) -> Optional[Dict[str, float]]:
        """``n_steps`` updates with on-device sampling + Philox noise (CUDA-graph replay)."""
        m = np.zeros(6, dtype=np.float32) if want_metrics else None
        self._check(self._lib.cql_update(self._h, int(n_steps), _ptr(m), stream), "cql_update")
        return dict(zip(METRIC_NAMES, map(float, m))) if want_metrics else None

    def timed_update(self, stream: int | None = None) -> Dict[str, float]:
        """One real sampled update with CUDA events around the heavy kernels (milliseconds)."""
        out = np.zeros(8, dtype=np.float32)
        self._check(self._lib.cql_timed_update(self._h, _ptr(out), stream), "cql_timed_update")
        keys = ("critic_fwd", "critic_bwd1", "critic_bwd2", "update", "actor_step_fwd", "actor_bwd", "actor_fwd", "other")
        return dict(zip(keys, map(float, out)))

    def mma_bench(self, mode: int, iters: int = 512):
        """Issue-rate microbenchmark of tcgen05.mma kind::f16 (see ``cql_mma_bench``): -> (clocks to issue, clocks to retire)."""
        out = np.zeros(2, dtype=np.int64)
        self._check(self._lib.cql_mma_bench(self._h, int(mode), int(iters), _ptr(out)), "cql_mma_bench")
        return int(out[0]), int(out[1])

    def selftest_umma(self, A: np.ndarray, B: np.ndarray, precision: str, a_in_tmem: bool = False) -> np.ndarray:
        """D = A @ B.T on the tensor cores (A [128,k], B [n,k]); building-block self-test."""
        A, B = _f32(A), _f32(B)
        n, k = B.shape
        if A.shape != (128, k):
            raise ValueError("A must be [128, k]")
        D = np.empty((128, n), dtype=np.float32)
        self._check(self._lib.cql_selftest_umma(self._h, PRECISIONS[precision] + (0x100 if a_in_tmem else 0), _ptr(A), _ptr(B), n, k, _ptr(D)),
                    "cql_selftest_umma")
        return D

    def pack_noise(self, noise: Dict[str, np.ndarray]) -> np.ndarray:
        B, n = self.hp.batch_size, self.hp.n_action_samples
        parts = []
        for key in NOISE_KEYS:
            want = (B, 1) if key in ("temp_eps", "actor_eps") else (B, n)
            parts.append(_f32(noise[key], want).reshape(-1))
        return np.concatenate(parts)

    def update_batch(self, batch: Dict[str, np.ndarray], noise: Optional[Dict[str, np.ndarray]] = None,
                     want_grads: bool = False, stream: int | None = None):
        """One update on a host minibatch (parity / end-to-end entry).  -> (metrics, grads|None)

        ``batch["discount"]`` (optional, [B] or [B, 1]): each row's TD discount (gamma^k of an n-step row, see
        ``cql_set_n_steps``) in place of gamma; needs ``n_steps > 1``.  ``rew`` is then the n-step return and
        ``next_obs`` / ``term`` those of the window's last step."""
        B = self.hp.batch_size
        obs, nobs = _f32(batch["obs"], (B, 2)), _f32(batch["next_obs"], (B, 2))
        act, rew, term = (_f32(np.reshape(batch[k], -1), (B,)) for k in ("act", "rew", "term"))
        nz = self.pack_noise(noise) if noise is not None else None
        m = np.zeros(6, dtype=np.float32)
        g = np.zeros(layout.grad_floats(self.hp.n_critics), dtype=np.float32) if want_grads else None
        if batch.get("discount") is not None:
            if self.hp.n_steps == 1:
                raise ValueError("batch['discount'] needs n_steps > 1 (with n_steps = 1 the TD discount is gamma)")
            disc = _f32(np.reshape(batch["discount"], -1), (B,))
            rows = np.ascontiguousarray(np.concatenate([obs, act[:, None], rew[:, None], nobs, term[:, None],
                                                        disc[:, None]], axis=1))
            self._check(self._lib.cql_update_batch_rows(self._h, _ptr(rows), _ptr(nz), _ptr(m), _ptr(g), stream),
                        "cql_update_batch_rows")
        else:
            self._check(self._lib.cql_update_batch(self._h, _ptr(obs), _ptr(act), _ptr(rew), _ptr(nobs), _ptr(term),
                                                   _ptr(nz), _ptr(m), _ptr(g), stream), "cql_update_batch")
        metrics = dict(zip(METRIC_NAMES, map(float, m)))
        return metrics, (layout.unpack_grads(g, self.hp.n_critics) if want_grads else None)

    def update_batches(self, batches, stream: int | None = None):
        """Consecutive updates on host minibatches (Philox noise), pipelined inside the library: per step the batch goes
        host -> pinned ring -> device and the six metrics come back.  ``batches``: a sequence of batch dicts, or one dict of
        stacked arrays ``obs [n,B,2], act [n,B], rew [n,B], next_obs [n,B,2], term [n,B]``.  -> list of metric dicts."""
        B = self.hp.batch_size
        if not isinstance(batches, dict):
            if len(batches) == 0:
                return []
            batches = {k: np.stack([np.reshape(np.asarray(b[k], dtype=np.float32), (B, -1)) for b in batches])
                       for k in ("obs", "act", "rew", "next_obs", "term")}
        n = int(np.asarray(batches["act"]).reshape(-1, B).shape[0])
        obs = _f32(np.reshape(batches["obs"], (n * B, 2)), (n * B, 2))
        nobs = _f32(np.reshape(batches["next_obs"], (n * B, 2)), (n * B, 2))
        act, rew, term = (_f32(np.reshape(batches[k], -1), (n * B,)) for k in ("act", "rew", "term"))
        m = np.zeros((n, 6), dtype=np.float32)
        self._check(self._lib.cql_update_batches(self._h, n, _ptr(obs), _ptr(act), _ptr(rew), _ptr(nobs), _ptr(term),
                                                 _ptr(m), stream), "cql_update_batches")
        return [dict(zip(METRIC_NAMES, map(float, row))) for row in m]

    def device_buffer(self, which: int):
        ptr, n = C.c_void_p(), C.c_int64()
        self._check(self._lib.cql_device_buffer(self._h, which, C.byref(ptr), C.byref(n)), "cql_device_buffer")
        return int(ptr.value), int(n.value)

    def grad_tensor(self, which: int = _lib.BUF_ALL_GRADS):
        """torch view (no copy) of a gradient buffer, for ``torch.distributed.all_reduce``."""
        import torch
        ptr, n = self.device_buffer(which)
        return torch.as_tensor(_DevView(ptr, n), device=f"cuda:{self.device}")

    def step_phase(self, phase: int, stream: int | None = None) -> None:
        self._check(self._lib.cql_step_phase(self._h, phase, stream), "cql_step_phase")

    def upload_batch(self, batch: Dict[str, np.ndarray], stream: int | None = None) -> None:
        B = self.hp.batch_size
        obs, nobs = _f32(batch["obs"], (B, 2)), _f32(batch["next_obs"], (B, 2))
        act, rew, term = (_f32(np.reshape(batch[k], -1), (B,)) for k in ("act", "rew", "term"))
        self._check(self._lib.cql_upload_batch(self._h, _ptr(obs), _ptr(act), _ptr(rew), _ptr(nobs), _ptr(term), stream),
                    "cql_upload_batch")

    def dp_attach(self, world: int, rank: int, stage_ptrs, signal_ptrs, stage_floats: int,
                  buffer_floats: int | None = None) -> None:
        """Hand the library every rank's symmetric staging buffer / signal pad (raw device pointers).
        ``buffer_floats`` = floats in each staging buffer (default: the two staging halves only, no fused exchange)."""
        PtrArr = C.c_void_p * len(stage_ptrs)
        total = int(buffer_floats) if buffer_floats is not None else 2 * int(stage_floats)
        self._check(self._lib.cql_dp_attach(self._h, int(world), int(rank), PtrArr(*[int(p) for p in stage_ptrs]),
                                            PtrArr(*[int(p) for p in signal_ptrs]), int(stage_floats), total), "cql_dp_attach")

    def dp_allreduce(self, which: int, stream: int | None = None) -> None:
        """Mean over ranks of one gradient buffer through NVLink peer memory (after ``dp_attach``)."""
        self._check(self._lib.cql_dp_allreduce(self._h, int(which), self._torch_stream(stream)), "cql_dp_allreduce")

    @property
    def dp_fused(self) -> bool:
        """True when (after ``dp_attach``) the update kernels exchange the gradients themselves: ``update`` /
        ``update_batches`` are then data-parallel as they are and ``dp_allreduce`` is a no-op."""
        flag = C.c_int32(0)
        self._check(self._lib.cql_dp_mode(self._h, C.byref(flag)), "cql_dp_mode")
        return bool(flag.value)

    def dp_error(self) -> bool:
        flag = C.c_int32(0)
        self._check(self._lib.cql_dp_error(self._h, C.byref(flag)), "cql_dp_error")
        return bool(flag.value)

    def update_data_parallel(self, allreduce_mean: Callable[[int], None], stream: int | None = None,
                             uploaded_batch: bool = False) -> None:
        """One data-parallel update: the host averages the three gradient groups between phases.

        ``allreduce_mean(buffer_id)`` must average that device buffer over ranks on ``stream``
        (see ``parallel.GradAllReducer``).  Weights stay bit-identical across ranks because every
        rank applies the same Adam step to the same reduced gradient.
        """
        self.step_phase(4 if uploaded_batch else 0, stream)
        allreduce_mean(_lib.BUF_SCALAR_GRADS)
        self.step_phase(1, stream)
        allreduce_mean(_lib.BUF_CRITIC_GRADS)
        self.step_phase(2, stream)
        allreduce_mean(_lib.BUF_ACTOR_GRADS)
        self.step_phase(3, stream)

    def read_metrics(self) -> Dict[str, float]:
        import torch
        ptr, n = self.device_buffer(_lib.BUF_METRICS)
        t = torch.as_tensor(_DevView(ptr, n), device=f"cuda:{self.device}").cpu().numpy()
        return dict(zip(METRIC_NAMES, map(float, t[:6])))

    # ------------------------------------------------------------------ offline evaluation
    def offline_metrics(self, return_threshold: Optional[float] = None, stream: int | None = None) -> Dict[str, float]:
        """d3rlpy's offline scorers over the loaded one-step replay table (``cql_offline_eval``) as float64 sums and
        int counts (keys ``OFFLINE_SUM_KEYS``; ``offline_scores`` turns them into the metric values).  Episodes whose
        raw return is >= ``return_threshold`` (float32) feed the soft-OPC sums; None leaves them 0.  Weights, Adam
        state, step counter, table and captured update graphs are untouched."""
        thr = float("nan") if return_threshold is None else float(return_threshold)
        if return_threshold is not None and not np.isfinite(thr):
            raise ValueError("return_threshold must be a finite number or None")
        out = _lib.OfflineSums()
        self._check(self._lib.cql_offline_eval(self._h, thr, C.byref(out), stream), "cql_offline_eval")
        return {k: (int if k.startswith("n_") else float)(getattr(out, k)) for k in OFFLINE_SUM_KEYS}

    # ------------------------------------------------------------------ fitted Q evaluation
    def fqe_enable(self, target_update_interval: int) -> None:
        """FQE mode (``cql_fqe_enable``): from now on this engine trains its critics by FQE updates under the policy in
        its actor slot; the CQL update calls are refused."""
        self._check(self._lib.cql_fqe_enable(self._h, int(target_update_interval)), "cql_fqe_enable")

    def fqe_update(self, n_steps: int = 1, stream: int | None = None) -> float:
        """``n_steps`` sampled FQE updates (CUDA-graph replays) -> the last update's loss."""
        loss = np.zeros(1, dtype=np.float32)
        self._check(self._lib.cql_fqe_update(self._h, int(n_steps), _ptr(loss), stream), "cql_fqe_update")
        return float(loss[0])

    def fqe_update_rows(self, rows, want_grads: bool = False, stream: int | None = None):
        """One FQE update on [B, 8] table-format rows (raw) -> (loss, [n_critics] gradient dicts or None)."""
        rows = _f32(rows, (self.hp.batch_size, 8))
        loss = np.zeros(1, dtype=np.float32)
        C = self.hp.n_critics
        g = np.zeros(C * layout.NET_STRIDE, dtype=np.float32) if want_grads else None
        self._check(self._lib.cql_fqe_update_rows(self._h, _ptr(rows), _ptr(loss), _ptr(g), stream), "cql_fqe_update_rows")
        grads = None
        if want_grads:
            grads = [layout.unpack_net(g[c * layout.NET_STRIDE:(c + 1) * layout.NET_STRIDE], layout.CRITIC_IN,
                                       layout.CRITIC_OUT) for c in range(C)]
        return float(loss[0]), grads

    def copy_table_from(self, other: "CqlEngine", stream: int | None = None) -> None:
        """This engine's replay table := ``other``'s (device to device, ``cql_copy_table``); ``other`` is unchanged."""
        self._check(self._lib.cql_copy_table(self._h, other._h, stream), "cql_copy_table")

    # ------------------------------------------------------------------ scoring
    def score_topk(self, users, items, k: int, seen_indptr=None, seen_items=None, mode: str = "q"):
        """Top-``k`` unseen items per user.  -> (items [U,k] int32 (-1 pad), scores [U,k] float32 (-inf pad))"""
        if mode not in SCORE_MODES:
            raise ValueError(f"mode must be one of {sorted(SCORE_MODES)}")
        if not 1 <= int(k) <= _lib.MAX_TOPK:
            raise ValueError(f"k must be in 1..{_lib.MAX_TOPK}")
        users = np.ascontiguousarray(users, dtype=np.int32).reshape(-1)
        items = np.ascontiguousarray(items, dtype=np.int32).reshape(-1)
        U = users.size
        out_i = np.full((U, k), -1, dtype=np.int32)
        out_s = np.full((U, k), -np.inf, dtype=np.float32)
        if U == 0:
            return out_i, out_s
        if seen_indptr is not None:
            seen_indptr = np.ascontiguousarray(seen_indptr, dtype=np.int64)
            seen_items = np.ascontiguousarray(seen_items if seen_items is not None else [], dtype=np.int32)
            if seen_indptr.size < int(users.max()) + 2:
                raise ValueError("seen_indptr must cover every requested user id (+1)")
        self._check(self._lib.cql_score_topk(self._h, _ptr(users), U, _ptr(items), items.size, _ptr(seen_indptr),
                                             _ptr(seen_items) if seen_indptr is not None else None, int(k),
                                             SCORE_MODES[mode], _ptr(out_i), _ptr(out_s), None), "cql_score_topk")
        return out_i, out_s

    def score_pairs(self, users, items, mode: str = "q") -> np.ndarray:
        users = np.ascontiguousarray(users, dtype=np.int32).reshape(-1)
        items = np.ascontiguousarray(items, dtype=np.int32).reshape(-1)
        if users.size != items.size:
            raise ValueError("users and items must have the same length")
        out = np.empty(users.size, dtype=np.float32)
        self._check(self._lib.cql_score_pairs(self._h, _ptr(users), _ptr(items), users.size, SCORE_MODES[mode],
                                              _ptr(out), None), "cql_score_pairs")
        return out

    # ------------------------------------------------------------------ per-observation inference
    def predict_value(self, users, items, actions=None, with_std: bool = False, stream: int | None = None):
        """d3rlpy's ``predict_value(x, action, with_std)`` for ``x = (users[i], items[i])`` (``cql_predict_value``):
        float32 ``mean_c Q_c(x, a)`` per pair, and with ``with_std`` also the population std over the critics
        (``(mean, std)``).  ``actions`` are raw rating units (the action scaler maps them into Q); None = the greedy
        action ``tanh(mu(x))`` in network space, as ``score_pairs(mode="q")``.  The model is not modified."""
        u, i, a = inference_inputs(users, items, actions)
        mean = np.empty(u.size, dtype=np.float32)
        std = np.empty(u.size, dtype=np.float32) if with_std else None
        self._check(self._lib.cql_predict_value(self._h, _ptr(u), _ptr(i), _ptr(a), u.size, _ptr(mean), _ptr(std),
                                                stream), "cql_predict_value")
        return (mean, std) if with_std else mean

    def predict_action(self, users, items, stream: int | None = None) -> np.ndarray:
        """d3rlpy's ``predict(x)``: the greedy action ``tanh(mu(x))`` reverse-transformed into rating units (the value of
        ``score_pairs(mode="policy")``), float32 (``cql_sample_action`` with ``greedy = 1``)."""
        return self._sample(users, items, 1, stream)

    def sample_action(self, users, items, stream: int | None = None) -> np.ndarray:
        """d3rlpy's ``sample_action(x)``: ``reverse(tanh(mu + exp(clamp(logstd, -20, 2)) * eps))`` per pair, float32.
        ``eps`` is drawn from this engine's Philox stream numbered by its earlier ``sample_action`` calls (DESIGN.md
        section 1, "Inference"): consecutive calls differ, a fresh engine with the same seed repeats them.  The counter
        is not part of the update state; the model is not modified."""
        return self._sample(users, items, 0, stream)

    def _sample(self, users, items, greedy: int, stream) -> np.ndarray:
        u, i, _ = inference_inputs(users, items)
        out = np.empty(u.size, dtype=np.float32)
        self._check(self._lib.cql_sample_action(self._h, _ptr(u), _ptr(i), u.size, int(greedy), _ptr(out), stream),
                    "cql_sample_action")
        return out

    METRIC_NAMES = ("NDCG", "HitRate", "MAP", "MRR", "Precision", "Recall")

    def rank_metrics(self, rec_items, users, gt_indptr, gt_items, ks) -> dict:
        """Ranking metrics of a [U, k_rec] recommendation table (best first, -1 padded) against the ground truth
        CSR (over user id, items sorted per user), computed on the GPU.  Returns {metric: {k: mean over users}}
        with the reference's per-user definitions (replay/metrics/*.py ``_get_metric_value_by_user``)."""
        rec_items = np.ascontiguousarray(rec_items, dtype=np.int32)
        if rec_items.ndim != 2:
            raise ValueError("rec_items must be [n_users, k_rec]")
        users = np.ascontiguousarray(users, dtype=np.int32).reshape(-1)
        if users.size != rec_items.shape[0]:
            raise ValueError("one user id per row of rec_items")
        gt_indptr = np.ascontiguousarray(gt_indptr, dtype=np.int64)
        gt_items = np.ascontiguousarray(gt_items, dtype=np.int32)
        ks = [int(k) for k in (ks if hasattr(ks, "__iter__") else [ks])]
        if not ks or len(ks) > 8 or min(ks) < 1:
            raise ValueError("ks: 1 to 8 cut-offs, each >= 1")
        if users.size and gt_indptr.size < int(users.max()) + 2:
            raise ValueError("gt_indptr must cover every user id")
        ks_a = np.asarray(ks, dtype=np.int32)
        out = np.zeros((len(self.METRIC_NAMES), len(ks)), dtype=np.float64)
        self._check(self._lib.cql_rank_metrics(self._h, _ptr(rec_items), users.size, max(1, rec_items.shape[1]), _ptr(users),
                                               _ptr(gt_indptr), _ptr(gt_items), _ptr(ks_a), len(ks), _ptr(out), None),
                    "cql_rank_metrics")
        return {name: {k: float(out[m, q]) for q, k in enumerate(ks)} for m, name in enumerate(self.METRIC_NAMES)}

    def score_topk_device(self, users_t, items_t, k: int, seen_indptr_t=None, seen_items_t=None, mode: str = "q",
                          out_items=None, out_scores=None, stream: int | None = None):
        """HBM-resident variant: every argument is a cuda tensor (int32 ids, int64 indptr)."""
        import torch
        U = users_t.numel()
        if out_items is None:
            out_items = torch.empty((U, k), dtype=torch.int32, device=users_t.device)
        if out_scores is None:
            out_scores = torch.empty((U, k), dtype=torch.float32, device=users_t.device)
        stream = self._torch_stream(stream)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        self._check(self._lib.cql_score_topk_dev(self._h, p(users_t), U, p(items_t), items_t.numel(),
                                                 p(seen_indptr_t), p(seen_items_t), int(k), SCORE_MODES[mode],
                                                 p(out_items), p(out_scores), stream), "cql_score_topk_dev")
        return out_items, out_scores

    def seen_csr_device(self, log_users, log_items, n_users_dim: int, wanted=None, stream: int | None = None):
        """Seen-items CSR of a log built on the device (``cql_seen_csr``): int32 id columns (host, any order, duplicates
        allowed) -> (indptr int64 [n_users_dim + 1], seen int32 [n_seen]) as cuda tensors, per user ascending and
        de-duplicated.  ``wanted``: bool / uint8 mask over user ids -- only those users' rows are kept."""
        import torch
        lu = np.ascontiguousarray(log_users, dtype=np.int32).reshape(-1)
        li = np.ascontiguousarray(log_items, dtype=np.int32).reshape(-1)
        if lu.size != li.size:
            raise ValueError("log_users and log_items must have the same length")
        dev = torch.device("cuda", self.device)
        indptr = torch.empty(int(n_users_dim) + 1, dtype=torch.int64, device=dev)
        seen = torch.empty(max(1, lu.size), dtype=torch.int32, device=dev)
        w = None
        if wanted is not None:
            w = np.ascontiguousarray(wanted, dtype=np.uint8).reshape(-1)
            if w.size < int(n_users_dim):
                w = np.concatenate([w, np.zeros(int(n_users_dim) - w.size, dtype=np.uint8)])
        n_seen = C.c_int64(0)
        stream = self._torch_stream(stream)
        self._check(self._lib.cql_seen_csr(self._h, _ptr(lu) if lu.size else None, _ptr(li) if li.size else None, lu.size,
                                           int(n_users_dim), _ptr(w) if w is not None else None,
                                           C.c_void_p(indptr.data_ptr()), C.c_void_p(seen.data_ptr()), C.byref(n_seen), stream),
                    "cql_seen_csr")
        return indptr, seen[: n_seen.value]

    def topk_filter_device(self, scores_t, k: int, users_t=None, items_t=None, seen_indptr_t=None,
                           seen_items_t=None, stream: int | None = None):
        """Stand-alone top-k + lazy seen filter over a materialised cuda score matrix [U, I]."""
        import torch
        U, I = scores_t.shape
        out_items = torch.empty((U, k), dtype=torch.int32, device=scores_t.device)
        out_scores = torch.empty((U, k), dtype=torch.float32, device=scores_t.device)
        stream = self._torch_stream(stream)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        self._check(self._lib.cql_topk_filter_dev(self._h, p(scores_t), U, I, p(users_t), p(items_t),
                                                  p(seen_indptr_t), p(seen_items_t), int(k), p(out_items),
                                                  p(out_scores), stream), "cql_topk_filter_dev")
        return out_items, out_scores

    @property
    def launch_count(self) -> int:
        return int(self._lib.cql_launch_count(self._h))
