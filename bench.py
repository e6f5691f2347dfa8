#!/usr/bin/env python
"""bench.py -- CQL updates/s (batch 1024) and users scored top-10/s on the ML-20M-shaped synthetic log.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun ... bench.py --gpus N ...        (N > 1: one rank per GPU, NCCL)

One JSON line on stdout (rank 0).  A *step* is one CQL update (temp -> alpha -> critic ->
actor -> Polyak) on one batch of 1024 transitions per GPU.  ``value`` = batch-1024 updates
per second over all ranks with the replay table resident in HBM and sampling on the GPU;
``e2e`` = the same update through the host-buffer C-ABI call (`cql_update_batch`: pinned
minibatch H2D + metrics D2H every step).  ``scoring`` carries the second half of the
BASELINE.json metric (users scored to top-10 per second, seen filter on).
``--impl reference`` times the CPU oracle (eager PyTorch restatement of d3rlpy's update --
d3rlpy/pyspark cannot be installed here, DESIGN.md) on the host cores for the same config.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True    # the benchmark writes nothing into the source tree (it may be read-only)

BATCH = 1024
K_TOP = 10
WORKLOAD = "ml20m-train"          # BASELINE.json configs[2]: 138 493 users x 26 744 items, 20 000 263 rows
SCORE_WARM_USERS = 2048           # users of the untimed warm-up scoring pass (the timed pass scores ALL users, configs[3])
FLOP_PER_ROW = 2 * (3 * 256 + 256 * 256 + 256)   # f_c = 133 120 (SURVEY 8d)
FLOP_PER_UPDATE_PER_B = 269 * FLOP_PER_ROW       # 269 forward-equivalent rows per batch element
FLOP_PER_PAIR = 3 * FLOP_PER_ROW                 # 2 critics + actor = 399 360
DTYPES = {"fp32": "f32", "tf32x3": "f32 (tf32x3: tensor-core 3-term split, fp32 accumulate, 1e-4 parity-gated)",
          "f16x3": "f32 (f16x3: tensor-core fp16 hi/lo 3-term split with exact power-of-two row scales, fp32 accumulate, 1e-4 parity-gated)",
          "bf16": "bf16 (fp32 accumulate; non-parity variant)"}
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from one `ncu --set full` capture
# (profiles/r01_tc_fwd_ts_ncu_summary.txt, profiles/r02_big3_ncu_summary.txt); null where no capture exists for that variant
KERNEL_TRAFFIC = {"fp32": None, "tf32x3": 3.226112e6 + 11.174144e6, "f16x3": 2.134784e6 + 16.243456e6, "bf16": None}
TRAFFIC_SOURCE = {"fp32": None, "tf32x3": "ncu --set full capture profiles/r01_tc_fwd_ts_ncu_summary.txt (not measured in this run)",
                  "f16x3": "ncu --set full capture profiles/r02_big3_ncu_summary.txt: tc_fwd_h2_kernel<3,1> dram read 2.13 MB + write 16.24 MB "
                           "(not measured in this run; algorithmic: 2.0 MB of input rows + 65 MB of stored H2, most of which stays in L2)", "bf16": None}
KERNEL_NAMES = {"fp32": "mlp_fwd_kernel<3,1> (critic forward, FP32 CUDA-core path)",
                "tf32x3": "tc_fwd_ts_kernel<3,1> (critic forward: tcgen05 kind::tf32 3-term split, A operand in TMEM)",
                "f16x3": "tc_fwd_h2_kernel<3,1> (critic forward on CTA pairs: tcgen05 cta_group::2 kind::f16, fp16 hi/lo 3-term split, A operand in TMEM)",
                "bf16": "tc_fwd_kernel<bf16,3,1> (critic forward, tcgen05 kind::f16)"}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_first(self, timeout: float = 5.0):
        """Block until nvidia-smi has delivered a sample (it can take seconds to start when 8 ranks launch it at once):
        a timed region shorter than the sampling period otherwise ends before the first line arrives."""
        t0 = time.time()
        while self.proc is not None and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t_from: float | None = None, t_to: float | None = None):
        """Summary of the samples taken in [t_from, t_to] (host clock); all samples if the window holds none."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        n0, t0 = len(self.lines), time.time()
        while len(self.lines) == n0 and time.time() - t0 < 1.0:      # one more sample after the region
            time.sleep(0.02)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def summarise(rows):
            sm, mx, reasons = [], [], set()
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(names, f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons

        win = [r for r in self.lines if (t_from is None or r[0] >= t_from) and (t_to is None or r[0] <= t_to + 0.12)]
        sm, mx, reasons = summarise(win)
        window = "timed region"
        if not sm:                       # region shorter than the sampling period: report the neighbouring samples
            sm, mx, reasons = summarise(self.lines)
            window = "around the timed region"
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def build_workload(log_rows: int | None = None):
    from replay_cql_b200.synthetic import make_log, SHAPES
    log = make_log("ml20m", seed=12345, n_rows=log_rows)
    return log, SHAPES["ml20m"]


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_update_rate(steps: int, warmup: int, threads: int | None = None):
    """Oracle updates/s at B=1024 on the host cores (bounded sample: `steps` updates)."""
    import torch
    from oracle import cql_oracle as O
    from tests import helpers as Hp
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = O.OracleConfig()
    st = O.init_state(cfg, seed=7)
    batches = [Hp.make_batch(BATCH, seed=s, n_users=138_493, n_items=26_744) for s in range(4)]
    noises = [O.make_noise(BATCH, cfg.n_action_samples, seed=50 + s) for s in range(4)]
    for s in range(warmup):
        O.update(cfg, st, batches[s % 4], noises[s % 4])
    t0 = time.perf_counter()
    for s in range(steps):
        O.update(cfg, st, batches[s % 4], noises[s % 4])
    dt = time.perf_counter() - t0
    return steps / dt, dt, threads


def cpu_scoring_rate(n_users: int, n_items: int = 26_744, threads: int | None = None):
    """Per-user loop in the style of replay/models/neuromf.py:394-438 (users/s, k=10, filter seen)."""
    import torch
    from oracle import cql_oracle as O
    from oracle import recs_oracle
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    st = O.init_state(O.OracleConfig(), seed=7)
    rng = np.random.default_rng(0)
    users = rng.choice(138_493, size=n_users, replace=False).astype(np.int32)
    items = np.arange(n_items, dtype=np.int32)
    seen = {int(u): set(rng.choice(n_items, size=144, replace=False).tolist()) for u in users}
    t0 = time.perf_counter()
    recs_oracle.brute_force_topk(lambda obs: O.relevance(st, torch.from_numpy(obs), "q").numpy(), users, items, seen, K_TOP)
    dt = time.perf_counter() - t0
    return n_users / dt, dt, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 200))      # bounded sample: ~0.04-0.2 s per oracle update
    rate, dt, threads = cpu_update_rate(steps, max(1, min(args.warmup, 5)))
    srate, sdt, _ = cpu_scoring_rate(8)
    line = {
        "impl": "reference", "metric": "CQL updates/sec (batch 1024)", "value": rate, "unit": "updates/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "users": 138_493, "items": 26_744, "rows": 20_000_263,
                   "batch_per_gpu": BATCH, "global_batch": BATCH, "parallelism": "cpu", "grad_exchange": "none",
                   "hidden": 256, "n_critics": 2, "n_action_samples": 10, "precision": "fp32 (PyTorch CPU)",
                   "note": "CPU oracle = eager PyTorch restatement of d3rlpy CQL._update (d3rlpy and Spark are not "
                           "installable here); minibatches of the same shape and id ranges pre-built in host memory "
                           "(the cost of an update does not depend on the log it was sampled from)"},
        "cpu_baseline": {"value": rate, "unit": "updates/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} updates at batch 1024 after warm-up, torch threads={threads}"},
        "e2e": {"value": rate, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "scoring": {"metric": "users scored top-10/sec", "value": srate, "unit": "users/s",
                    "sample": f"8 users x 26744 items, per-user loop, filter_seen, {sdt:.1f} s"},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from replay_cql_b200 import _lib
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    from replay_cql_b200.mdp import seen_csr
    from replay_cql_b200.parallel import GradAllReducer, shard_range

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.gpus != world and rank == 0 and world > 1:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    pk, pk_kind = peaks()

    from replay_cql_b200.mdp import build_mdp, build_mdp_on_device
    log, shape = build_workload(args.rows)
    eng = CqlEngine(CqlHyperParams(batch_size=BATCH, seed=12345, precision=args.precision), device=local_rank,
                    rank=rank, world_size=world)
    import pyarrow as pa
    from replay_cql_b200.mdp import ingest_log
    log_arrow = pa.Table.from_pandas(log, preserve_index=False)        # the log as Arrow columns (what Spark's Arrow path hands over)
    ingest_log(eng, log_arrow.slice(0, 100_000), top_k=K_TOP)          # warm-up (CUB temp, allocator, pinned ring)
    mdp_times = []
    for _ in range(3):                                                 # Arrow buffers -> pinned ring -> HBM, sorts, replay table
        t0 = time.perf_counter()
        ingest_log(eng, log_arrow, top_k=K_TOP, action_randomization_scale=1e-3)
        mdp_times.append(time.perf_counter() - t0)
    mdp_gpu_s = float(np.median(mdp_times))
    n_rows = eng.n_transitions
    mdp_host = None
    if rank == 0 and world == 1 and not args.no_cpu:                    # host builder on a bounded 2M-row sample
        sub = log.iloc[:2_000_000]
        t0 = time.perf_counter()
        build_mdp(sub, top_k=K_TOP, seed=12345)
        mdp_host = {"rows": len(sub), "seconds": time.perf_counter() - t0}
    stream = torch.cuda.Stream(device=dev)
    sh = stream.cuda_stream

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    from replay_cql_b200.parallel import DataParallelStepper, make_grad_exchange
    # N > 1: gradient exchange over NVLink peer memory.  With the f16x3 kernels it is FUSED into the update (the reduce
    # kernels publish, the Adam kernels read the peers' buffers): the library's own step graph is data-parallel as it is.
    # Otherwise (NCCL fallback / other precisions) the four phases + exchanges are captured as one graph by the stepper.
    reducer = make_grad_exchange(eng) if world > 1 else None
    fused_dp = world > 1 and bool(getattr(reducer, "fused", False))
    stepper = DataParallelStepper(eng, reducer=reducer) if (world > 1 and not fused_dp) else None
    if stepper is not None:
        stream = stepper.stream
        sh = stream.cuda_stream
    stepper_e2e = None
    if stepper is not None:        # same stream and exchange; the captured step reads the uploaded minibatch
        stepper_e2e = DataParallelStepper(eng, uploaded_batch=True, reducer=reducer)
        stepper_e2e.stream = stream
    if world > 1:
        dist.barrier()

    def do_steps(k):
        if stepper is None:
            with torch.cuda.stream(stream):
                eng.update(k, want_metrics=False, stream=sh)
        else:
            stepper.run(k)

    # ---- HBM-resident updates/s ----
    clocks = ClockSampler(local_rank)      # started before the warm-up so that it is already sampling in the timed region
    clocks.start()
    do_steps(max(3, args.warmup))
    clocks.wait_first()
    barrier()
    l0 = eng.launch_count
    r0 = stepper.replayed_steps if stepper is not None else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_w0 = time.time()
    e0.record(stream)
    do_steps(args.steps)
    e1.record(stream)
    barrier()
    t_w1 = time.time()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = eng.launch_count - l0           # eager / library-graph launches are counted by the library itself
    if stepper is not None:                    # graph replays: kernels captured per update x replayed updates
        launches += stepper.launches_per_step * (stepper.replayed_steps - r0)
    clk = clocks.stop(t_w0, t_w1)
    value = world * args.steps / (ms / 1e3)
    dump = {}                      # --dump-outputs (rank 0): name -> array
    dumping = bool(args.dump_outputs) and rank == 0
    if dumping:                    # the learner after the last timed update, read back outside the timed region
        adam_m, adam_v, _ = eng.get_optimizer()
        dump.update(update_state=eng.get_state(), update_adam_m=adam_m, update_adam_v=adam_v,
                    update_metrics=np.array(list(eng.read_metrics().values()), dtype=np.float32))

    # ---- per-kernel durations (events inside one real update), rank 0 reporting ----
    timings = [eng.timed_update(stream=sh) for _ in range(5)][1:]
    tk = {k: float(np.mean([t[k] for t in timings])) for k in timings[0]}
    n3 = 30
    fwd_rows = 2 * (BATCH * n3 + BATCH * (n3 + 1) + BATCH)        # alpha + critic + target rows, 2 nets
    fwd_flop = fwd_rows * FLOP_PER_ROW
    achieved = fwd_flop / (tk["critic_fwd"] / 1e3) / 1e12
    peak_tf = pk.get("bf16_tflops_sustained", 1400.0)

    # ---- e2e: host minibatch in, metrics out, every step ----
    rng = np.random.default_rng(rank)
    n_e2e = max(10, min(args.steps, 500))
    pool = []
    for _ in range(8):          # host minibatches: rows read back from the replay table
        rows = eng.sample_rows(BATCH, idx=rng.integers(0, n_rows, BATCH)).cpu().numpy()
        pool.append({"obs": np.ascontiguousarray(rows[:, 0:2]), "act": np.ascontiguousarray(rows[:, 2:3]),
                     "rew": np.ascontiguousarray(rows[:, 3:4]), "next_obs": np.ascontiguousarray(rows[:, 4:6]),
                     "term": np.ascontiguousarray(rows[:, 6:7])})
    def e2e_step(i):
        if stepper is None:
            eng.update_batch(pool[i % 8])
        else:   # host minibatch in, the data-parallel step (gradient exchanges included) as one graph, metrics out
            with torch.cuda.stream(stream):
                eng.upload_batch(pool[i % 8], stream=sh)
                stepper_e2e.run(1)
                eng.read_metrics()
    if stepper is None:
        # the host loop of a trainer that owns its minibatches: every step's batch goes host -> pinned ring -> device and
        # its six metrics come back; the library pipelines copies and steps (cql_update_batches).  N > 1 (fused exchange):
        # every rank runs the same call on its own minibatches, the kernels average the gradients across the ranks.
        stacked = {k: np.stack([pool[i % 8][k] for i in range(n_e2e)]) for k in pool[0]}
        eng.update_batches([pool[i] for i in range(3)])
        barrier()
        t0 = time.perf_counter()
        e2e_metrics = eng.update_batches(stacked)
        torch.cuda.synchronize(dev)
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        assert len(e2e_metrics) == n_e2e and all(np.isfinite(m["critic_loss"]) for m in e2e_metrics)
        if reducer is not None:
            reducer.check()
    else:
        for i in range(3):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(n_e2e):
            e2e_step(i)
        torch.cuda.synchronize(dev)
        e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * n_e2e / e2e_s

    # ---- scoring (BASELINE configs[3]): ALL users sharded over ranks, all items, seen filter, k=10 ----
    n_score = shape["n_users"]
    users_all = np.arange(n_score, dtype=np.int32)
    lo, hi = shard_range(n_score, rank, world)
    users = users_all[lo:hi]
    items = np.arange(shape["n_items"], dtype=np.int32)
    lo_row, hi_row = np.searchsorted(log["user_idx"].to_numpy(), [lo, hi])      # the generator's log is user-major
    indptr, seen = seen_csr(log.iloc[lo_row:hi_row], shape["n_users"])
    n_warm = min(SCORE_WARM_USERS, users.size)
    with torch.cuda.stream(stream):
        d_users = torch.from_numpy(users).to(dev)
        d_items = torch.from_numpy(items).to(dev)
        d_ptr = torch.from_numpy(indptr).to(dev)
        d_seen = torch.from_numpy(seen).to(dev)
        oi = torch.empty((users.size, K_TOP), dtype=torch.int32, device=dev)
        osc = torch.empty((users.size, K_TOP), dtype=torch.float32, device=dev)
        eng.score_topk_device(d_users[:64], d_items, K_TOP, d_ptr, d_seen, out_items=oi[:64], out_scores=osc[:64], stream=sh)
        eng.score_topk_device(d_users[:n_warm], d_items, K_TOP, d_ptr, d_seen, out_items=oi[:n_warm], out_scores=osc[:n_warm], stream=sh)
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l1 = eng.launch_count
    SCORE_REPS = 1
    score_clocks = ClockSampler(local_rank)      # seconds of sustained tensor + CUDA-core load: the power cap may bite
    score_clocks.start()
    score_clocks.wait_first()
    s0.record(stream)
    with torch.cuda.stream(stream):
        for _ in range(SCORE_REPS):
            eng.score_topk_device(d_users, d_items, K_TOP, d_ptr, d_seen, out_items=oi, out_scores=osc, stream=sh)
    s1.record(stream)
    barrier()
    score_clk = score_clocks.stop()
    score_ms_local = s0.elapsed_time(s1) / SCORE_REPS
    score_ms = max_over_ranks(score_ms_local)
    score_ms_ranks = [score_ms_local]
    if world > 1:
        tl = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(tl, torch.tensor([score_ms_local], dtype=torch.float64, device=dev))
        score_ms_ranks = [float(t.item()) for t in tl]
    score_launches = (eng.launch_count - l1) // SCORE_REPS
    users_per_s = n_score / (score_ms / 1e3)
    top_dev = oi.cpu().numpy()
    assert (top_dev[:, 0] >= 0).all() and not np.isin(top_dev[0], seen[indptr[users[0]]:indptr[users[0] + 1]]).any()
    if dumping:                    # item ids < 2**24: exact in float32
        dump.update(score_top_items=top_dev.astype(np.float32), score_top_scores=osc.cpu().numpy())
    eng.score_topk(users[:n_warm], items, K_TOP, indptr, seen)         # warm-up of the host-buffer entry (scratch allocation)
    barrier()
    t0 = time.perf_counter()
    top_host, _ = eng.score_topk(users, items, K_TOP, indptr, seen)   # host ids + CSR in, top-k out: every user of this rank
    score_e2e_s = max_over_ranks(time.perf_counter() - t0)
    assert np.array_equal(top_host, top_dev)
    pairs = float(users.size) * shape["n_items"]
    score_tf = pairs * FLOP_PER_PAIR / (score_ms / 1e3) / 1e12

    # ---- stand-alone top-k + lazy seen filter over a MATERIALISED score matrix (HBM-bound: 4 B/pair read) ----
    TOPK_ROWS = 8192                                                 # 8192 rows x 26744 fp32 = 876 MB >> L2
    sc_mat = torch.randn((TOPK_ROWS, shape["n_items"]), dtype=torch.float32, device=dev)
    tk_users = d_users[torch.randint(0, users.size, (TOPK_ROWS,), device=dev)]
    with torch.cuda.stream(stream):
        eng.topk_filter_device(sc_mat, K_TOP, users_t=tk_users, items_t=d_items, seen_indptr_t=d_ptr, seen_items_t=d_seen, stream=sh)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(5):
            eng.topk_filter_device(sc_mat, K_TOP, users_t=tk_users, items_t=d_items, seen_indptr_t=d_ptr, seen_items_t=d_seen, stream=sh)
        f1.record(stream)
    torch.cuda.synchronize(dev)
    topk_ms = f0.elapsed_time(f1) / 5
    topk_gbs = sc_mat.numel() * 4 / (topk_ms / 1e3) / 1e9
    del sc_mat

    # ---- K1 stand-alone gather sweep (HBM random gather, 36 B/row algorithmic) ----
    cnt = 1 << 20
    out = torch.empty((cnt, 8), dtype=torch.float32, device=dev)
    with torch.cuda.stream(stream):
        eng.sample_rows(cnt, pos=0, out=out, stream=sh)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for r in range(10):
            eng.sample_rows(cnt, pos=(r + 1) * cnt, out=out, stream=sh)
        g1.record(stream)
    torch.cuda.synchronize(dev)
    gather_gbs = 10 * cnt * 64 / (g0.elapsed_time(g1) / 1e3) / 1e9    # 32 B read + 32 B written per row

    # ---- the product path: replay.models.CQL().fit(log) / .predict(log, 10) through the Recommender API (pandas in / out) ----
    product = None
    if world == 1:
        from replay_cql_b200.models import CQL
        n_fit = max(50, min(args.steps, 2000))
        model = CQL(n_epochs=1, n_steps_per_epoch=n_fit, batch_size=BATCH, seed=12345)      # every default incl. precision
        t0 = time.perf_counter()
        model.fit(log)                                   # fit_users/fit_items, MDP build on the GPU, n_fit updates
        torch.cuda.synchronize(dev)
        fit_s = time.perf_counter() - t0
        pu = log[["user_idx"]].drop_duplicates().iloc[:: max(1, shape["n_users"] // 4096)]
        t0 = time.perf_counter()
        recs = model.predict(log, K_TOP, users=pu, filter_seen_items=True)
        pred_s = time.perf_counter() - t0
        assert len(recs) == len(pu) * K_TOP
        product = {"api": "replay_cql_b200.models.CQL(n_epochs=1, n_steps_per_epoch=%d).fit(log); .predict(log, 10, users=<%d users>)" % (n_fit, len(pu)),
                   "precision": model.precision, "fit_seconds": fit_s, "fit_updates": n_fit,
                   "fit_note": "wall clock of the whole call: distinct users/items (pandas), host columns -> HBM + GPU MDP build, updates",
                   "predict_seconds": pred_s, "predict_users": int(len(pu)), "predict_users_per_s": len(pu) / pred_s,
                   "predict_note": "wall clock incl. pandas cold filter, seen CSR build from the 20M-row log, fused scoring, result frame"}
        model.engine.close()

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            rate, dt, threads = cpu_update_rate(40, 3)
            cpu = {"value": rate, "unit": "updates/s", "cores": threads, "kind": "port",
                   "sample": f"40 oracle updates at batch 1024 ({dt:.1f} s), torch threads={threads}"}
        line = {
            "metric": "CQL updates/sec (batch 1024)", "value": value, "unit": "updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPES[args.precision], "data": "synthetic",
            "config": {"workload": WORKLOAD, "users": shape["n_users"], "items": shape["n_items"],
                       "rows": int(n_rows), "batch_per_gpu": BATCH, "global_batch": BATCH * world,
                       "parallelism": f"dp{world}",
                       "grad_exchange": ("none" if world == 1 else
                                         "NVLink peer memory, fused into the update kernels (reduce kernels publish + signal, Adam kernels read the "
                                         "peers' buffers: no exchange launch; csrc/dp_peer.cuh)" if fused_dp else
                                         {"PeerGradExchange": "NVLink peer-memory one-shot all-reduce kernel (csrc/dp_peer.cuh), 3 per update",
                                          "GradAllReducer": "NCCL all-reduce, 3 per update"}.get(type(reducer).__name__, type(reducer).__name__)),
                       "hidden": 256, "n_critics": 2, "n_action_samples": 10,
                       "precision": args.precision,
                       "l2": "inputs larger than L2: 640 MB replay table, fresh random gather every step; "
                             "weights/activations are the step-to-step state of the algorithm"},
            "e2e": {"value": e2e_value, "unit": "updates/s", "h2d_bytes_per_step": BATCH * 32,
                    "d2h_bytes_per_step": 32, "steps": n_e2e, "api": "cql_update_batches (host minibatches in, per-step metrics out; every step's H2D and D2H copies ride on the library's own copy streams while the previous step computes)" if stepper is None else
                           "cql_upload_batch + the data-parallel step as one CUDA graph (cql_step_phase x4 with the gradient exchange between phases) + metrics D2H"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": KERNEL_NAMES[args.precision],
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "peak_source": f"bf16_tflops_sustained ({pk_kind})", "traffic": KERNEL_TRAFFIC[args.precision],
                         "traffic_source": TRAFFIC_SOURCE[args.precision],
                         "flop_per_launch": fwd_flop, "ms_per_launch": tk["critic_fwd"],
                         "update_tflops": value / world * BATCH * FLOP_PER_UPDATE_PER_B / 1e12},
            "kernel_ms": tk,
            "kernel_ms_note": "one eager update with CUDA events between the launches and programmatic dependent launch "
                              "switched OFF (with PDL a kernel's prologue overlaps its predecessor and events no longer "
                              "separate them); 'update' here is therefore longer than ms_per_step (graph replay, PDL on)",
            "cpu_baseline": cpu,
            "product_path": product,
            "scoring": {"metric": "users scored top-10/sec", "value": users_per_s, "unit": "users/s",
                        "users": int(n_score), "users_note": "every user of the ML-20M shape, sharded over the ranks (configs[3])",
                        "items": shape["n_items"], "k": K_TOP, "filter_seen": True,
                        "ms": score_ms, "ms_per_rank": score_ms_ranks, "tflops": score_tf * world, "frac_of_peak": score_tf / peak_tf,
                        "gpu_launches": int(score_launches), "clocks": score_clk,
                        "e2e": {"value": n_score / score_e2e_s, "unit": "users/s",
                                "h2d_bytes": int(users.nbytes + items.nbytes + indptr.nbytes + seen.nbytes),
                                "d2h_bytes": int(users.size * K_TOP * 8), "api": "cql_score_topk (host ids + CSR in, top-k out)"}},
            "topk_filter": {"metric": "stand-alone top-10 + seen filter over materialised fp32 scores", "value": topk_gbs,
                            "unit": "GB/s", "rows": int(TOPK_ROWS), "cols": shape["n_items"], "ms": topk_ms,
                            "bound": "hbm", "peak": pk.get("hbm_gbs", 6650.0), "frac": topk_gbs / pk.get("hbm_gbs", 6650.0),
                            "bytes_per_pair": 4},
            "mdp_build": {"metric": "ingestion: pyarrow.Table columns (pageable host memory) -> pinned ring -> replay table (HBM)",
                          "rows": int(n_rows), "gpu_seconds": mdp_gpu_s, "gpu_seconds_runs": mdp_times, "rows_per_s": n_rows / mdp_gpu_s,
                          "host_bytes": int(n_rows) * 24, "host_numpy_sample": mdp_host},
            "sampler": {"metric": "replay gather", "value": gather_gbs, "unit": "GB/s", "rows": cnt,
                        "frac_of_hbm": gather_gbs / pk.get("hbm_gbs", 6650.0)},
        }
        if dumping:
            assert sum(a.nbytes for a in dump.values()) <= 64 << 20
            out_dir = Path(args.dump_outputs)
            out_dir.mkdir(parents=True, exist_ok=True)
            for name, a in dump.items():
                np.save(out_dir / f"{name}.npy", a)
        print(json.dumps(line), flush=True)
    # teardown: graphs first (NCCL communicators must not be destroyed under a live captured graph); a watchdog
    # guarantees the process exits even if a collective teardown stalls -- the JSON line is already out
    sys.stdout.flush()
    wd = threading.Timer(45.0, lambda: os._exit(0))
    wd.daemon = True
    wd.start()
    if stepper is not None:
        stepper.graph = None
        stepper_e2e.graph = None
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()             # no rank frees its staging buffers while a peer's kernel may still read them
    eng.close()
    if world > 1:
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass
    wd.cancel()


# ----------------------------------------------------------------------------- BASELINE configs[0,1]: ML-1M fit + predict
def run_ml1m(args):
    """fit + predict wall clock on the ML-1M-shaped log (6 040 x 3 706, 1 000 209 rows) through the Recommender API with
    default hyper-parameters -- the `fit_pred_time` protocol of the reference's leaderboard
    (docs/pages/useful_data/res_1m.csv:1-15) -- next to the CPU path (oracle updates + per-user scoring loop in the style of
    replay/models/neuromf.py:394-438), which is timed on a bounded sample and extrapolated (stated)."""
    import torch
    from replay_cql_b200.models import CQL
    from replay_cql_b200.synthetic import make_log, SHAPES
    shape = SHAPES["ml1m"]
    log = make_log("ml1m", seed=12345)
    dev = torch.device("cuda", 0)
    warm = CQL(n_epochs=1, n_steps_per_epoch=3, batch_size=BATCH)      # context / allocator warm-up (fit returns None, as the reference's)
    warm.fit(log.iloc[:50_000])
    warm.engine.close()
    # The whole measurement is ~0.4 s of wall clock on a shared host: it is repeated (a fresh model each time) and the
    # MEDIAN run is reported, all runs listed -- single runs on one box ranged 0.44 .. 1.9 s with the GPU time unchanged.
    clocks = ClockSampler(0); clocks.start(); clocks.wait_first()
    runs = []
    for rep in range(5):
        model = CQL(n_epochs=1, batch_size=BATCH, seed=12345)
        t0 = time.perf_counter()
        model.fit(log)
        torch.cuda.synchronize(dev)
        fit_s = time.perf_counter() - t0
        t1 = time.perf_counter()
        recs = model.predict(log, K_TOP, filter_seen_items=True)
        pred_s = time.perf_counter() - t1
        n_updates = model.engine.get_optimizer()[2]
        launches = model.engine.launch_count
        assert recs.groupby("user_idx").size().max() <= K_TOP and recs["user_idx"].nunique() == shape["n_users"]
        model.engine.close()
        runs.append((fit_s + pred_s, fit_s, pred_s))
    clk = clocks.stop()
    runs_sorted = sorted(runs)
    _, fit_s, pred_s = runs_sorted[len(runs) // 2]
    cpu = None
    if not args.no_cpu:
        rate, dt, threads = cpu_update_rate(40, 3)
        srate, sdt, _ = cpu_scoring_rate(24, n_items=shape["n_items"])
        cpu = {"value": n_updates / rate + shape["n_users"] / srate, "unit": "s (extrapolated fit+predict)", "cores": threads, "kind": "port",
               "sample": f"40 oracle updates at batch 1024 ({dt:.1f} s) -> {rate:.1f} updates/s x {n_updates} updates; "
                         f"24 users x {shape['n_items']} items per-user loop ({sdt:.1f} s) -> {srate:.2f} users/s x {shape['n_users']} users"}
    line = {"metric": "CQL fit+predict wall clock, ML-1M shape (fit_pred_time)", "value": fit_s + pred_s, "unit": "s", "n_gpus": 1,
            "steps": int(n_updates), "warmup": 3, "ms_per_step": 1e3 * fit_s / max(1, n_updates), "higher_is_better": False,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPES[model.precision], "data": "synthetic",
            "config": {"workload": "ml1m-fit-predict", "users": shape["n_users"], "items": shape["n_items"], "rows": shape["n_rows"],
                       "batch_per_gpu": BATCH, "n_epochs": 1, "k": K_TOP, "filter_seen_items": True, "precision": model.precision,
                       "api": "replay_cql_b200.models.CQL().fit(log); .predict(log, 10)"},
            "fit_seconds": fit_s, "predict_seconds": pred_s, "runs_fit_predict_seconds": [[round(f, 4), round(p_, 4)] for _, f, p_ in runs],
            "runs_note": "5 runs, a fresh model each; value = the median run", "gpu_launches": int(launches), "clocks": clk, "cpu_baseline": cpu,
            "e2e": {"value": fit_s + pred_s, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "the whole measurement IS end to end: pandas frames in, pandas frame out"}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- BASELINE configs[4]: stress shape, scaled
def run_stress(args):
    """10M users x 1M items, 1e9-row replay table (32 GB) resident in HBM, batch 8192, the bf16 tensor-core critic variant
    (stated tolerance 2e-2 on losses, not a parity mode).  The table is generated ON the device (`cql_synth_table`): the
    log's 24 GB of columns are not worth moving through the host.  Scoring: a stated user sample x all 1M items."""
    import torch
    import torch.distributed as dist
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    from replay_cql_b200.parallel import DataParallelStepper, shard_range
    from replay_cql_b200.synthetic import SHAPES
    world = int(os.environ.get("WORLD_SIZE", 1)); rank = int(os.environ.get("RANK", 0)); local_rank = int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    shape = dict(SHAPES["stress"]); shape["n_rows"] = args.stress_rows
    B = 8192
    prec = args.stress_precision
    eng = CqlEngine(CqlHyperParams(batch_size=B, seed=12345, precision=prec), device=local_rank, rank=rank, world_size=world)
    t0 = time.perf_counter()
    eng.synth_table(shape["n_rows"], shape["n_users"], shape["n_items"], seed=12345)
    synth_s = time.perf_counter() - t0
    stepper = DataParallelStepper(eng) if world > 1 else None
    stream = stepper.stream if stepper else torch.cuda.Stream(device=dev)
    def do_steps(k):
        if stepper: stepper.run(k)
        else:
            with torch.cuda.stream(stream): eng.update(k, want_metrics=False, stream=stream.cuda_stream)
    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1: dist.barrier()
    steps = max(20, min(args.steps, 300))
    clocks = ClockSampler(local_rank); clocks.start()
    do_steps(max(3, min(args.warmup, 10))); clocks.wait_first(); barrier()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); do_steps(steps); e1.record(stream); barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    clk = clocks.stop()
    m = eng.read_metrics()
    assert all(np.isfinite(v) for v in m.values()), m
    n_su = 64                                           # users scored per rank: 64 x 1e6 pairs each
    rng = np.random.default_rng(7 + rank)
    users = np.sort(rng.choice(shape["n_users"], size=n_su, replace=False)).astype(np.int32)
    items = np.arange(shape["n_items"], dtype=np.int32)
    eng.score_topk(users[:4], items, K_TOP)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    ti, _ = eng.score_topk(users, items, K_TOP)         # host ids in, top-k out (no seen filter: the synthetic table has no log)
    score_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([score_s], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); score_s = float(t.item())
    if rank == 0:
        pk, pk_kind = peaks()
        value = world * steps / (ms / 1e3)
        line = {"metric": "CQL updates/sec (batch 8192, stress shape)", "value": value, "unit": "updates/s", "n_gpus": world, "steps": steps,
                "warmup": max(3, min(args.warmup, 10)), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPES[prec], "data": "synthetic (generated on the device, cql_synth_table)",
                "config": {"workload": "stress", "users": shape["n_users"], "items": shape["n_items"], "rows": int(shape["n_rows"]),
                           "table_gb": shape["n_rows"] * 32 / 1e9, "table": "replicated on every rank", "batch_per_gpu": B, "global_batch": B * world,
                           "parallelism": f"dp{world}", "precision": prec, "table_generation_seconds": synth_s,
                           "l2": "32 GB replay table >> L2, fresh random gather every step"},
                "gpu_launches": int(eng.launch_count - l0) + (stepper.launches_per_step * stepper.replayed_steps if stepper else 0),
                "clocks": clk, "update_tflops": value / world * B * FLOP_PER_UPDATE_PER_B / 1e12,
                "update_frac_of_bf16_sustained": value / world * B * FLOP_PER_UPDATE_PER_B / 1e12 / pk.get("bf16_tflops_sustained", 1400.0),
                "last_metrics": m,
                "scoring": {"metric": "users scored top-10/sec over 1e6 items", "value": world * n_su / score_s, "unit": "users/s",
                            "users": world * n_su, "sample": f"{n_su} random users per rank x all 1 000 000 items (of 10M users: a bounded sample)",
                            "tflops": world * n_su * shape["n_items"] * FLOP_PER_PAIR / score_s / 1e12, "api": "cql_score_topk (host ids in, top-k out)"},
                "e2e": None, "cpu_baseline": None}
        print(json.dumps(line), flush=True)
    if stepper: stepper.graph = None
    torch.cuda.synchronize(dev)
    eng.close()
    if world > 1:
        try:
            dist.barrier(); dist.destroy_process_group()
        except Exception:
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--rows", type=int, default=None, help="override the log size (debugging)")
    ap.add_argument("--precision", choices=["fp32", "tf32x3", "f16x3", "bf16"], default="f16x3",
                    help="hidden-layer contraction: fp32 = CUDA-core FMA; tf32x3 = tcgen05 3-term split (FP32-grade, "
                         "default); bf16 = tcgen05 bf16 operands (non-parity variant)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workload", choices=["ml20m", "ml1m", "stress"], default="ml20m",
                    help="ml20m = the headline line (BASELINE configs[2,3]); ml1m = fit+predict wall clock beside the CPU "
                         "per-user path (configs[0,1]); stress = 1e9-row table, batch 8192, bf16 (configs[4], scaled scoring)")
    ap.add_argument("--stress-rows", type=int, default=1_000_000_000)
    ap.add_argument("--stress-precision", choices=["fp32", "tf32x3", "f16x3", "bf16"], default="bf16",
                    help="stress workload: bf16 = the variant BASELINE configs[4] names; f16x3 = the FP32-grade product path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="ml20m workload: write what the timed paths computed as DIR/<name>.npy (float32, rank 0): the learner "
                         "state, Adam moments and metrics after the last timed update, and the top-10 items and scores of the "
                         "timed scoring pass (rank 0's users).  Inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "ml20m"):
        ap.error("--dump-outputs is implemented for --impl ours --workload ml20m")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "ml1m":
        run_ml1m(args)
    elif args.workload == "stress":
        run_stress(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
