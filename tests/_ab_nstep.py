"""Measurements of n-step TD returns (cql_set_n_steps) on one GPU.

1. Update: HBM-resident updates at batch 1024 (f16x3) on a 20M-row synthetic table, n_steps 1 against 3, the arms
   alternating in fresh processes; best of three timed windows of `steps` graph-replayed updates per run, in us/update.
2. Table build: the ML-20M-shaped log through CqlEngine.build_mdp_on_device (which returns after a synchronise) at
   n_steps 1, 3 and 10, best of three after a warm-up build; and the n-step expansion kernel (k_nstep_rows) alone, its
   device time from torch.profiler over the same builds, as bytes per second (32 B read + 32 B written per row, plus
   the n_steps - 1 halo rows each 256-row block reads again) against a measured copy peak.
The GPU's name, power limit and maximum SM clock are read in the same run.
python tests/_ab_nstep.py [steps] [rounds]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

COPY_PEAK_GBS = 6472.0        # device-to-device copy on a B200 (DESIGN.md section 3)


def child_update(n_steps: int, steps: int) -> None:
    import torch
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=12345, precision="f16x3", n_steps=n_steps), device=0)
    eng.synth_table(20_000_263, 138_493, 26_744, seed=12345)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        eng.update(50, want_metrics=False, stream=st.cuda_stream)
        times = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            eng.update(steps, want_metrics=False, stream=st.cuda_stream)
            e1.record(st)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / steps * 1e3)
    print(json.dumps({"us": min(times), "windows": times}), flush=True)
    eng.close()


def table_build() -> None:
    import torch
    from torch.profiler import ProfilerActivity, profile
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    from replay_cql_b200.synthetic import make_log_arrays
    a = make_log_arrays("ml20m")
    n = a["user_idx"].size
    cols = (a["user_idx"], a["item_idx"], a["timestamp"], a["relevance"])
    out = {}
    # copy peak of this run: device-to-device copy of a table-sized buffer
    src = torch.empty(n * 8, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    out["copy_gbs"] = 2 * src.numel() * 4 * 20 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del src, dst
    for ns in (1, 3, 10):
        eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=12345, precision="f16x3", n_steps=ns), device=0)
        eng.build_mdp_on_device(*cols)
        wall = []
        for _ in range(3):
            t0 = time.perf_counter()
            eng.build_mdp_on_device(*cols)
            wall.append(time.perf_counter() - t0)
        rec = {"build_s": min(wall), "build_windows_s": wall}
        if ns > 1:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    eng.build_mdp_on_device(*cols)
                torch.cuda.synchronize()
            k = [e.device_time_total for e in prof.key_averages() if "k_nstep_rows" in e.key]
            cnt = [e.count for e in prof.key_averages() if "k_nstep_rows" in e.key]
            us = k[0] / cnt[0]
            blocks = (n + 255) // 256
            byts = 64 * n + 32 * blocks * (ns - 1)
            rec.update(expand_us=us, expand_gbs=byts / (us * 1e-6) / 1e9,
                       expand_share_of_copy_peak=byts / (us * 1e-6) / 1e9 / COPY_PEAK_GBS)
        out[f"n_steps={ns}"] = rec
        eng.close()
    print(json.dumps(out), flush=True)


def gpu_info() -> str:
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def main() -> None:
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    print("gpu:", gpu_info(), flush=True)
    res = {1: [], 3: []}
    for r in range(rounds):
        for ns in (1, 3):
            p = subprocess.run([sys.executable, __file__, "--update", str(ns), str(steps)], capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit(f"n_steps={ns} run {r} failed:\n{p.stdout}\n{p.stderr}")
            d = json.loads(p.stdout.strip().splitlines()[-1])
            res[ns].append(d["us"])
            print(f"update n_steps={ns} run {r}: {d['us']:.2f} us/update", flush=True)
    for ns, us in res.items():
        us = sorted(us)
        print(f"update n_steps={ns}: median {us[len(us) // 2]:.2f} us/update, min {us[0]:.2f}, max {us[-1]:.2f}")
    p = subprocess.run([sys.executable, __file__, "--build"], capture_output=True, text=True)
    if p.returncode != 0:
        sys.exit(f"table build failed:\n{p.stdout}\n{p.stderr}")
    print("table build:", p.stdout.strip().splitlines()[-1])
    print("gpu:", gpu_info(), flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--update":
        child_update(int(sys.argv[2]), int(sys.argv[3]))
    elif len(sys.argv) > 1 and sys.argv[1] == "--build":
        table_build()
    else:
        main()
