"""Measurements of the scalers (cql_set_preprocessing, cql_get_table_stats) on one GPU.

1. Update: HBM-resident updates at batch 1024 (f16x3) on a 20M-row synthetic table, without preprocessing against
   all three scalers, the arms alternating in fresh processes; best of three timed windows of `steps` graph-replayed
   updates per run, in us/update.
2. Scoring: users/s of score_topk_device (k = 10, 26,744 items, 4,096 users, no seen filter) with and without an
   observation scaler (and the action scaler, policy mode), best of three timed windows after a warm-up call.
3. Table build: the ML-20M-shaped log through CqlEngine.build_mdp_on_device (which returns after a synchronise), best
   of three after a warm-up build, in this tree (with the statistics pass) and, when given, in the tree of the parent
   commit, the arms alternating in fresh processes.
The GPU's name, power limit and maximum SM clock are read in the same run.
python tests/_ab_scalers.py [steps] [rounds] [parent_tree]"""
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)

PREP = {"scaler": {"type": "standard", "mean": [69246.0, 4000.0], "std": [40000.0, 6000.0]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]},
        "reward_scaler": {"type": "standard", "mean": [0.05], "std": [0.2]}}


def child_update(scaled: bool, steps: int) -> None:
    import torch
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=12345, precision="f16x3"), device=0)
    eng.synth_table(20_000_263, 138_493, 26_744, seed=12345)
    if scaled:
        eng.set_preprocessing(**PREP)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        l0 = eng.launch_count
        eng.update(50, want_metrics=False, stream=st.cuda_stream)
        launches = (eng.launch_count - l0) // 50
        times = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            eng.update(steps, want_metrics=False, stream=st.cuda_stream)
            e1.record(st)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / steps * 1e3)
    print(json.dumps({"us": min(times), "windows": times, "launches_per_update": launches}), flush=True)
    eng.close()


def scoring() -> None:
    import torch
    from replay_cql_b200 import layout
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=12345, precision="f16x3"), device=0)
    eng.set_state(layout.init_state(2, 5))
    users = torch.arange(4096, dtype=torch.int32, device="cuda") * 33
    items = torch.arange(26_744, dtype=torch.int32, device="cuda")
    out = {}
    for name, prep, mode in (("plain_q", {}, "q"), ("obs_scaler_q", {"scaler": PREP["scaler"]}, "q"),
                             ("plain_policy", {}, "policy"),
                             ("obs_action_scaler_policy", {"scaler": PREP["scaler"],
                                                           "action_scaler": PREP["action_scaler"]}, "policy")):
        eng.set_preprocessing(**prep)
        eng.score_topk_device(users, items, 10, mode=mode)
        torch.cuda.synchronize()
        best = []
        for _ in range(3):
            t0 = time.perf_counter()
            eng.score_topk_device(users, items, 10, mode=mode)
            torch.cuda.synchronize()
            best.append(time.perf_counter() - t0)
        out[name] = {"users_per_s": users.numel() / min(best), "windows_s": best}
    print(json.dumps(out), flush=True)
    eng.close()


def child_build() -> None:
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    from replay_cql_b200.synthetic import make_log_arrays
    a = make_log_arrays("ml20m")
    cols = (a["user_idx"], a["item_idx"], a["timestamp"], a["relevance"])
    eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=12345, precision="f16x3"), device=0)
    eng.build_mdp_on_device(*cols)
    wall = []
    for _ in range(3):
        t0 = time.perf_counter()
        eng.build_mdp_on_device(*cols)
        wall.append(time.perf_counter() - t0)
    print(json.dumps({"build_s": min(wall), "windows_s": wall}), flush=True)
    eng.close()


def gpu_info() -> str:
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def _run(args, cwd=HERE):
    p = subprocess.run([sys.executable, os.path.abspath(__file__), *args], capture_output=True, text=True, cwd=cwd,
                       env=dict(os.environ, PYTHONPATH=cwd))
    if p.returncode != 0:
        sys.exit(f"{args} failed:\n{p.stdout}\n{p.stderr}")
    return json.loads(p.stdout.strip().splitlines()[-1])


def main() -> None:
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    parent = os.path.abspath(sys.argv[3]) if len(sys.argv) > 3 else None
    print("gpu:", gpu_info(), flush=True)
    res = {"plain": [], "scalers": []}
    for r in range(rounds):
        for arm in res:
            d = _run(["--update", arm, str(steps)])
            res[arm].append(d["us"])
            print(f"update {arm} run {r}: {d['us']:.2f} us/update, {d['launches_per_update']} launches", flush=True)
    for arm, us in res.items():
        us = sorted(us)
        print(f"update {arm}: median {us[len(us) // 2]:.2f} us/update, min {us[0]:.2f}, max {us[-1]:.2f}")
    print("scoring:", json.dumps(_run(["--score"])), flush=True)
    builds = {"this": []} if parent is None else {"this": [], "parent": []}
    for r in range(rounds):
        for arm in builds:
            # the parent tree runs this tree's child code against its own package (cwd / PYTHONPATH)
            d = _run(["--build"], cwd=HERE if arm == "this" else parent)
            builds[arm].append(d["build_s"])
            print(f"build {arm} run {r}: {d['build_s'] * 1e3:.1f} ms", flush=True)
    print("gpu:", gpu_info(), flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--update":
        child_update(sys.argv[2] == "scalers", int(sys.argv[3]))
    elif len(sys.argv) > 1 and sys.argv[1] == "--score":
        scoring()
    elif len(sys.argv) > 1 and sys.argv[1] == "--build":
        sys.path.insert(0, os.getcwd())
        child_build()
    else:
        main()
