"""A/B harness for the folded gradient reduction of the f16x3 update (k_adam_pack sums the backward's partials, the bwd1
kernels zero their own partial slots) against the separate k_reduce_grads_tc launches and memsets (CQL_NO_FOLD=1).

Arms alternate in fresh processes (the switch is read once per process).  Each run: HBM-resident updates at batch 1024
on a 20M-row synthetic table, best of three timed windows of `steps` graph-replayed updates, launches per update from
the library's counter; then the learner state, both Adam moments and the metrics after those updates are compared
bit for bit between the arms (same seeds, same number of updates).
python tests/_ab_fold.py [steps] [rounds] [out_dir]"""
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def child(steps: int, out: str) -> None:
    import torch
    from replay_cql_b200.engine import CqlEngine, CqlHyperParams
    eng = CqlEngine(CqlHyperParams(batch_size=1024, seed=12345, precision="f16x3"), device=0)
    eng.synth_table(20_000_263, 138_493, 26_744, seed=12345)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        eng.update(50, want_metrics=False, stream=st.cuda_stream)
        times = []
        l0 = eng.launch_count
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            eng.update(steps, want_metrics=False, stream=st.cuda_stream)
            e1.record(st)
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / steps * 1e3)
        launches = (eng.launch_count - l0) / (3 * steps)
    m, v, _ = eng.get_optimizer()
    np.savez(out, state=eng.get_state(), adam_m=m, adam_v=v,
             metrics=np.array(list(eng.read_metrics().values()), dtype=np.float32))
    print(json.dumps({"us": min(times), "windows": times, "launches_per_update": launches}), flush=True)
    eng.close()


def main() -> None:
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    out_dir = sys.argv[3] if len(sys.argv) > 3 else "."
    os.makedirs(out_dir, exist_ok=True)
    res = {"fold": [], "no_fold": []}
    for r in range(rounds):
        for arm in ("no_fold", "fold"):
            env = dict(os.environ)
            env.pop("CQL_NO_FOLD", None)
            if arm == "no_fold":
                env["CQL_NO_FOLD"] = "1"
            out = os.path.join(out_dir, f"ab_fold_{arm}_{r}.npz")
            p = subprocess.run([sys.executable, __file__, "--child", str(steps), out], env=env, capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit(f"{arm} run {r} failed:\n{p.stdout}\n{p.stderr}")
            d = json.loads(p.stdout.strip().splitlines()[-1])
            d["out"] = out
            res[arm].append(d)
            print(arm, r, "us/update %.2f" % d["us"], "launches/update %.2f" % d["launches_per_update"], flush=True)
    for arm, runs in res.items():
        us = sorted(d["us"] for d in runs)
        print(f"{arm}: median {us[len(us) // 2]:.2f} us/update, min {us[0]:.2f}, max {us[-1]:.2f}, "
              f"spread {us[-1] - us[0]:.2f}, launches/update {runs[0]['launches_per_update']:.2f}")
    a, b = np.load(res["no_fold"][0]["out"]), np.load(res["fold"][0]["out"])
    same = {k: bool(np.array_equal(a[k], b[k])) for k in a.files}
    print("bitwise equal after the same updates:", same)
    if not all(same.values()):
        sys.exit(1)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(int(sys.argv[2]), sys.argv[3])
    else:
        main()
