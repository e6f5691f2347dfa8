"""torchrun --nproc-per-node 2 tests/_offline_metrics_dp_check.py : ``CQL.offline_metrics`` data parallel.  A model fitted
on a replay table sharded by user evaluates its sharded table and a log (each rank its own user range); rank 0 also
evaluates the whole log on one engine holding the same networks.  Each rank prints its results as JSON; the caller
(tests/test_gpu_offline_metrics.py) checks that the ranks agree bit for bit and match the one-engine result within float64
reordering.  No action noise (``action_randomization_scale=0``): the sharded and the whole-log tables hold the same rows."""
import dataclasses
import json
import os
import sys

sys.path.insert(0, ".")
import torch
import torch.distributed as dist

from replay_cql_b200.engine import CqlEngine, offline_scores
from replay_cql_b200.mdp import build_mdp_on_device
from replay_cql_b200.models import CQL
from replay_cql_b200.synthetic import make_log

rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
log = make_log("tiny")
m = CQL(shard_table=True, top_k=3, batch_size=64, seed=4, n_steps_per_epoch=6, precision="fp32",
        action_randomization_scale=0.0, scaler="standard")
m.fit(log)
out = {"table": m.offline_metrics(return_threshold=2.0), "log": m.offline_metrics(log, return_threshold=2.0)}
if rank == 0:
    one = CqlEngine(dataclasses.replace(m.engine.hp, n_steps=1), device=local)
    one.set_state(m.engine.get_state())
    one.set_preprocessing(**m.engine.get_preprocessing())
    build_mdp_on_device(one, log, top_k=3, action_randomization_scale=0.0)
    out["single"] = offline_scores(one.offline_metrics(2.0), soft_opc=True)
    one.close()
print(f"rank {rank} result {json.dumps(out, sort_keys=True)}", flush=True)
m.engine.close()
dist.destroy_process_group()
