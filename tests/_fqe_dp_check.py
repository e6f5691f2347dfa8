"""torchrun --nproc-per-node 2 tests/_fqe_dp_check.py : ``FQE`` in a data-parallel job.  A replicated CQL model is
fitted on both ranks; each rank runs FQE on a device copy of the model's table and on the log (which FQE builds whole on
every rank), then prints a digest of its FQE state, its last loss and its offline metrics as JSON.  The caller
(tests/test_gpu_fqe.py) checks that both ranks give identical bits: every rank trains the same replica from the same
inputs."""
import hashlib
import json
import os
import sys

sys.path.insert(0, ".")
import torch
import torch.distributed as dist

from replay_cql_b200.models import CQL
from replay_cql_b200.ope import FQE
from replay_cql_b200.synthetic import make_log

rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
log = make_log("tiny")
m = CQL(shard_table=False, top_k=3, batch_size=64, seed=4, n_steps_per_epoch=6, scaler="standard")
m.fit(log)
out = {}
for name, arg in (("table", None), ("log", log)):
    f = FQE(m, n_critics=2, batch_size=32, target_update_interval=5)
    f.fit(arg, n_steps=23)
    out[name] = {"state": hashlib.sha256(f.engine.get_state().tobytes()).hexdigest(), "loss": f.last_loss,
                 "metrics": f.offline_metrics() if arg is None else None}
    f.close()
print(f"rank {rank} result {json.dumps(out, sort_keys=True)}", flush=True)
m.engine.close()
dist.destroy_process_group()
