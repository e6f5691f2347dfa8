"""torchrun --nproc-per-node 2 tests/_scalers_dp_check.py : a data-parallel fit with the three scalers on a replay table
sharded by user.  Each rank prints its fitted preprocessing parameters and a digest of its final learner state; the
caller (tests/test_gpu_scalers.py) checks that both ranks print the same."""
import hashlib
import json
import os
import sys

sys.path.insert(0, ".")
import torch
import torch.distributed as dist

from replay_cql_b200.models import CQL
from replay_cql_b200.synthetic import make_log

rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
m = CQL(scaler="standard", action_scaler="min_max", reward_scaler="standard", shard_table=True, top_k=3, batch_size=64,
        seed=4, n_steps_per_epoch=6)
m.fit(make_log("tiny"))
prep = json.dumps(m.engine.get_preprocessing(), sort_keys=True)
digest = hashlib.sha256(m.engine.get_state().tobytes()).hexdigest()
print(f"rank {rank} prep {prep} state {digest}", flush=True)
m.engine.close()
dist.destroy_process_group()
