"""torchrun --nproc-per-node 2 tests/_large_ensemble_dp_check.py : one f16x3 update at (C, n) = (10, 32) on two GPUs with
the fused peer exchange, from the float32 oracle's state with non-trivial Adam moments.  Each rank takes its half of a
128-row minibatch.  Checks: the replicas are bit-identical, and each matches the float32 oracle run on the same halves with
its gradients averaged over the two ranks (grad_hook over a gloo group) within the update gate 1e-4.  Prints dp-ok."""
import os
import sys

sys.path.insert(0, '.')
import numpy as np
import torch
import torch.distributed as dist

from oracle import cql_oracle as O
from replay_cql_b200.engine import CqlEngine, CqlHyperParams
from replay_cql_b200.parallel import PeerGradExchange
from tests import helpers as Hp

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
cpu = dist.new_group(backend="gloo")
B, C, n = 64, 10, 32                                   # per rank
cfg = O.OracleConfig(n_critics=C, n_action_samples=n)
st = O.init_state(cfg, seed=7)
O.update(cfg, st, Hp.make_batch(64, seed=17, scale=1e-3), O.make_noise(64, n, seed=18))   # Adam warm-up
batch, noise = Hp.make_batch(world * B, seed=1, scale=1e-3), O.make_noise(world * B, n, seed=2)
lo, hi = rank * B, (rank + 1) * B
shard = {k: v[lo:hi] for k, v in batch.items()}
nshard = {k: v[lo:hi] for k, v in noise.items()}

eng = CqlEngine(CqlHyperParams(batch_size=B, n_critics=C, n_action_samples=n, precision="f16x3"), device=local,
                rank=rank, world_size=world)
eng.set_state(Hp.oracle_state_to_flat(st))
eng.set_optimizer(*Hp.oracle_adam_to_flat(st))
ex = PeerGradExchange(eng)
assert ex.fused, "the fused peer exchange is not available"
m_gpu, _ = eng.update_batch(Hp.batch_to_numpy(shard), Hp.noise_to_numpy(nshard))
torch.cuda.synchronize()
got = eng.get_state()
assert not eng.dp_error(), "peer exchange wait timed out"


def hook(gs):
    for g in gs:
        dist.all_reduce(g, group=cpu)
        g /= world
    return gs


O.update(cfg, st, shard, nshard, grad_hook=hook)
ref = Hp.oracle_state_to_flat(st)
err = Hp.rel_err(got, ref)
both = [torch.empty(got.size, dtype=torch.float32) for _ in range(world)]
dist.all_gather(both, torch.from_numpy(got), group=cpu)
identical = all(torch.equal(both[0], t) for t in both)
print(f"rank {rank}: replicas identical: {identical}; state rel err vs oracle {err:.3e}; metrics {m_gpu}", flush=True)
assert identical
assert err <= 1e-4, err
eng.close()
dist.barrier(group=cpu)
dist.destroy_process_group()
print("dp-ok", flush=True)
