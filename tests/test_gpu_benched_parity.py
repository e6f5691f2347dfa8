"""GPU parity on the configuration that is BENCHED (VERDICT r01 item 1): the regime the product runs in.

* update: precision "f16x3" (the product / bench default) and "fp32", batch 1024 with raw ML-20M-range indices
  (users < 138 493, items < 26 744) and batch 8192 with stress-range indices (users < 1e7, items < 1e6) as
  observations -- six losses, EVERY updated tensor (actor, critics, both target sets, log_temp, log_alpha) and the
  Adam moments against the float32 CPU oracle at 1e-4 (max-abs / max-abs per tensor, as DESIGN.md states).
  The float64-budget rule (within 4x of the float32 oracle's own distance from the float64 oracle) is used ONLY
  where the float32 oracle itself is further than 1e-4 from the float64 one -- the test asserts that, so a budgeted
  comparison documents a spot where the CPU float32 path itself misses (SURVEY.md:289-291: raw indices as floats).
  Every step restarts from the oracle's state WITH non-trivial Adam moments, so the weights move by
  lr * m / (sqrt(v) + eps) with the gradient's magnitude in it, not just by its sign (first-step Adam).
* fused scorer (tc_score_kernel<SplitF16>): I = 26 744 items, U = 2048 users, the bench's heavy-tailed seen lists, against
  the brute-force per-user oracle on a user sample.
"""
import numpy as np
import pytest
import torch

from oracle import cql_oracle as O
from oracle import recs_oracle
from replay_cql_b200 import layout
from tests import helpers as Hp

pytestmark = pytest.mark.gpu
TOL = Hp.TOL


@pytest.mark.parametrize("precision", ["f16x3", "fp32"])
@pytest.mark.parametrize("B,n_users,n_items", [(1024, 138_493, 26_744), (8192, 10_000_000, 1_000_000)])
def test_update_on_benched_configuration(engine_factory, precision, B, n_users, n_items):
    cfg = O.OracleConfig()
    C = cfg.n_critics
    st = O.init_state(cfg, seed=7)
    eng = engine_factory(batch_size=B, precision=precision)
    budgeted = []
    for step in range(3):
        batch = Hp.make_batch(B, seed=500 + step, n_users=n_users, n_items=n_items, scale=1.0)
        noise = O.make_noise(B, cfg.n_action_samples, seed=600 + step)
        eng.set_state(Hp.oracle_state_to_flat(st))
        eng.set_optimizer(*Hp.oracle_adam_to_flat(st))
        st64 = O.cast_state(st, torch.float64)
        m64, _ = O.update(cfg, st64, {k: v.double() for k, v in batch.items()}, {k: v.double() for k, v in noise.items()})
        m32, _ = O.update(cfg, st, batch, noise)                       # st advances: next step starts from it
        mg, _ = eng.update_batch(Hp.batch_to_numpy(batch), Hp.noise_to_numpy(noise))
        for name in Hp.METRIC_NAMES:
            e32 = abs(mg[name] - m32[name])
            if e32 <= TOL * max(1.0, abs(m32[name])):
                continue
            d = abs(m32[name] - m64[name])
            assert d > TOL / 4 * max(1.0, abs(m64[name])), (step, name, mg[name], m32[name], m64[name])
            assert abs(mg[name] - m64[name]) <= max(TOL * max(1.0, abs(m64[name])), 4 * d), (step, name, mg[name], m32[name], m64[name])
            budgeted.append(((step, name), e32, abs(mg[name] - m64[name]), d))
        # every updated tensor, targets included
        g_t = Hp.state_tensors(eng.get_state(), C)
        r32 = Hp.state_tensors(Hp.oracle_state_to_flat(st), C)
        r64 = Hp.state_tensors(Hp.oracle_state_to_flat(O.cast_state(st64, torch.float32)), C)
        for tag in r32:
            Hp.check_f64_budget((step, "state") + tag, g_t[tag], r32[tag], r64[tag], budgeted)
        # Adam moments (the gradients of this step are in them: m = 0.9 m' + 0.1 g) and the step counter
        gm, gv, gstep = eng.get_optimizer()
        om, ov, ostep = Hp.oracle_adam_to_flat(st)
        om64, ov64, _ = Hp.oracle_adam_to_flat(O.cast_state(st64, torch.float32))
        assert gstep == ostep == step + 1
        for name, g_, o_, o64_ in (("adam_m", gm, om, om64), ("adam_v", gv, ov, ov64)):
            gt, ot, ot64 = Hp.state_tensors(g_, C), Hp.state_tensors(o_, C), Hp.state_tensors(o64_, C)
            for tag in ot:
                if tag[0].startswith("targ"):
                    continue
                Hp.check_f64_budget((step, name) + tag, gt[tag], ot[tag], ot64[tag], budgeted)
    print(f"\n[{precision} B={B}] comparisons that needed the float64 budget: {len(budgeted)}")
    for b in budgeted:
        print("   ", b)


def test_fused_scorer_at_baseline_item_count(engine_factory):
    """tc_score_kernel<SplitF16> on the BASELINE shape: all 26 744 items, 2048 users, the ML-20M-shaped log's real
    heavy-tailed seen lists (a few users have thousands of seen items), k = 10 -- scores within 1e-5 of max|Q| and
    lists identical up to (near-)ties against the brute-force oracle on 24 of the users (first, last, the three
    longest seen lists, and a random draw)."""
    from replay_cql_b200.mdp import seen_csr
    from replay_cql_b200.synthetic import SHAPES, make_log
    shape = SHAPES["ml20m"]
    log = make_log("ml20m", seed=12345)                               # the bench's log (20 000 263 rows)
    cfg = O.OracleConfig()
    flat = layout.init_state(cfg.n_critics, 11)
    st = Hp.flat_to_oracle_state(flat, cfg)
    eng = engine_factory(batch_size=64, precision="f16x3")
    eng.set_state(flat)
    present = np.sort(log["user_idx"].unique())
    rng = np.random.default_rng(1)
    users = np.sort(rng.choice(present, size=2048, replace=False)).astype(np.int32)
    items = np.arange(shape["n_items"], dtype=np.int32)
    sub = log[log["user_idx"].isin(users)]
    indptr, seen = seen_csr(sub, int(users.max()) + 1)
    k = 10
    ti, ts = eng.score_topk(users, items, k, indptr, seen)
    lens = indptr[users + 1] - indptr[users]
    pick = {0, users.size - 1, *np.argsort(lens)[-3:].tolist(), *rng.choice(users.size, size=19, replace=False).tolist()}
    pick = np.array(sorted(pick))
    seen_sets = {int(u): set(seen[indptr[u]:indptr[u + 1]].tolist()) for u in users[pick]}
    ri, rs = recs_oracle.brute_force_topk(lambda obs: O.relevance(st, torch.from_numpy(obs), "q").numpy(),
                                          users[pick], items, seen_sets, k)
    scale = max(1.0, float(np.max(np.abs(rs))))
    assert np.max(np.abs(ts[pick] - rs)) <= 1e-5 * scale, (np.max(np.abs(ts[pick] - rs)), scale)
    for row, (a, b) in enumerate(zip(ti[pick], ri)):
        for c in np.nonzero(a != b)[0]:                               # a swap is only legal between near-equal scores
            assert abs(rs[row, c] - ts[pick][row, c]) <= 1e-5 * scale
            assert a[c] in b or np.any(np.abs(rs[row] - ts[pick][row, c]) <= 1e-5 * scale)
    # no recommended item is a seen one, for ALL 2048 users
    for r, u in enumerate(users):
        s = seen[indptr[u]:indptr[u + 1]]
        assert not np.isin(ti[r], s).any(), int(u)
    assert int(lens.max()) > 1000                                     # the heavy tail is really in the sample
