"""Attribution of the oracle-gate misses of tests/test_gpu_scalers.py::test_scaled_update_batch_matches_oracle.

For every (prep, precision, shape) case of that test, both steps run through tests/test_gpu_update_shapes.py's
_compare_step with every gate recorded instead of asserted, so that all misses of a step are listed.  For each net with
a miss, the float64 oracle's hidden pre-activations of the step are scanned for the ones nearest to zero (relative to
their row's largest), and those ReLU masks are toggled in the float64 oracle one at a time; a toggle is kept when it
brings the oracle's gradient of that net closer to the GPU's.  Printed: the misses, the kept toggles with their
pre-activation ratio, and the GPU's error on the missed tensors against the plain and the toggled float64 oracle.
python tests/_diag_scaler_gates.py"""
import sys

sys.path.insert(0, ".")
import numpy as np
import torch

from oracle import cql_oracle as O
from replay_cql_b200.engine import CqlEngine, CqlHyperParams
from tests import helpers as Hp
from tests import scaler_oracle as S
from tests import test_gpu_scalers as T
from tests import test_gpu_update_shapes as U

_orig_mlp = O.mlp
_REC = None          # list of (call, label, layer, z) while recording
_TOG = set()         # {(call, layer, row, unit)} masks to toggle
_CALL = [0]
_LABELS = {}


def _label(net):
    return _LABELS.get(float(net["W1"].reshape(-1)[0]), "in%d(updated)" % net["W1"].shape[1])


def _mlp(net, x):
    c = _CALL[0]
    _CALL[0] += 1
    h = x
    for layer, (w, b) in enumerate(((net["W1"], net["b1"]), (net["W2"], net["b2"]))):
        z = h @ w.T + b
        if _REC is not None:
            _REC.append((c, _label(net), layer, z.detach().clone()))
        flips = [(r, u) for (cc, ll, r, u) in _TOG if cc == c and ll == layer]
        h = torch.relu(z)
        if flips:
            m = torch.zeros_like(z, dtype=torch.bool)
            for r, u in flips:
                m[r, u] = True
            h = torch.where(m, torch.where(z > 0, z * 0, z), h)
    return h @ net["W3"].T + net["b3"]


O.mlp = _mlp


def _run64(step):
    _CALL[0] = 0
    st64 = O.cast_state(step.st0, torch.float64)
    m, g = O.update(step.cfg, st64, U._as64(step.batch), U._as64(step.noise), want_grads=True)
    return g, O.cast_state(st64, torch.float32)


def _net_grad(g, net):
    return g["actor"] if net[0] == "actor" else g["critics"][net[1]]


def case(prep, precision, B, C, n):
    global _REC
    P = T.PREP if prep == "standard" else T.PREP_MM
    cfg = O.OracleConfig(n_critics=C, n_action_samples=n)
    st = O.init_state(cfg, seed=7)
    O.update(cfg, st, Hp.make_batch(64, seed=17, scale=1e-3), O.make_noise(64, n, seed=18))
    eng = CqlEngine(CqlHyperParams(batch_size=B, n_critics=C, n_action_samples=n, precision=precision), device=0)
    eng.set_preprocessing(**P)
    for s in range(2):
        raw = Hp.make_batch(B, seed=5000 + 10 * B + s, term_frac=0.2)
        step = U._Step(cfg, st, S.transform_batch(P, raw), O.make_noise(B, n, seed=6000 + 10 * B + s))
        misses = []
        orig = Hp.check_f64_budget

        def rec(tag, *a, **k):
            try:
                orig(tag, *a, **k)
            except AssertionError as e:
                misses.append(e.args[0])
        Hp.check_f64_budget = rec
        try:
            U._compare_step(T._RawBatchEngine(eng, raw, P), step, precision, (B, C, n), s, [])
        except AssertionError as e:
            misses.append(("non-tensor gate", str(e)[:200]))
        finally:
            Hp.check_f64_budget = orig
        print(f"[{prep} {precision} B={B} C={C} n={n} step {s}] misses: {len(misses)}", flush=True)
        for m in misses:
            print("   ", m, flush=True)
        if not misses:
            continue
        # GPU gradients of this step (same start, same inputs)
        U._start(eng, step)
        _, g_gpu = eng.update_batch(Hp.batch_to_numpy(raw), Hp.noise_to_numpy(step.noise), want_grads=True)
        nets = []
        for m in misses:
            tag = m[0] if isinstance(m, tuple) and isinstance(m[0], tuple) else ()
            if len(tag) > 2 and tag[1] in ("grad", "state", "adam_m", "adam_v"):
                net = ("actor",) if tag[2] in ("actor", "targ_actor") else \
                    ("critic", tag[3]) if tag[2] in ("critic", "critics", "targ_critics") else None
                if net is not None and net not in nets:
                    nets.append(net)
        for k, v in st0_labels(step).items():
            _LABELS[k] = v
        _REC = []
        g64, _ = _run64(step)
        rec_calls = _REC
        _REC = None
        cands = []
        for c, lab, layer, z in rec_calls:
            rowmax = z.abs().max(dim=1, keepdim=True).values.clamp_min(1e-300)
            ratio = (z.abs() / rowmax).numpy()
            for r, u in zip(*np.unravel_index(np.argsort(ratio, axis=None)[:4], ratio.shape)):
                cands.append((float(ratio[r, u]), c, lab, layer, int(r), int(u)))
        cands.sort()
        cands = cands[:24]
        for net in nets:
            keys = ("W1", "b1", "W2", "b2", "W3")

            def err(gr):
                return {k: float(np.max(np.abs(_net_grad(g_gpu, net)[k] - _net_grad(gr, net)[k].numpy()))
                                 / np.max(np.abs(_net_grad(gr, net)[k].numpy()))) for k in keys}
            base = err(g64)
            kept = []
            _TOG.clear()
            best = base
            for cand in cands:
                _TOG.add((cand[1], cand[3], cand[4], cand[5]))
                gt, _ = _run64(step)
                e = err(gt)
                if max(e.values()) < 0.5 * max(best.values()):
                    kept.append(cand)
                    best = e
                else:
                    _TOG.discard((cand[1], cand[3], cand[4], cand[5]))
            print(f"    net {net}: GPU vs float64 oracle, grad max-norm rel err " +
                  " ".join(f"{k} {v:.3e}" for k, v in base.items()), flush=True)
            for cand in kept:
                print(f"      toggled: call {cand[1]} ({cand[2]}), layer {cand[3] + 1}, row {cand[4]}, unit {cand[5]}, "
                      f"|pre-activation| {cand[0]:.2e} of the row's largest", flush=True)
            if kept:
                gt, st_t = _run64(step)
                print("      GPU vs toggled float64 oracle: " + " ".join(f"{k} {v:.3e}" for k, v in err(gt).items()),
                      flush=True)
                sg = Hp.state_tensors(eng.get_state(), C)
                so = Hp.state_tensors(Hp.oracle_state_to_flat(st_t), C)
                sp = Hp.state_tensors(step.r64()[2], C)
                for t in so:
                    if (net[0] == "actor" and t[0] == "actor") or (net[0] == "critic" and t[0] == "critics" and t[1] == net[1]):
                        print(f"      state {t}: vs float64 {Hp.rel_err(sg[t], sp[t]):.3e}, vs toggled {Hp.rel_err(sg[t], so[t]):.3e}",
                              flush=True)
            _TOG.clear()
    eng.close()


def st0_labels(step):
    st = step.st0
    out = {float(st["actor"]["W1"].reshape(-1)[0]): "actor", float(st["targ_actor"]["W1"].reshape(-1)[0]): "targ_actor"}
    for i, c in enumerate(st["critics"]):
        out[float(c["W1"].reshape(-1)[0])] = f"critic{i}"
    for i, c in enumerate(st["targ_critics"]):
        out.setdefault(float(c["W1"].reshape(-1)[0]), f"targ_critic{i}")
    return out


if __name__ == "__main__":
    for prep in ("standard", "min_max"):
        for precision in ("fp32", "tf32x3", "f16x3"):
            for B, C, n in T.GATES:
                case(prep, precision, B, C, n)
