"""CPU: the host reference of the update's sampling and noise (tests/sampling_oracle.py) pinned on its own.

Philox against Random123's published known answers, the epoch permutation as a bijection at every small size and
around every power of two up to 2^22, the stream positions' epoch and data-parallel properties, and the statistics of
the noise an update draws.  The GPU side is compared with this reference in tests/test_gpu_sampling.py.
"""
import numpy as np
import pytest
from scipy import stats

from tests import sampling_oracle as S


# ---------------------------------------------------------------- Philox4x32-10
# Random123 kat_vectors, philox4x32_10: (counter; key) -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(w) for w in S.philox4x32_raw(ctr, key)) == want


def test_philox_word_order():
    """(seed, stream, index) map to key (seed lo, seed hi) and counter (index lo, index hi, stream lo, stream hi)."""
    seed, stream, index = 0x0123456789ABCDEF, 0x1122334455667788, 0x99AABBCCDDEEFF00
    got = S.philox4x32_10(seed, stream, np.array([index], dtype=np.uint64))
    want = S.philox4x32_raw((0xDDEEFF00, 0x99AABBCC, 0x55667788, 0x11223344), (0x89ABCDEF, 0x01234567))
    assert [int(w[0]) for w in got] == [int(w) for w in want]


def test_u01_float32_edges():
    """((x >> 8) + 0.5) * 2^-24 rounded in float32: the sum rounds to even from 2^23 on, and the top 256 inputs give
    exactly 1.0, so a uniform draw 2 u - 1 lies in (-1, 1] and a Gaussian draw's u1 = 1 gives 0."""
    x = np.array([0, 255, 256, 0x7FFFFF00, 0x80000000, 0x80000100, 0xFFFFFEFF, 0xFFFFFF00, 0xFFFFFFFF], dtype=np.uint32)
    u = S.u01(x)
    assert u.dtype == np.float32
    want = [2.0 ** -25, 2.0 ** -25, 1.5 * 2.0 ** -24, 0.5 - 2.0 ** -25, 0.5, 0.5 + 2.0 ** -23, 1 - 2.0 ** -23, 1.0, 1.0]
    assert u.astype(np.float64).tolist() == want
    assert S.box_muller(np.array([0xFFFFFFFF], np.uint32), np.array([0], np.uint32))[0] == 0.0


# ---------------------------------------------------------------- epoch permutation
def _key(n):
    return int(S.epoch_key(12345 + n, n % 5)[0])


def _is_bijection(n):
    out = S.feistel_perm(np.arange(n, dtype=np.uint64), n, _key(n))
    return out.size == n and np.array_equal(np.sort(out), np.arange(n, dtype=np.uint64))


def test_feistel_is_a_bijection_for_every_small_n():
    bad = [n for n in range(1, 4097) if not _is_bijection(n)]
    assert not bad, bad[:20]


@pytest.mark.parametrize("k", range(1, 23))
def test_feistel_is_a_bijection_around_powers_of_two(k):
    for n in (2 ** k - 1, 2 ** k, 2 ** k + 1):
        assert _is_bijection(n), n


def test_feistel_depends_on_the_key():
    x = np.arange(1000, dtype=np.uint64)
    a, b = S.feistel_perm(x, 1000, 1), S.feistel_perm(x, 1000, 2)
    assert np.mean(a != b) > 0.95


SEEDS = [0, 9, 2 ** 40 + 3]


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("n,chunk", [(1, 1), (7, 3), (37, 37), (100, 37), (1000, 64), (4737 * 2 + 17, 4737)])
def test_stream_epochs_are_permutations(seed, n, chunk):
    """Each epoch is n_eff = n - n mod chunk distinct rows (d3rlpy drops the last partial minibatch); consecutive epochs
    draw different permutations; an epoch starts at position epoch * n_eff."""
    n_eff = n - n % chunk
    eps = [S.stream_index(np.arange(e * n_eff, (e + 1) * n_eff), n, chunk, seed) for e in range(3)]
    for e, idx in enumerate(eps):
        assert np.unique(idx).size == n_eff and idx.min() >= 0 and idx.max() < n, e
        assert np.array_equal(idx, S.feistel_perm(np.arange(n_eff), n, S.epoch_key(seed, e)).astype(np.int64))
    if n_eff > 3:
        assert not np.array_equal(eps[0], eps[1]) and not np.array_equal(eps[1], eps[2])


@pytest.mark.parametrize("n,chunk", [(1, 5), (4, 5), (36, 37), (37 * 8 - 1, 37 * 8)])
def test_stream_with_fewer_rows_than_a_chunk(n, chunk):
    """n < chunk: n_eff = n, so an epoch is every row once and a minibatch spans epochs."""
    p = np.arange(3 * n)
    idx = S.stream_index(p, n, chunk, 9)
    for e in range(3):
        assert np.array_equal(np.sort(idx[e * n:(e + 1) * n]), np.arange(n))


@pytest.mark.parametrize("W", [2, 8])
@pytest.mark.parametrize("B,n", [(37, 37 * 8 * 3 + 5), (300, 300 * 8 * 2), (1, 100), (64, 64 * 8 * 7 + 63)])
def test_data_parallel_ranks_draw_disjoint_rows_in_an_epoch(W, B, n):
    """At world W each step's W * B rows (rank r: positions ((step * W + r) * B + j), chunk B * W) are pairwise distinct
    inside an epoch, and one epoch's steps over all ranks visit each of its n_eff rows once: data-parallel training sees
    every row once per epoch."""
    chunk = B * W
    n_eff = n - n % chunk
    if n_eff == 0:
        pytest.skip("the table is smaller than one data-parallel step")
    steps = n_eff // chunk
    for epoch in range(2):
        seen = []
        for s in range(epoch * steps, (epoch + 1) * steps):
            step_rows = np.concatenate([S.sampled_indices(s, B, r, W, False, n, 5) for r in range(W)])
            assert np.unique(step_rows).size == W * B, (epoch, s)
            seen.append(step_rows)
        assert np.unique(np.concatenate(seen)).size == n_eff, epoch


def test_sharded_positions():
    """A sharded table: every rank walks its own permutation with positions step * B + j, chunk B."""
    B, n = 37, 500
    for done in (0, 3, 2 ** 33 + 3):
        want = S.stream_index(done * B + np.arange(B), n, B, 9)
        for r, W in ((0, 1), (1, 2), (7, 8)):
            assert np.array_equal(S.sampled_indices(done, B, r, W, True, n, 9), want)


def test_positions_past_2_to_the_32_steps():
    """Step counters past 2^32 keep their int64 positions: the epoch and the row within it follow p exactly."""
    B, W, n = 4737, 8, 2 ** 24 + 5
    done = 2 ** 33 + 3
    p = (done * W + 7) * B + np.arange(B, dtype=np.int64)
    n_eff = n - n % (B * W)
    idx = S.sampled_indices(done, B, 7, W, False, n, 9)
    want = S.feistel_perm(p % n_eff, n, S.epoch_key(9, p // n_eff)).astype(np.int64)
    assert np.array_equal(idx, want)
    assert p.min() > 2 ** 48 and (p // n_eff).min() > 2 ** 24


# ---------------------------------------------------------------- update noise
def _corr_bound(m):
    return 5.0 / np.sqrt(m)           # five standard deviations of a sample correlation of m independent pairs


GAUSS_KEYS = ("temp_eps", "alpha_eps_t", "alpha_eps_t1", "critic_eps_t", "critic_eps_t1", "actor_eps")


@pytest.mark.parametrize("seed", SEEDS)
def test_noise_blocks_have_their_distributions(seed):
    B, n = 2000, 10
    nz = S.update_noise(seed, 3, 1, B, n)
    assert set(nz) == set(S.NOISE_KEYS)
    for k in S.NOISE_KEYS:
        assert nz[k].shape == ((B, 1) if k in ("temp_eps", "actor_eps") else (B, n)), k
    for k in GAUSS_KEYS:
        x = nz[k].ravel()
        assert nz[k].dtype == np.float64
        assert stats.kstest(x, "norm").pvalue > 1e-4, k
    for k in ("alpha_u", "critic_u"):
        x = nz[k].ravel()
        assert nz[k].dtype == np.float32
        assert x.min() > -1.0 and x.max() <= 1.0, k
        assert stats.kstest(x.astype(np.float64), "uniform", args=(-1.0, 2.0)).pvalue > 1e-4, k


def test_noise_blocks_steps_and_ranks_are_uncorrelated():
    """Within one update every pair of equally sized blocks, and each block against the same block of the next step and
    of the next rank, correlate no more than independent samples of that size would."""
    B, n = 1000, 10
    a = S.update_noise(9, 5, 0, B, n)
    step = S.update_noise(9, 6, 0, B, n)
    rank = S.update_noise(9, 5, 1, B, n)
    big = [k for k in S.NOISE_KEYS if a[k].shape[1] == n]
    bound = _corr_bound(B * n)
    corr = lambda x, y: abs(np.corrcoef(np.ravel(x).astype(np.float64), np.ravel(y).astype(np.float64))[0, 1])
    for i, k in enumerate(big):
        for k2 in big[i + 1:]:
            assert corr(a[k], a[k2]) < bound, (k, k2)
    assert corr(a["temp_eps"], a["actor_eps"]) < _corr_bound(B)
    for k in S.NOISE_KEYS:
        m = a[k].size
        assert corr(a[k], step[k]) < _corr_bound(m), ("step", k)
        assert corr(a[k], rank[k]) < _corr_bound(m), ("rank", k)
        assert not np.array_equal(a[k], step[k]) and not np.array_equal(a[k], rank[k]), k


def test_noise_stream_packing():
    """The stream is (done << 8) | (rank & 0xff): rank 256 would repeat rank 0 (why cql_create takes at most 256 ranks),
    and the step counter's high word reaches the counter's fourth word."""
    assert S.noise_stream(5, 256) == S.noise_stream(5, 0)
    assert S.noise_stream(2 ** 33 + 3, 7) == ((2 ** 33 + 3) << 8) | 7
    a = S.update_noise_packed(9, 2 ** 33 + 3, 7, 3, 2)
    b = S.update_noise_packed(9, 3, 7, 3, 2)
    assert not np.array_equal(a, b)


def test_mdp_action_noise_is_seeded_per_row():
    rows = np.arange(200_000)
    z = S.mdp_action_noise(3, rows, 1.0)
    assert stats.kstest(z, "norm").pvalue > 1e-4
    assert np.array_equal(S.mdp_action_noise(3, rows[::-1], 1.0), z[::-1])
    assert abs(np.corrcoef(z, S.mdp_action_noise(4, rows, 1.0))[0, 1]) < _corr_bound(rows.size)
    assert np.array_equal(S.mdp_action_noise(3, rows[:10], 1e-3), S.box_muller(*S.philox4x32_10(
        3 ^ S.MDP_SEED_XOR, S.MDP_STREAM, rows[:10])[:2]) * float(np.float32(1e-3)))
