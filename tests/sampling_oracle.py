"""Host reference of the update's input definitions: the minibatch positions of the epoch permutation, the Philox noise
of an update and the MDP builder's seeded action noise.  TEST INFRASTRUCTURE ONLY.

Written from the definitions (DESIGN.md section 1, "Sampling and noise"), vectorised in numpy; it shares no code with
``csrc/common.cuh`` / ``csrc/update.cuh`` / ``csrc/mdp_gpu.cu``.

One float32 detail is part of the definition: ``u01(x) = ((x >> 8) + 0.5) * 2^-24`` is formed in float32, so for
``x >> 8 >= 2^23`` the ``+ 0.5`` rounds to even, and ``x >> 8 = 2^24 - 1`` gives exactly 1.0.  ``u01`` below returns
that float32 value; the uniform draws ``2 u1 - 1`` are exact in float32 from it, and the Gaussian draws are evaluated
in float64 from the float32 ``u1``, ``u2``.
"""
from __future__ import annotations

import numpy as np

M32 = np.uint64(0xFFFFFFFF)
NOISE_KEYS = ("temp_eps", "alpha_eps_t", "alpha_eps_t1", "alpha_u",
              "critic_eps_t", "critic_eps_t1", "critic_u", "actor_eps")
NOISE_SEED_XOR = 0x5851F42D4C957F2D
MDP_SEED_XOR, MDP_STREAM = 0xA0761D6478BD642F, 0x4D4450
PERM_SEED_MUL, PERM_EPOCH_MUL = 0x9E3779B97F4A7C15, 0xD1B54A32D192ED03
MASK64 = (1 << 64) - 1


def _u64(x) -> np.ndarray:
    """Python int / int array -> uint64 array (mod 2^64)."""
    if isinstance(x, (int, np.integer)):
        return np.asarray(int(x) & MASK64, dtype=np.uint64)
    return np.asarray(x).astype(np.uint64)


def philox4x32_raw(ctr, key):
    """Philox4x32-10 on a counter (four uint32 words, arrays broadcast) and a key (two words) -> four uint32 arrays."""
    c = [np.asarray(w).astype(np.uint64) & M32 for w in ctr]
    k0, k1 = (np.asarray(w).astype(np.uint64) & M32 for w in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return [w.astype(np.uint32) for w in c]


def philox4x32_10(seed, stream, index):
    """Key (seed lo, seed hi), counter (index lo, index hi, stream lo, stream hi); each argument mod 2^64."""
    s, st, ix = _u64(seed), _u64(stream), _u64(index)
    sh = np.uint64(32)
    return philox4x32_raw((ix & M32, ix >> sh, st & M32, st >> sh), (s & M32, s >> sh))


def u01(x) -> np.ndarray:
    """32 random bits -> float32 in (0, 1]: ((x >> 8) + 0.5) * 2^-24, the sum rounded to float32."""
    hi = (np.asarray(x, dtype=np.uint32) >> np.uint32(8)).astype(np.float32)
    return (hi + np.float32(0.5)) * np.float32(2.0 ** -24)


def box_muller(r0, r1) -> np.ndarray:
    """sqrt(-2 ln u1) * cos(2 pi u2) in float64 from the float32 u1 = u01(r0), u2 = u01(r1)."""
    u1, u2 = u01(r0).astype(np.float64), u01(r1).astype(np.float64)
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def noise_stream(done: int, rank: int) -> int:
    """Philox stream of the update that starts after ``done`` completed updates on ``rank``."""
    return ((int(done) << 8) | (int(rank) & 0xFF)) & MASK64


def uniform_mask(B: int, n: int) -> np.ndarray:
    """Which of the 2B + 6Bn packed draws are uniform: element i with a = i - B in [0, 6Bn) and (a div Bn) mod 3 == 2
    (alpha_u, critic_u)."""
    Bn = B * n
    a = np.arange(2 * B + 6 * Bn, dtype=np.int64) - B
    return (a >= 0) & (a < 6 * Bn) & ((np.maximum(a, 0) // Bn) % 3 == 2)


def update_noise_packed(seed: int, done: int, rank: int, B: int, n: int) -> np.ndarray:
    """The 2B + 6Bn draws of one update in ``cql_update_batch``'s noise packing, float64 (uniform entries exact)."""
    i = np.arange(2 * B + 6 * B * n, dtype=np.int64)
    r = philox4x32_10(int(seed) ^ NOISE_SEED_XOR, noise_stream(done, rank), i)
    uniform = uniform_mask(B, n)
    out = box_muller(r[0], r[1])
    out[uniform] = 2.0 * u01(r[0][uniform]).astype(np.float64) - 1.0
    return out


def unpack_noise(flat, B: int, n: int) -> dict:
    """Packed noise -> {NOISE_KEYS: [B, 1] or [B, n]} (dtype kept)."""
    flat = np.asarray(flat)
    sizes = [B] + [B * n] * 6 + [B]
    assert flat.size == sum(sizes), (flat.size, sizes)
    out, o = {}, 0
    for key, s in zip(NOISE_KEYS, sizes):
        out[key] = flat[o:o + s].reshape(B, s // B)
        o += s
    return out


def update_noise(seed: int, done: int, rank: int, B: int, n: int) -> dict:
    """The seven draws of one update by key: uniform blocks (alpha_u, critic_u) float32 (exact), the rest float64."""
    out = unpack_noise(update_noise_packed(seed, done, rank, B, n), B, n)
    for key in ("alpha_u", "critic_u"):
        out[key] = out[key].astype(np.float32)
    return out


# ---------------------------------------------------------------- epoch permutation
def _mix32(x):
    x = x ^ (x >> np.uint64(16))
    x = (x * np.uint64(0x7FEB352D)) & M32
    x = x ^ (x >> np.uint64(15))
    x = (x * np.uint64(0x846CA68B)) & M32
    return x ^ (x >> np.uint64(16))


def _feistel_round4(x, hb: int, key):
    """The 4-round Feistel network on 2*hb-bit values (one pass, no cycle walk)."""
    h = np.uint64(hb)
    mask = np.uint64((1 << hb) - 1)
    l, r = x >> h, x & mask
    for i in range(4):
        kw = (key >> np.uint64(13 * i)) & M32
        f = _mix32(((r & M32) * np.uint64(0x9E3779B1) + kw + np.uint64((0x85EBCA6B * (i + 1)) & 0xFFFFFFFF)
                    + ((r >> np.uint64(16)) & M32) * np.uint64(0xC2B2AE35)) & M32)
        l, r = r, (l ^ f) & mask
    return (l << h) | r


def feistel_perm(x, n: int, key) -> np.ndarray:
    """Bijection of [0, n): the Feistel network on the smallest even bit count 2*hb >= log2(n) (2 <= 2*hb <= 62),
    re-applied to values that land outside [0, n) until they fall inside (cycle walking).  ``key`` mod 2^64, scalar or
    broadcast with ``x``."""
    bits = 2
    while bits < 62 and (1 << bits) < n:
        bits += 2
    x = _u64(x).copy().reshape(-1)
    key = np.broadcast_to(_u64(key), x.shape).copy()
    nn = np.uint64(n)
    todo = np.arange(x.size)
    while todo.size:                     # do { ... } while (x >= n): every value takes at least one pass
        x[todo] = _feistel_round4(x[todo], bits // 2, key[todo])
        todo = todo[x[todo] >= nn]
    return x


def epoch_key(seed: int, epoch) -> np.ndarray:
    """seed * 0x9E3779B97F4A7C15 + epoch * 0xD1B54A32D192ED03 + 1 (mod 2^64)."""
    base = np.uint64((int(seed) * PERM_SEED_MUL + 1) & MASK64)
    return np.atleast_1d(_u64(epoch)) * np.uint64(PERM_EPOCH_MUL) + base


def stream_index(p, n: int, chunk: int, seed: int) -> np.ndarray:
    """Position(s) p >= 0 of the sampling stream -> transition index.  An epoch covers n_eff = n - n mod chunk positions
    (n when that is 0) and permutes all n rows with its own key."""
    n_eff = n - n % chunk
    if n_eff <= 0:
        n_eff = n
    p = np.asarray(p, dtype=np.int64).reshape(-1)
    epoch, q = p // n_eff, p % n_eff
    return feistel_perm(q, n, epoch_key(seed, epoch)).astype(np.int64)


def sampled_indices(done: int, B: int, rank: int, world: int, sharded: bool, n: int, seed: int) -> np.ndarray:
    """Table rows of the sampled update after ``done`` completed updates: replicated table, positions
    (done * W + rank) * B + j with chunk B * W; a sharded table (this rank holds its own rows), done * B + j, chunk B."""
    j = np.arange(B, dtype=np.int64)
    if sharded:
        return stream_index(int(done) * B + j, n, B, seed)
    return stream_index((int(done) * world + rank) * B + j, n, B * world, seed)


# ---------------------------------------------------------------- MDP builder
def mdp_action_noise(seed: int, rows, scale: float) -> np.ndarray:
    """The builder's seeded action noise of original rows ``rows``, float64 (``scale`` as the float32 it is passed as)."""
    r = philox4x32_10(int(seed) ^ MDP_SEED_XOR, MDP_STREAM, np.asarray(rows, dtype=np.int64))
    return box_muller(r[0], r[1]) * float(np.float32(scale))


def mdp_actions(seed: int, relevance, scale: float) -> np.ndarray:
    """float32 action of every original row: (float)((double)(float)relevance + noise)."""
    rel = np.asarray(relevance, dtype=np.float64).astype(np.float32).astype(np.float64)
    return (rel + mdp_action_noise(seed, np.arange(rel.size), scale)).astype(np.float32)
