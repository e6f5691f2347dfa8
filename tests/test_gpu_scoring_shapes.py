"""GPU parity of user x item scoring (``cql_score_topk``, ``cql_score_pairs``) at the critic counts, k, candidate counts
and user counts the API accepts.

``cql_create`` takes n_critics 1..4 and ``cql_score_topk`` k 1..CQL_MAX_TOPK = 1024.  The precision picks the top-k
scorer (``score_topk_dev_impl`` in ``csrc/capi.cu``); k picks the tensor-core scorers' fold, the candidate count their
merge:

    precision      top-k scorer                                       fold                                  merge
    fp32           k_score_topk (64-item tiles, grid (chunks, users)  warp_fold_tile                        k_topk_merge when
                   in slabs of 65 535 users)                                                                chunks > 1
    tf32x3, bf16   tc_score_kernel (W2 packed by k_pack_w2,           fold_block_select for k <= 32,        k_topk_merge when
                   gridDim.y = C)                                     warp 0's sequential fold for k > 32   I > 2048
    f16x3          tc_score_h_kernel (k_pack_multi_h, C + 1 jobs)     same                                  same
    all            k_score_pairs                                      --                                    --

A tensor-core block is SC_CH * 128 = 2048 items of one user; the U * chunks blocks are split over min(U * chunks, SMs)
persistent CTAs (``blk_lo`` / ``blk_hi``), and a CTA that moves to another user re-stages its seen list.  The FP32 scorer
cuts the list into chunks = clamp(ceil(8 SMs / U), 1, ceil(I / 64)) (rounded to whole tiles per chunk).  The matrix
(``CASES``, every precision x C = 1..4 in mode "q", C = 1 and 4 in mode "policy"); the fp32 columns are for 148 SMs:

    U, I, k            fp32 tiles / chunks   tensor-core blocks per user, CTAs       TC fold, boundary
    1, 1, 1            1 / 1                 1 block of 1 row, 1 CTA                  select; one candidate
    2, 63, 100         1 / 1                 1 block of 63 rows                       warp 0; k > I: padded rows
    3, 129, 33         3 / 3 + merge         1 block, last tile of 1 row              warp 0 at k = 33
    SMs-1, 65, 7       2 / 2 + merge         1, SMs - 1 CTAs of one user              select
    SMs+1, 128, 32     2 / 2 + merge         1, one CTA takes two users               select at k = 32
    5, 2049, 1024      33 / 33 + merge       2 (the 2nd holds 1 row < k) + merge      warp 0 at k = CQL_MAX_TOPK
    4, 4097, 10        65 / 65 + merge       3 (the 3rd holds 1 row) + merge          select
    2SMs+3, 2048, 10   32 / 4 + merge        1, 2SMs + 3 blocks on SMs CTAs           select; CTAs change user
    37, 26744, 10      418 / 30 + merge      14 + merge, 518 blocks on SMs CTAs       select; users split over CTAs
    4, 4097, 10 scaled same as 4, 4097, 10 with the observation and action scalers on (item_x, act_rev)

The last two unscaled cases compare a named user sample with the oracle (first, last and the users of the CTA
partition boundaries, ``_sample_rows``); the bit-exact invariances below cover the others.

Reference: ``cql_oracle.relevance`` in float32 on the raw-index observations, cached per (state, users, items, mode,
scalers) so that every precision meets the same matrix; the reference list is ``recs_oracle.brute_force_topk``'s rule
(seen items dropped, order (-score as float64, item id)), vectorised, and checked against ``brute_force_topk`` itself on
two rows per case.  Candidate ids are non-contiguous and in random order, so a score paired with the wrong position
changes the item.  Each returned row must pass ``_check_rows``: items are unseen candidates, unique; each score is within
TOL = 1e-5 max|Q| of the oracle score of that item; the row is ordered by (score desc, id asc) on its own scores; it has
exactly min(k, unseen candidates) real entries, then -1 / -inf; no omitted unseen candidate scores above the k-th score
plus the gate; positions differ from the reference only between scores within the gate.  A row whose float32 oracle
itself misses the float64 one by more than a quarter of the gate is compared with the float64 twin instead, within
max(gate, 4x that miss) (``Hp.check_f64_budget``'s rule); such rows are printed.

Further tests: exact ties (every score equal, the list is the k smallest unseen ids); the seen filter inside the fused
scorers (seen top-N, lists around SEEN_CACHE = 4096, seen ids that are not candidates, a block fully seen, everything
seen); bit-exact invariances (users alone / among many / reversed / twice, permuted candidates, the device entry on a
non-default stream, bf16 == tf32x3, the FP32 slab edge, two halves merged); ``score_pairs`` against the oracle and
against ``score_topk``; ``CQL.predict`` against ``predict_pairs`` at C = 1 and 4; negative candidate ids.
"""
import numpy as np
import pytest
import torch

from oracle import cql_oracle as O
from oracle import recs_oracle
from replay_cql_b200 import layout
from tests import helpers as Hp
from tests import scaler_oracle as S

pytestmark = pytest.mark.gpu
TOL = 1e-5
PRECISIONS = ("fp32", "tf32x3", "bf16", "f16x3")
PREP = {"scaler": {"type": "standard", "mean": [3000.5, 1850.25], "std": [1740.0, 1070.0]},
        "action_scaler": {"type": "min_max", "minimum": [0.99], "maximum": [5.01]}}
TC_BLOCK = 16 * 128                     # SC_CH * TM items per tensor-core block
CHUNK_ROWS = 1 << 17                    # oracle rows per forward (bounds the CPU memory of the hidden layers)

# (U, I, k, scaled); U may be a formula in the SM count
CASES = [(1, 1, 1, False), (2, 63, 100, False), (3, 129, 33, False), ("SMs-1", 65, 7, False), ("SMs+1", 128, 32, False),
         (5, 2049, 1024, False), (4, 4097, 10, False), ("2SMs+3", 2048, 10, False), (37, 26744, 10, False),
         (4, 4097, 10, True)]
SAMPLED = {"2SMs+3", 37}
_U = {"SMs-1": lambda s: s - 1, "SMs+1": lambda s: s + 1, "2SMs+3": lambda s: 2 * s + 3}
_case_id = lambda c: f"U{c[0]}-I{c[1]}-k{c[2]}" + ("-scaled" if c[3] else "")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _n_users(u):
    return _U[u](_sms()) if isinstance(u, str) else u


# ---------------------------------------------------------------- oracle, cached
_STATE = {}


def _state(C, seed=11, ties=False):
    """-> (flat, float32 oracle state, float64 oracle state); ties: every critic's W3 and the actor's mean row zeroed"""
    key = (C, seed, ties)
    if key not in _STATE:
        flat = layout.init_state(C, seed)
        if ties:
            un = layout.unpack_state(flat, C)
            for c in un["critics"]:
                c["W3"][:] = 0.0
            un["actor"]["W3"][0] = 0.0
            flat = layout.pack_state(un["actor"], un["critics"], un["targ_actor"], un["targ_critics"], un["log_temp"],
                                     un["log_alpha"])
        cfg = O.OracleConfig(n_critics=C)
        _STATE[key] = (flat, Hp.flat_to_oracle_state(flat, cfg), Hp.flat_to_oracle_state(flat, cfg, dtype=torch.float64))
    return _STATE[key]


def _relevance(st, obs, mode, scaled, dtype):
    """raw float32 observations [n, 2] -> relevance.  The scalers run in float32 (as on the GPU); the float64 twin starts
    from the same float32 scaled observations."""
    x = S.obs_fwd(PREP["scaler"] if scaled else None, torch.from_numpy(np.ascontiguousarray(obs, dtype=np.float32)))
    out = []
    for i in range(0, x.shape[0], CHUNK_ROWS):
        r = O.relevance(st, x[i:i + CHUNK_ROWS].to(dtype), mode).reshape(-1)
        if mode == "policy" and scaled:
            r = S.act_rev(PREP["action_scaler"], r)
        out.append(r)
    return torch.cat(out).numpy() if out else np.zeros(0, np.float64 if dtype == torch.float64 else np.float32)


def _grid_obs(users, items):
    return np.stack([np.repeat(users, items.size), np.tile(items, users.size)], 1).astype(np.float32)


_Q = {}


def _oracle(C, users, items, mode, scaled=False, dtype=torch.float32, seed=11, ties=False):
    """relevance matrix [len(users), len(items)] of the state _state(C, seed, ties), cached.  One forward per user, as
    brute_force_topk runs it (the CPU matmul's bits depend on the row count)."""
    key = (C, seed, ties, mode, scaled, dtype, users.tobytes(), items.tobytes())
    if key not in _Q:
        _, st32, st64 = _state(C, seed, ties)
        st = st64 if dtype == torch.float64 else st32
        _Q[key] = np.stack([_relevance(st, _grid_obs(users[r:r + 1], items), mode, scaled, dtype)
                            for r in range(users.size)]) if users.size else np.zeros((0, items.size), np.float32)
    return _Q[key]


def _ref_topk(Q, items, seen_mask, k):
    """brute_force_topk's rule on whole rows: -> column indices [R, min(k, I)] ordered by (-score as float64, item id),
    seen columns last, and the number of unseen candidates per row"""
    key = np.where(seen_mask, np.inf, -np.asarray(Q, dtype=np.float64))
    order = np.lexsort((np.broadcast_to(items, Q.shape), key), axis=-1)[:, :k]
    return order, (~seen_mask).sum(1)


def _as_lists(Q, items, seen_mask, k):
    order, n_unseen = _ref_topk(Q, items, seen_mask, k)
    R = Q.shape[0]
    ri = np.full((R, k), -1, np.int32)
    rs = np.full((R, k), -np.inf, np.float32)
    for r in range(R):
        n = min(k, int(n_unseen[r]))
        ri[r, :n] = items[order[r, :n]]
        rs[r, :n] = Q[r, order[r, :n]]
    return ri, rs


# ---------------------------------------------------------------- inputs
def _candidates(rng, I, pool=None):
    """I distinct, non-contiguous ids in random order"""
    return rng.choice(pool or max(4000, 2 * I), size=I, replace=False).astype(np.int32)


def _csr(users, seen):
    """seen: {user id: iterable of item ids} -> (indptr over user id 0..max, sorted unique items)"""
    n = int(users.max()) + 1
    indptr = np.zeros(n + 1, dtype=np.int64)
    flat = []
    for u in range(n):
        s = sorted(set(int(x) for x in seen.get(u, ())))
        flat.extend(s)
        indptr[u + 1] = len(flat)
    return indptr, np.asarray(flat, dtype=np.int32)


def _seen_mask(users, items, seen):
    return np.stack([np.isin(items, np.fromiter(seen.get(int(u), ()), dtype=np.int64)) for u in users]) \
        if users.size else np.zeros((0, items.size), bool)


# ---------------------------------------------------------------- the validity check
def _check_rows(tag, ti, ts, k, items, seen_mask, Q, q64, budgeted, scale=None):
    """ti / ts [R, k] returned by the scorer, Q [R, I] float32 oracle rows of the same users, seen_mask [R, I];
    q64(r) -> the float64 twin of row r (computed only where the budget rule needs it).  -> the gate scale used."""
    R, I = Q.shape
    ref_order, n_unseen = _ref_topk(Q, items, seen_mask, k)
    if scale is None:
        best = [Q[r, ref_order[r, :min(k, int(n_unseen[r]))]] for r in range(R)]
        best = np.concatenate(best) if best else np.zeros(0)
        scale = max(1.0, float(np.max(np.abs(best)))) if best.size else 1.0
    sorter = np.argsort(items, kind="stable")
    for r in range(R):
        where = (tag, r)
        n = min(k, int(n_unseen[r]))
        it, sc = ti[r], ts[r]
        assert np.all(it[n:] == -1) and np.all(np.isneginf(sc[n:])), (where, "padding", it, sc)
        it, sc = it[:n].astype(np.int64), sc[:n].astype(np.float64)
        assert np.all(it >= 0) and np.all(np.isfinite(sc)), (where, "real entries", it, sc)
        p = sorter[np.clip(np.searchsorted(items, it, sorter=sorter), 0, I - 1)]
        assert np.array_equal(items[p], it), (where, "not a candidate", it[items[p] != it])
        assert np.unique(it).size == n, (where, "duplicate item")
        assert not seen_mask[r, p].any(), (where, "seen item returned", it[seen_mask[r, p]])
        if n > 1:
            assert np.all((sc[:-1] > sc[1:]) | ((sc[:-1] == sc[1:]) & (it[:-1] < it[1:]))), (where, "order", it, sc)
        ref, gate = np.asarray(Q[r], np.float64), TOL * scale
        err = float(np.max(np.abs(sc - ref[p]), initial=0.0))
        if err > gate:
            ref64 = np.asarray(q64(r), np.float64)
            d = float(np.max(np.abs(ref[p] - ref64[p])))
            assert d > gate / 4, (where, "float32 oracle is accurate here, the GPU must be too", err / scale, d / scale)
            ref, gate = ref64, max(gate, 4 * d)
            budgeted.append((where, err / scale, float(np.max(np.abs(sc - ref[p]))) / scale, d / scale))
        assert np.max(np.abs(sc - ref[p]), initial=0.0) <= gate, (where, "score", np.max(np.abs(sc - ref[p])) / scale)
        unseen = ~seen_mask[r]
        if n == k:
            omitted = unseen.copy()
            omitted[p] = False
            if omitted.any():
                assert ref[omitted].max() <= sc[-1] + gate, (where, "omitted candidate", ref[omitted].max(), sc[-1])
        cols = np.nonzero(unseen)[0]                                  # the reference list on the row's reference
        want = cols[np.lexsort((items[cols], -ref[cols]))[:n]]
        diff = p != want
        assert np.all(np.abs(ref[p[diff]] - ref[want[diff]]) <= gate), (where, "position", it[diff], items[want[diff]])
    return scale


def _two_rows_equal_brute_force(C, users, items, seen, k, mode, scaled, rows):
    """the vectorised reference equals recs_oracle.brute_force_topk (its own forward passes) on the given rows"""
    _, st, _ = _state(C)
    score = lambda obs: _relevance(st, obs, mode, scaled, torch.float32)
    u = users[rows]
    bi, bs = recs_oracle.brute_force_topk(score, u, items, {int(x): set(seen.get(int(x), ())) for x in u}, k)
    ri, rs = _as_lists(_oracle(C, u, items, mode, scaled), items, _seen_mask(u, items, seen), k)
    assert np.array_equal(bi, ri) and np.array_equal(bs, rs)


def _report(tag, budgeted):
    print(f"\n[{tag}] comparisons that needed the float64 budget: {len(budgeted)}")
    for b in budgeted:
        print("   ", b)


# ---------------------------------------------------------------- engines, one per (precision, C)
_ENG = {}


def _engine(engine_factory, precision, C, flat):
    key = (precision, C)
    if key not in _ENG:
        _ENG[key] = engine_factory(batch_size=64, n_critics=C, precision=precision)
    eng = _ENG[key]
    eng.set_state(flat)
    eng.set_preprocessing()
    return eng


def _tc_boundary_rows(U, I):
    """user rows of a tensor-core launch that meet a CTA partition boundary (first / last block of a CTA)"""
    tiles = -(-I // 128)
    chunks = -(-tiles // 16)
    n_blocks = U * chunks
    grid = min(n_blocks, _sms())
    rows = set()
    for b in range(1, grid):
        lo = n_blocks * b // grid
        rows.update((lo // chunks, (lo - 1) // chunks))
    return sorted(rows)


def _sample_rows(U, I):
    """first, last and (up to 8, evenly spread) users on CTA partition boundaries"""
    b = _tc_boundary_rows(U, I)
    pick = [b[i] for i in np.linspace(0, len(b) - 1, min(8, len(b))).astype(int)] if b else []
    return np.array(sorted({0, U - 1, *pick}))


# ---------------------------------------------------------------- 3. the shape matrix
MATRIX = [pytest.param(p, C, "q", c, id=f"{p}-C{C}-q-{_case_id(c)}") for C in (1, 2, 3, 4) for c in CASES
          for p in PRECISIONS]
MATRIX += [pytest.param(p, C, "policy", c, id=f"{p}-C{C}-policy-{_case_id(c)}") for C in (1, 4) for c in CASES
           for p in PRECISIONS]


@pytest.mark.parametrize("precision,C,mode,case", MATRIX)
def test_topk_matches_oracle_at_shape(engine_factory, precision, C, mode, case):
    """score_topk against the float32 oracle under _check_rows, and every returned (user, item, score) against
    score_pairs within the same gate."""
    u_spec, I, k, scaled = case
    U = _n_users(u_spec)
    rng = np.random.default_rng(1000 * I + U)
    users = rng.choice(6040, size=U, replace=False).astype(np.int32)
    items = _candidates(rng, I)
    seen = {}
    for r, u in enumerate(users):
        m = int(rng.integers(0, min(60, I // 3) + 1))
        s = set(rng.choice(items, size=m, replace=False).tolist())
        s.update(rng.integers(0, 3 * I + 10, 5).tolist())          # ids that may not be candidates
        seen[int(u)] = s
    if U > 1:
        seen[int(users[-1])] = set(items.tolist())                 # a user who has seen everything
    indptr, flat_seen = _csr(users, seen)
    flat, _, _ = _state(C)
    eng = _engine(engine_factory, precision, C, flat)
    if scaled:
        eng.set_preprocessing(scaler=PREP["scaler"], action_scaler=PREP["action_scaler"])
    ti, ts = eng.score_topk(users, items, k, indptr, flat_seen, mode=mode)
    rows = _sample_rows(U, I) if u_spec in SAMPLED else np.arange(U)
    Q = _oracle(C, users[rows], items, mode, scaled)
    q64 = lambda r: _oracle(C, users[rows[r:r + 1]], items, mode, scaled, torch.float64)[0]
    budgeted = []
    scale = _check_rows((precision, C, mode, case), ti[rows], ts[rows], k, items, _seen_mask(users[rows], items, seen),
                        Q, q64, budgeted)
    _two_rows_equal_brute_force(C, users, items, seen, k, mode, scaled, rows[:2] if U > 1 else rows)
    real = ti >= 0
    if real.any():
        pu = np.broadcast_to(users[:, None], ti.shape)[real]
        ps = eng.score_pairs(pu, ti[real], mode=mode)
        assert np.max(np.abs(ps.astype(np.float64) - ts[real])) <= TOL * scale, "score_topk vs score_pairs"
    _report(f"{precision} C={C} {mode} {_case_id(case)}", budgeted)


# ---------------------------------------------------------------- 4. exact ties
@pytest.mark.parametrize("mode", ["q", "policy"])
@pytest.mark.parametrize("k", [10, 32, 33, 1024])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_exact_ties_return_smallest_unseen_ids(engine_factory, precision, k, mode):
    """Every critic's W3 and the actor's mean row zeroed: every score is the same bias value, so the list is the k
    smallest unseen candidate ids and the real scores of a row are bit-equal.  I = 4097 (three tensor-core blocks, the
    last of one row): fold_block_select's candidate overflow (FB_CAP) and k_topk_merge's tie rule."""
    C, I = 3, 4097
    rng = np.random.default_rng(44)
    items = _candidates(rng, I)
    users = rng.choice(6040, size=6, replace=False).astype(np.int32)
    small = np.sort(items)
    seen = {int(users[0]): set(),
            int(users[1]): set(small[:5].tolist()),                               # the best 5 (by id) seen
            int(users[2]): set(small[::3].tolist()),
            int(users[3]): set(small[:1100].tolist()) | set(rng.choice(items, 200).tolist()),
            int(users[4]): set(small[5:].tolist()),                               # 5 unseen candidates left
            int(users[5]): set(rng.choice(items, 50).tolist()) | {int(small[-1]) + 1}}
    indptr, flat_seen = _csr(users, seen)
    flat, _, _ = _state(C, ties=True)
    eng = _engine(engine_factory, precision, C, flat)
    ti, ts = eng.score_topk(users, items, k, indptr, flat_seen, mode=mode)
    want = _oracle(C, users[:1], items[:1], mode, ties=True)[0, 0]
    for r, u in enumerate(users):
        unseen = np.sort(np.setdiff1d(items, np.fromiter(seen[int(u)], np.int64)))
        n = min(k, unseen.size)
        assert np.array_equal(ti[r, :n], unseen[:n]), (r, ti[r, :n], unseen[:n])
        assert np.all(ti[r, n:] == -1) and np.all(np.isneginf(ts[r, n:]))
        assert np.all(ts[r, :n] == ts[r, 0]), (r, np.unique(ts[r, :n]))
        assert abs(float(ts[r, 0]) - float(want)) <= TOL * max(1.0, abs(float(want)))


# ---------------------------------------------------------------- 5. the seen filter inside the fused scorers
def _seen_filter_users(k):
    """12 users over I = 26 744 non-contiguous candidates; seen lists from the oracle's order of each user"""
    C, I = 2, 26744
    rng = np.random.default_rng(55)
    items = _candidates(rng, I)
    users = rng.choice(6040, size=12, replace=False).astype(np.int32)
    Q = _oracle(C, users, items, "q")
    order = np.lexsort((np.broadcast_to(items, Q.shape), -Q.astype(np.float64)), axis=-1)
    others = np.setdiff1d(np.arange(2 * I), items)                 # ids that are not candidates
    seen = {}
    for r, n in enumerate((k - 1, k, 5 * k, 2100, I - 3)):         # the user's oracle top N
        seen[int(users[r])] = items[order[r, :n]]
    for r, n in zip(range(5, 9), (4095, 4096, 4097, 12000)):         # around SEEN_CACHE: a quarter of the best items
        top = items[order[r, :n // 4]]
        rest = rng.choice(items[order[r, n // 4:]], size=n - n // 4, replace=False)
        seen[int(users[r])] = np.concatenate([top, rest])
    seen[int(users[9])] = np.concatenate([items[order[9, :3 * k]], rng.choice(others, 3000, replace=False)])
    seen[int(users[10])] = items[:TC_BLOCK]                         # every candidate of block 0, none of the others
    seen[int(users[11])] = items                                     # everything
    for u, s in seen.items():
        assert np.unique(s).size == len(s), u
    return C, users, items, {u: set(s.tolist()) for u, s in seen.items()}


@pytest.mark.parametrize("k", [10, 32, 33])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_seen_filter_in_fused_scorers(engine_factory, precision, k):
    """A user who has seen their top k - 1, k, 5k, 2100 (across a block boundary) or all but 3 items; seen lists of
    4095, 4096, 4097 and 12 000 ids (the shared-memory cache and the global binary search); seen ids that are not
    candidates; block 0 fully seen; everything seen (an all-padding row).  Every user against the oracle."""
    C, users, items, seen = _seen_filter_users(k)
    indptr, flat_seen = _csr(users, seen)
    assert np.diff(indptr)[users].tolist()[5:9] == [4095, 4096, 4097, 12000]
    flat, _, _ = _state(C)
    eng = _engine(engine_factory, precision, C, flat)
    ti, ts = eng.score_topk(users, items, k, indptr, flat_seen)
    budgeted = []
    _check_rows((precision, k), ti, ts, k, items, _seen_mask(users, items, seen), _oracle(C, users, items, "q"),
                lambda r: _oracle(C, users[r:r + 1], items, "q", dtype=torch.float64)[0], budgeted)
    assert np.all(ti[11] == -1) and np.sum(ti[4] >= 0) == 3
    _report(f"{precision} seen filter k={k}", budgeted)


# ---------------------------------------------------------------- 6. bit-exact invariances
def _same(a, b, what):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), what


def _invariance_inputs(I=4097):
    rng = np.random.default_rng(66)
    n_other = 3 * _sms() + 1
    users = rng.choice(6040, size=n_other + 1, replace=False).astype(np.int32)
    items = _candidates(rng, I)
    seen = {int(u): set(rng.choice(items, size=int(rng.integers(0, 80)), replace=False).tolist()) for u in users}
    others = np.setdiff1d(np.arange(max(4000, 2 * I)), items)            # a list past SEEN_CACHE, partly non-candidates
    seen[int(users[7])] = set(rng.choice(items, size=3000, replace=False).tolist()) | \
        set(rng.choice(others, size=1500, replace=False).tolist())
    return rng, users, items, seen


def _merge(a, b, k):
    """two top-k results of the same users over disjoint candidate lists -> one, by (score desc, id asc)"""
    i = np.concatenate([a[0], b[0]], 1)
    s = np.concatenate([a[1], b[1]], 1)
    oi = np.full(a[0].shape, -1, np.int32)
    os_ = np.full(a[1].shape, -np.inf, np.float32)
    for r in range(i.shape[0]):
        ok = i[r] >= 0
        o = np.lexsort((i[r][ok], -s[r][ok].astype(np.float64)))[:k]
        oi[r, :o.size], os_[r, :o.size] = i[r][ok][o], s[r][ok][o]
    return oi, os_


@pytest.mark.parametrize("k", [10, 33])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_user_row_is_independent_of_the_call(engine_factory, precision, k):
    """A user's row is the same bits scored alone, among 3 SMs + 1 other users, with the users reversed, twice in one
    call, with the candidate list permuted, through score_topk_device on a non-default stream; and the two halves of the
    candidate list, merged by (score, id), give the full list."""
    C = 3
    rng, users, items, seen = _invariance_inputs()
    indptr, flat_seen = _csr(users, seen)
    flat, _, _ = _state(C)
    eng = _engine(engine_factory, precision, C, flat)
    mid = users.size // 2
    target = users[mid:mid + 1]
    alone = eng.score_topk(target, items, k, indptr, flat_seen)
    many = eng.score_topk(users, items, k, indptr, flat_seen)
    _same((many[0][mid:mid + 1], many[1][mid:mid + 1]), alone, "alone vs among many")
    rev = eng.score_topk(users[::-1].copy(), items, k, indptr, flat_seen)
    _same((rev[0][::-1], rev[1][::-1]), many, "reversed users")
    twice = eng.score_topk(np.array([users[0], target[0], users[1], target[0]], np.int32), items, k, indptr, flat_seen)
    for r in (1, 3):
        _same((twice[0][r:r + 1], twice[1][r:r + 1]), alone, "the user twice")
    perm = eng.score_topk(target, rng.permutation(items), k, indptr, flat_seen)
    _same(perm, alone, "permuted candidates")
    dev = torch.device("cuda", eng.device)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        di, ds = eng.score_topk_device(torch.from_numpy(target).to(dev), torch.from_numpy(items).to(dev), k,
                                       torch.from_numpy(indptr).to(dev), torch.from_numpy(flat_seen).to(dev))
    side.synchronize()
    _same((di.cpu().numpy(), ds.cpu().numpy()), alone, "score_topk_device on a side stream")
    few = users[:9]
    h = items.size // 2
    halves = _merge(eng.score_topk(few, items[:h], k, indptr, flat_seen),
                    eng.score_topk(few, items[h:], k, indptr, flat_seen), k)
    _same(halves, (many[0][:9], many[1][:9]), "two halves merged")


@pytest.mark.parametrize("k", [10, 33])
def test_bf16_scores_equal_tf32x3(engine_factory, k):
    """bf16 handles score through the same tf32 split as tf32x3: the same bits."""
    C = 2
    _, users, items, seen = _invariance_inputs()
    indptr, flat_seen = _csr(users, seen)
    flat, _, _ = _state(C)
    for mode in ("q", "policy"):
        a = _engine(engine_factory, "bf16", C, flat).score_topk(users, items, k, indptr, flat_seen, mode=mode)
        b = _engine(engine_factory, "tf32x3", C, flat).score_topk(users, items, k, indptr, flat_seen, mode=mode)
        _same(a, b, mode)


def test_fp32_user_slab_edge(engine_factory):
    """k_score_topk puts users on gridDim.y in slabs of 65 535: 65 637 users, rows 65 533..65 537 equal per-user calls
    (which take the multi-chunk + k_topk_merge path) and the oracle."""
    C, I, k = 2, 192, 10
    rng = np.random.default_rng(77)
    users = rng.integers(0, 6040, 65537 + 100).astype(np.int32)
    items = _candidates(rng, I)
    flat, _, _ = _state(C)
    eng = _engine(engine_factory, "fp32", C, flat)
    ti, ts = eng.score_topk(users, items, k)
    rows = np.arange(65533, 65538)
    for r in rows:
        _same((ti[r:r + 1], ts[r:r + 1]), eng.score_topk(users[r:r + 1], items, k), f"row {r}")
    budgeted = []
    _check_rows("slab", ti[rows], ts[rows], k, items, np.zeros((rows.size, I), bool), _oracle(C, users[rows], items, "q"),
                lambda r: _oracle(C, users[rows[r:r + 1]], items, "q", dtype=torch.float64)[0], budgeted)
    _report("fp32 slab edge", budgeted)


# ---------------------------------------------------------------- 7. score_pairs and predict
PAIRS = [pytest.param(p, C, m, id=f"{p}-C{C}-{m}") for C in (1, 2, 3, 4) for m in ("q", "policy") for p in PRECISIONS]


@pytest.mark.parametrize("precision,C,mode", PAIRS)
def test_score_pairs_matches_oracle(engine_factory, precision, C, mode):
    """k_score_pairs at n = 1, 63, 64, 65 (one 64-row tile and its edges) and 100 003 pairs."""
    rng = np.random.default_rng(88)
    n_max = 100003
    u = rng.integers(0, 6040, n_max).astype(np.int32)
    i = rng.integers(0, 30000, n_max).astype(np.int32)
    key = ("pairs", C, mode)
    if key not in _Q:
        _, st, _ = _state(C)
        _Q[key] = _relevance(st, np.stack([u, i], 1), mode, False, torch.float32)
    ref = _Q[key]
    flat, _, st64 = _state(C)
    eng = _engine(engine_factory, precision, C, flat)
    budgeted = []
    for n in (1, 63, 64, 65, n_max):
        got = eng.score_pairs(u[:n], i[:n], mode=mode)
        scale = max(1.0, float(np.max(np.abs(ref[:n]))))
        err = lambda a, b: float(np.max(np.abs(np.asarray(a, np.float64) - b))) / scale
        Hp.check_f64_budget((n,), got, ref[:n],
                            lambda n=n: _relevance(st64, np.stack([u[:n], i[:n]], 1), mode, False, torch.float64),
                            budgeted, tol=TOL, err=err)
    _report(f"{precision} C={C} {mode} pairs", budgeted)


@pytest.mark.parametrize("C", [1, 4])
def test_predict_and_predict_pairs_agree_at_critic_count(C):
    from replay_cql_b200.models import CQL
    from replay_cql_b200.synthetic import make_log
    log = make_log("tiny")
    model = CQL(top_k=3, n_epochs=2, batch_size=64, seed=3, n_critics=C)
    model.fit(log)
    try:
        recs = model.predict(log, k=4, filter_seen_items=False)
        pairs = model.predict_pairs(recs[["user_idx", "item_idx"]], log)
        merged = recs.merge(pairs, on=["user_idx", "item_idx"], suffixes=("_a", "_b"))
        assert len(merged) == len(recs) > 0
        scale = max(1.0, merged["relevance_a"].abs().max())
        assert (merged["relevance_a"] - merged["relevance_b"]).abs().max() <= TOL * scale
    finally:
        model.engine.close()


# ---------------------------------------------------------------- 8. negative candidate ids
@pytest.mark.parametrize("k", [10, 33])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_negative_candidate_ids_are_skipped(engine_factory, precision, k):
    """-1 entries in the candidate list are never returned: every row equals, bit for bit, the result without them
    (score_topk and score_topk_device).  A list shorter than k makes every entry a candidate of the fold."""
    C = 2
    rng = np.random.default_rng(99)
    users = rng.choice(6040, size=3, replace=False).astype(np.int32)
    flat, _, _ = _state(C)
    eng = _engine(engine_factory, precision, C, flat)
    dev = torch.device("cuda", eng.device)
    for I, n_neg in ((8, 3), (4097, 40)):
        clean = _candidates(rng, I)
        pos = np.sort(np.concatenate([[0, I], rng.choice(np.arange(1, I), n_neg - 2, replace=False)]))
        dirty = np.insert(clean, pos, -1).astype(np.int32)
        seen = {int(users[1]): set(rng.choice(clean, size=I // 4, replace=False).tolist())}
        indptr, flat_seen = _csr(users, seen)
        want = eng.score_topk(users, clean, k, indptr, flat_seen)
        got = eng.score_topk(users, dirty, k, indptr, flat_seen)
        real = got[0][np.isfinite(got[1])]
        assert not np.any(real < 0), (I, "a negative id was returned", got[0])
        _same(got, want, (I, "with -1 entries"))
        di, ds = eng.score_topk_device(*(torch.from_numpy(x).to(dev) for x in (users, dirty)), k,
                                       torch.from_numpy(indptr).to(dev), torch.from_numpy(flat_seen).to(dev))
        torch.cuda.synchronize()
        _same((di.cpu().numpy(), ds.cpu().numpy()), want, (I, "score_topk_device with -1 entries"))
