// score.cuh -- K5: batched user x item relevance, seen filter, per-user top-k.
//
// Scores are never materialised: a CTA owns (user, item chunk), pushes 64-item
// tiles through actor (greedy action) and the C critics, and a warp folds the
// tile into a running top-k held in shared memory.  The seen filter is *lazy*:
// only candidates that already beat the current k-th score are looked up in the
// user's sorted seen list (CSR), so the filter costs nothing on the hot loop.
// Order: relevance desc, then item id asc (the reference leaves ties arbitrary,
// replay/utils.py:125).
#pragma once
#include "engine.cuh"

namespace cql {

__device__ __forceinline__ bool better(float s, int i, float s2, int i2) {
  return s > s2 || (s == s2 && (unsigned)i < (unsigned)i2);  // item -1 (empty slot) sorts last
}

__device__ __forceinline__ bool is_seen(const int32_t* __restrict__ seen, int64_t lo, int64_t hi, int item) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int v = __ldg(seen + mid);
    if (v == item) return true;
    if (v < item) lo = mid + 1; else hi = mid;
  }
  return false;
}

// The lazy filter does one binary search per surviving candidate; from global memory that is ~8 dependent
// L2 round trips (~4 us), which dominated the fold.  Users' seen lists are short (ML-20M: 144 on average), so
// each CTA stages the current user's list in shared memory once and searches it there.
constexpr int SEEN_CACHE = 4096;       // ints of shared memory per CTA; longer lists fall back to global memory
struct SeenView {
  const int32_t* g;      // global list [lo, hi)
  const int32_t* s;      // shared-memory copy or nullptr
  int64_t lo, hi;
};
template <int MAXN = SEEN_CACHE>   // MAXN: power of two >= the longest cached list
__device__ __forceinline__ bool is_seen(const SeenView& v, int item) {
  if (v.s != nullptr) {
    // branch-free lower bound with a fixed trip count: the lanes of a warp that search at the same time stay
    // converged (a data-dependent loop serialises them -- measured 7 searching lanes ~ 3.5 k cycles)
    const int n = (int)(v.hi - v.lo);
    int lo = 0;
#pragma unroll
    for (int step = MAXN / 2; step >= 1; step >>= 1) {
      const int p = lo + step;
      if (p <= n && v.s[p - 1] < item) lo = p;
    }
    return lo < n && v.s[lo] == item;
  }
  return is_seen(v.g, v.lo, v.hi, item);
}
// cooperative stage by `nthreads` threads (tid in [0, nthreads)); caller synchronises afterwards
__device__ __forceinline__ SeenView stage_seen(const int64_t* __restrict__ indptr, const int32_t* __restrict__ seen,
                                               int user, int32_t* cache, int tid, int nthreads) {
  SeenView v{seen, nullptr, 0, 0};
  if (indptr == nullptr) return v;
  v.lo = indptr[user];
  v.hi = indptr[user + 1];
  const int64_t n = v.hi - v.lo;
  if (n <= SEEN_CACHE) {
    for (int64_t i = tid; i < n; i += nthreads) cache[i] = __ldg(seen + v.lo + i);
    v.s = cache;
  }
  return v;
}

// Whole-warp insertion of (s,i) into the descending list top[0..k).  Caller guarantees
// the candidate beats top[k-1].
__device__ __forceinline__ void warp_topk_insert(float* topS, int* topI, int k, float s, int i) {
  const int lane = threadIdx.x & 31;
  int cnt = 0;
  for (int e = lane; e < k; e += 32) cnt += better(topS[e], topI[e], s, i) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  const int pos = cnt;
  for (int base = ((k - 1) / 32) * 32; base + 31 > pos; base -= 32) {   // chunks from the top down
    const int e = base + lane;
    float ps = 0.f; int pi = 0;
    const bool mv = e > pos && e < k;
    if (mv) { ps = topS[e - 1]; pi = topI[e - 1]; }
    __syncwarp();
    if (mv) { topS[e] = ps; topI[e] = pi; }
    __syncwarp();
    if (base == 0) break;
  }
  if (lane == 0) { topS[pos] = s; topI[pos] = i; }
  __syncwarp();
}

// Fold up to 64 candidates (cs/ci in smem; invalid = item < 0) into the list.  Executed by warp 0.
__device__ __forceinline__ void warp_fold_tile(float* topS, int* topI, int k, const float* cs, const int* ci, int cnt,
                                               const int32_t* __restrict__ seen, int64_t lo, int64_t hi) {
  const int lane = threadIdx.x & 31;
  for (int base = 0; base < cnt; base += 32) {
    const int r = base + lane;
    const float s = r < cnt ? cs[r] : -INFINITY;
    const int i = r < cnt ? ci[r] : -1;
    bool cand = i >= 0 && better(s, i, topS[k - 1], topI[k - 1]);
    if (cand && seen != nullptr && is_seen(seen, lo, hi, i)) cand = false;
    unsigned m = __ballot_sync(0xffffffffu, cand);
    while (m) {
      const int src = __ffs(m) - 1;
      m &= m - 1;
      const float s2 = __shfl_sync(0xffffffffu, s, src);
      const int i2 = __shfl_sync(0xffffffffu, i, src);
      if (better(s2, i2, topS[k - 1], topI[k - 1])) warp_topk_insert(topS, topI, k, s2, i2);
    }
  }
}

// ---- order-independent fold of a block of scores into a (reset) top-k list, k <= 32, by 128 threads -------------
// The sequential fold above inserts every candidate that beats the current k-th entry: with scores that grow along
// the block (raw item ids as inputs make Q nearly monotone in the item index) EVERY item enters the list and the
// fold costs as much as the MMAs (measured 205 ms vs 130 ms per 2048 users).  This variant is a two-pass selection
// like topk_staged.cuh: thread maxima -> 32 group maxima -> threshold T = the (k + spare)-th largest -> only
// elements >= T are looked up (item id, seen list) and inserted; if seen items ate the candidates T is lowered and
// only the band [T_new, T_old) is collected.  Cost per block is ~constant.  Candidate overflow (massive ties)
// falls back to the sequential fold of the band.  `scr` = 4 + 32 + 2*FB_CAP words of shared memory; all 128
// threads call it (bar_id = their named barrier); the list topS/topI must be reset to (-inf, -1) by the caller.
constexpr int FB_CAP = 96;
constexpr int FB_SCRATCH_WORDS = 4 + 32 + 2 * FB_CAP;
__device__ __forceinline__ void fold_block_select(const float* __restrict__ score, int rows, const int32_t* __restrict__ items,
                                                  int64_t i0, const SeenView& sv, bool has_seen, int k, float* topS, int* topI,
                                                  float* scr, int etid, int bar_id) {
  volatile int* ncand = reinterpret_cast<volatile int*>(scr);
  volatile int* done = reinterpret_cast<volatile int*>(scr) + 1;
  volatile float* t_lo_s = scr + 2;
  volatile float* t_hi_s = scr + 3;
  float* gmax = scr + 4;
  float* candS = scr + 36;
  int* candI = reinterpret_cast<int*>(scr + 36 + FB_CAP);
  const int lane = etid & 31, ew = etid >> 5;
  // pass 1: thread maximum over its strided share, group maxima of 4 lanes
  float m = -INFINITY;
  for (int r = etid; r < rows; r += 128) m = fmaxf(m, score[r]);
  float g = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
  g = fmaxf(g, __shfl_xor_sync(0xffffffffu, g, 2));
  if ((lane & 3) == 0) gmax[ew * 8 + (lane >> 2)] = g;
  if (etid == 0) { *ncand = 0; *done = 0; }
  asm volatile("bar.sync %0, 128;" ::"r"(bar_id));
  // every warp ranks the 32 group maxima itself (counting, no dependent chain)
  const float mine = gmax[lane];
  int pos = 0;
#pragma unroll
  for (int t = 0; t < 32; ++t) {
    const float o = gmax[t];
    pos += (o > mine || (o == mine && t < lane)) ? 1 : 0;
  }
  int rank = min(32, k + 4 + (k >> 1));
  float t_hi = INFINITY;
  float t_lo = __shfl_sync(0xffffffffu, mine, __ffs(__ballot_sync(0xffffffffu, pos == rank - 1)) - 1);
  while (true) {
    // pass 2: elements of the band, unseen, with their item ids
    if (m >= t_lo) {
      for (int r = etid; r < rows; r += 128) {
        const float s = score[r];
        if (!(s >= t_lo && s < t_hi)) continue;
        const int item = __ldg(items + i0 + r);
        if (item < 0) continue;                        // never returned, as in the sequential folds
        if (has_seen && is_seen(sv, item)) continue;
        const int p = atomicAdd(const_cast<int*>(ncand), 1);
        if (p < FB_CAP) { candS[p] = s; candI[p] = item; }
      }
    }
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id));
    if (ew == 0) {
      const int n = *ncand;
      if (n > FB_CAP) {                               // overflow: sequential fold of the band
        for (int base = 0; base < rows; base += 32) {
          const int r = base + lane;
          const float s = r < rows ? score[r] : -INFINITY;
          const int item = r < rows ? __ldg(items + i0 + r) : -1;
          bool cand = item >= 0 && s >= t_lo && s < t_hi && better(s, item, topS[k - 1], topI[k - 1]);
          if (cand && has_seen && is_seen(sv, item)) cand = false;
          unsigned mm = __ballot_sync(0xffffffffu, cand);
          while (mm) {
            const int src = __ffs(mm) - 1;
            mm &= mm - 1;
            const float s2 = __shfl_sync(0xffffffffu, s, src);
            const int i2 = __shfl_sync(0xffffffffu, item, src);
            if (better(s2, i2, topS[k - 1], topI[k - 1])) warp_topk_insert(topS, topI, k, s2, i2);
          }
        }
      } else {
        for (int e = 0; e < n; ++e) {                  // ~k + 8 inserts, whatever the order of the scores
          const float s2 = candS[e];
          const int i2 = candI[e];
          if (better(s2, i2, topS[k - 1], topI[k - 1])) warp_topk_insert(topS, topI, k, s2, i2);
        }
      }
      __syncwarp();
      // nothing below t_lo can belong to the top-k once the k-th entry reaches t_lo
      const bool settled = (topI[k - 1] >= 0 && topS[k - 1] >= t_lo) || t_lo == -INFINITY;
      if (lane == 0) {
        if (settled) {
          *done = 1;
        } else {
          int n_ok = 0;
          for (int e = 0; e < k; ++e) n_ok += (topI[e] >= 0 && topS[e] >= t_lo) ? 1 : 0;
          int rk = rank + max(2, 2 * (k - n_ok));
          // (gmax is unsorted: the new threshold is recomputed by every warp from `rank`, published here)
          *t_hi_s = t_lo;
          *t_lo_s = __int_as_float(rk);                // carries the new rank; every warp derives t_lo from it
          *ncand = 0;
        }
      }
    }
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id));
    if (*done) break;
    rank = __float_as_int(*t_lo_s);
    t_hi = *t_hi_s;
    // skip group maxima equal to the old threshold (they were collected already)
    {
      float nt = -INFINITY;
      bool found = false;
      while (rank <= 32 && !found) {
        const unsigned hit = __ballot_sync(0xffffffffu, pos == rank - 1);
        nt = __shfl_sync(0xffffffffu, mine, __ffs(hit) - 1);
        if (nt < t_hi) found = true; else ++rank;
      }
      t_lo = found ? nt : -INFINITY;
    }
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id));     // every thread has read the round's control words
  }
}

struct ScoreArgs {
  const float* params;        // flat state
  const int32_t* users;       // [U]
  const int32_t* items;       // [I]
  const int64_t* seen_indptr; // [max_user+2] CSR over user id, or nullptr
  const int32_t* seen_items;
  int64_t n_users, n_items;
  int C, k, mode, chunks, tiles_per_chunk;
  float* part_s;              // [U][chunks][k]
  int* part_i;
  const float* item_x;        // [I] scaled item coordinates (obs scaler on), or nullptr: (float)item
  Prep prep;                  // user coordinate and the policy score's reverse action transform
};

constexpr int SCORE_SMEM_BASE = FWD_SMEM;
inline int score_smem(int k) { return SCORE_SMEM_BASE + k * 8 + BM * 8; }

// obs scaler on: the scaled item coordinates of a candidate list, once per scoring call -- the tensor-core producers
// would otherwise divide once per (user, item) pair
__global__ void k_scale_items(const int32_t* __restrict__ items, int64_t n, const Affine f, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = prep_fwd(f, (float)items[i]);
}

// relevance of the 64 rows in Xs (x = user, y = item); result in sc[r] (smem) after return
__device__ __forceinline__ void score_tile(const float* __restrict__ params, int C, int mode, float4* Xs, float* As,
                                           float* Bs, float* outs, float* sc, const Affine& act) {
  const int tid = threadIdx.x;
  fwd_tile<2, 2>(params + (size_t)slot_actor() * NET_STRIDE, Xs, As, Bs, outs, nullptr);
  float a = 0.f;
  if (tid < BM) {
    a = tanhf(outs[tid * 2]);
    Xs[tid].z = a;
  }
  __syncthreads();
  if (mode == CQL_SCORE_POLICY) {
    if (tid < BM) sc[tid] = act_rev(act, a);     // relevance in the data's action units
    __syncthreads();
    return;
  }
  float q = 0.f;
  for (int c = 0; c < C; ++c) {
    fwd_tile<3, 1>(params + (size_t)slot_critic(c) * NET_STRIDE, Xs, As, Bs, outs, nullptr);
    if (tid < BM) q += outs[tid];
    __syncthreads();
  }
  if (tid < BM) sc[tid] = q / (float)C;
  __syncthreads();
}

__global__ void __launch_bounds__(NT, 2) k_score_topk(const ScoreArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* As = smem;
  float* Bs = As + H * BM;
  float4* Xs = reinterpret_cast<float4*>(Bs + 2 * BK * H);
  float* topS = reinterpret_cast<float*>(Xs + BM);
  int* topI = reinterpret_cast<int*>(topS + a.k);
  float* cs = reinterpret_cast<float*>(topI + a.k);
  int* ci = reinterpret_cast<int*>(cs + BM);
  __shared__ float outs[BM * 2];
  const int tid = threadIdx.x;
  const int64_t urow = blockIdx.y;
  const int user = a.users[urow];
  const float uf = prep_fwd(a.prep.obs[0], (float)user);
  for (int e = tid; e < a.k; e += NT) { topS[e] = -INFINITY; topI[e] = -1; }
  int64_t lo = 0, hi = 0;
  if (a.seen_indptr) { lo = a.seen_indptr[user]; hi = a.seen_indptr[user + 1]; }
  const int64_t tile0 = (int64_t)blockIdx.x * a.tiles_per_chunk;
  for (int t = 0; t < a.tiles_per_chunk; ++t) {
    const int64_t i0 = (tile0 + t) * BM;
    if (i0 >= a.n_items) break;
    const int cnt = (int)min((int64_t)BM, a.n_items - i0);
    if (tid < BM) {
      const int item = tid < cnt ? a.items[i0 + tid] : -1;
      Xs[tid] = make_float4(uf, a.item_x && tid < cnt ? a.item_x[i0 + tid] : (float)max(item, 0), 0.f, 0.f);
      ci[tid] = item;
    }
    __syncthreads();
    score_tile(a.params, a.C, a.mode, Xs, As, Bs, outs, cs, a.prep.act);
    if (tid < 32) warp_fold_tile(topS, topI, a.k, cs, ci, cnt, a.seen_indptr ? a.seen_items : nullptr, lo, hi);
    __syncthreads();
  }
  float* ps = a.part_s + ((size_t)urow * a.chunks + blockIdx.x) * a.k;
  int* pi = a.part_i + ((size_t)urow * a.chunks + blockIdx.x) * a.k;
  for (int e = tid; e < a.k; e += NT) { ps[e] = topS[e]; pi[e] = topI[e]; }
}

// merge the per-chunk lists of one user (one warp per user; lists are sorted, already seen-filtered)
__global__ void k_topk_merge(const float* __restrict__ part_s, const int* __restrict__ part_i, int64_t n_users,
                             int chunks, int k, float* __restrict__ out_s, int* __restrict__ out_i) {
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int64_t u = (int64_t)blockIdx.x * wpb + warp;
  float* topS = smem + (size_t)warp * 2 * k;
  int* topI = reinterpret_cast<int*>(topS + k);
  if (u >= n_users) return;
  for (int e = lane; e < k; e += 32) { topS[e] = -INFINITY; topI[e] = -1; }
  __syncwarp();
  for (int c = 0; c < chunks; ++c) {
    const float* ps = part_s + ((size_t)u * chunks + c) * k;
    const int* pi = part_i + ((size_t)u * chunks + c) * k;
    for (int e = 0; e < k; ++e) {
      const float s = ps[e];
      const int i = pi[e];
      if (i < 0 || !better(s, i, topS[k - 1], topI[k - 1])) break;  // sorted: nothing further can enter
      warp_topk_insert(topS, topI, k, s, i);
    }
  }
  for (int e = lane; e < k; e += 32) { out_s[u * k + e] = topS[e]; out_i[u * k + e] = topI[e]; }
}

// explicit (user,item) pairs -> relevance
__global__ void __launch_bounds__(NT, 2) k_score_pairs(const float* __restrict__ params, const int32_t* __restrict__ users,
                                                       const int32_t* __restrict__ items, int64_t n, int C, int mode,
                                                       float* __restrict__ out, const Prep prep) {
  extern __shared__ __align__(16) float smem[];
  float* As = smem;
  float* Bs = As + H * BM;
  float4* Xs = reinterpret_cast<float4*>(Bs + 2 * BK * H);
  __shared__ float outs[BM * 2];
  __shared__ float sc[BM];
  const int tid = threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.x * BM;
  if (tid < BM) {
    const int64_t r = r0 + tid;
    Xs[tid] = r < n ? make_float4(prep_fwd(prep.obs[0], (float)users[r]), prep_fwd(prep.obs[1], (float)items[r]), 0.f, 0.f)
                    : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  score_tile(params, C, mode, Xs, As, Bs, outs, sc, prep.act);
  if (tid < BM && r0 + tid < n) out[r0 + tid] = sc[tid];
}

// ---- stand-alone HBM-bound top-k + lazy seen filter over materialised scores [U][I] ----
// One CTA per user row; each warp streams a strided share of the row with 16-byte loads and
// keeps its own list; warp 0 merges the lists.  k <= 32 per-warp lists live in smem.
__global__ void __launch_bounds__(256) k_topk_filter(const float* __restrict__ scores, int64_t n_items,
                                                     const int32_t* __restrict__ users, const int32_t* __restrict__ items,
                                                     const int64_t* __restrict__ seen_indptr,
                                                     const int32_t* __restrict__ seen_items, int k,
                                                     float* __restrict__ out_s, int* __restrict__ out_i) {
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  float* topS = smem + (size_t)warp * 2 * k;
  int* topI = reinterpret_cast<int*>(topS + k);
  const int64_t urow = blockIdx.x;
  const int user = users ? users[urow] : (int)urow;
  int32_t* cache = reinterpret_cast<int32_t*>(smem + (size_t)nw * 2 * k);
  const SeenView sv = stage_seen(seen_indptr, seen_items, user, cache, threadIdx.x, blockDim.x);
  for (int e = lane; e < k; e += 32) { topS[e] = -INFINITY; topI[e] = -1; }
  __syncthreads();
  const float* row = scores + (size_t)urow * n_items;
  const bool vec_ok = ((reinterpret_cast<uintptr_t>(row) & 15) == 0);
  const int64_t nvec = vec_ok ? n_items / 4 : 0;
  // vector body: 4 x float4 in flight per lane; one warp vote per 16 values decides whether ANY of them can
  // enter the list (after the first few hundred values almost none can), so the steady state is load + max
  for (int64_t v0 = (int64_t)warp * 128; v0 < nvec; v0 += (int64_t)nw * 128) {
    float4 x[4];
    int64_t vi[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      vi[q] = v0 + q * 32 + lane;
      x[q] = vi[q] < nvec ? __ldcs(reinterpret_cast<const float4*>(row) + vi[q])
                          : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
    float mx = -INFINITY;
#pragma unroll
    for (int q = 0; q < 4; ++q) mx = fmaxf(mx, fmaxf(fmaxf(x[q].x, x[q].y), fmaxf(x[q].z, x[q].w)));
    if (!__any_sync(0xffffffffu, mx >= topS[k - 1])) continue;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float vals[4] = {x[q].x, x[q].y, x[q].z, x[q].w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int64_t col = vi[q] * 4 + c;
        const float s = vals[c];
        int item = -1;
        bool cand = vi[q] < nvec && s >= topS[k - 1];
        if (cand) {
          item = items ? items[col] : (int)col;
          cand = better(s, item, topS[k - 1], topI[k - 1]);
          if (cand && seen_indptr && is_seen(sv, item)) cand = false;
        }
        unsigned m = __ballot_sync(0xffffffffu, cand);
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const float s2 = __shfl_sync(0xffffffffu, s, src);
          const int i2 = __shfl_sync(0xffffffffu, item, src);
          if (better(s2, i2, topS[k - 1], topI[k - 1])) warp_topk_insert(topS, topI, k, s2, i2);
        }
      }
    }
  }
  // scalar tail (and the whole row when it is not 16-byte aligned)
  for (int64_t c0 = nvec * 4 + (int64_t)warp * 32; c0 < n_items; c0 += (int64_t)nw * 32) {
    const int64_t col = c0 + lane;
    const float s = col < n_items ? row[col] : -INFINITY;
    int item = -1;
    bool cand = col < n_items && s >= topS[k - 1];
    if (cand) {
      item = items ? items[col] : (int)col;
      cand = better(s, item, topS[k - 1], topI[k - 1]);
      if (cand && seen_indptr && is_seen(sv, item)) cand = false;
    }
    unsigned m = __ballot_sync(0xffffffffu, cand);
    while (m) {
      const int src = __ffs(m) - 1;
      m &= m - 1;
      const float s2 = __shfl_sync(0xffffffffu, s, src);
      const int i2 = __shfl_sync(0xffffffffu, item, src);
      if (better(s2, i2, topS[k - 1], topI[k - 1])) warp_topk_insert(topS, topI, k, s2, i2);
    }
  }
  __syncthreads();
  if (warp == 0) {
    for (int w = 1; w < nw; ++w) {
      const float* ps = smem + (size_t)w * 2 * k;
      const int* pi = reinterpret_cast<const int*>(ps + k);
      for (int e = 0; e < k; ++e) {
        const float s = ps[e];
        const int i = pi[e];
        if (i < 0 || !better(s, i, topS[k - 1], topI[k - 1])) break;
        warp_topk_insert(topS, topI, k, s, i);
      }
    }
    for (int e = lane; e < k; e += 32) { out_s[urow * k + e] = topS[e]; out_i[urow * k + e] = topI[e]; }
  }
}

}  // namespace cql
