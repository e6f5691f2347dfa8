// update.cuh -- one CQL update: replay sampling, noise, loss glue, Adam/Polyak, phase driver.
//
// Order of one update (SURVEY.md Appendix A): temp -> alpha -> critic -> actor -> Polyak.
// The actor does not change until the very end, so its forward on s and s' is
// computed ONCE and shared by the temp step, both conservative-loss evaluations,
// the TD target and the actor step (a result-preserving saving, DESIGN.md).
#pragma once
#include <algorithm>
#include <utility>
#include "engine.cuh"
#include "mlp_tc.cuh"
#include "mlp_tc_ts.cuh"
#include <type_traits>
#include "mlp_tc_bwd1.cuh"
#include "mlp_tc_bwd2.cuh"
#include "mlp_tc_h.cuh"
#include "mlp_tc_h2.cuh"
#include "adam_pack.cuh"

namespace cql {

// ---------------------------------------------------------------- K1: replay sampling
// Bijective pseudo-random permutation of [0, n): 4-round Feistel over 2*hb bits + cycle walking.
__host__ __device__ inline uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
__host__ __device__ inline uint64_t feistel_perm(uint64_t x, uint64_t n, uint64_t key) {
  int bits = 2;
  while (bits < 62 && (1ull << bits) < n) bits += 2;   // even number of bits >= log2(n)
  const int hb = bits / 2;
  const uint64_t mask = (1ull << hb) - 1;
  do {
    uint64_t l = x >> hb, r = x & mask;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t f = mix32((uint32_t)r * 0x9E3779B1u + (uint32_t)(key >> (i * 13)) + 0x85ebca6bu * (i + 1) +
                               (uint32_t)(r >> 16) * 0xc2b2ae35u);
      const uint64_t nl = r, nr = (l ^ f) & mask;
      l = nl; r = nr;
    }
    x = (l << hb) | r;
  } while (x >= n);
  return x;
}

// position p of the sampling stream -> transition index.  An epoch covers n_eff = n - n % chunk
// positions (d3rlpy drops the last partial minibatch); each epoch uses a fresh permutation.
__host__ __device__ inline int64_t stream_index(int64_t p, int64_t n, int64_t chunk, uint64_t seed) {
  int64_t n_eff = n - n % chunk;
  if (n_eff <= 0) n_eff = n;
  const int64_t epoch = p / n_eff, q = p % n_eff;
  return (int64_t)feistel_perm((uint64_t)q, (uint64_t)n, seed * 0x9E3779B97F4A7C15ull + (uint64_t)epoch * 0xD1B54A32D192ED03ull + 1);
}

// One thread per row: two 16-byte loads of a 32-byte transition row (one DRAM sector).
__global__ void k_sample(const float4* __restrict__ table, int64_t n_trans, const int64_t* __restrict__ idx,
                         const long long* __restrict__ step_dev, int64_t pos0, int64_t count, int64_t chunk,
                         int rank, int world, uint64_t seed, float4* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= count) return;
  int64_t t;
  if (idx) {
    t = idx[j];
  } else {
    // training: position = (completed_steps * world + rank) * B + j ; stand-alone sweep: pos0 + j
    const int64_t p = step_dev ? ((int64_t)(*step_dev) * world + rank) * count + j : pos0 + j;
    t = stream_index(p, n_trans, chunk, seed);
  }
  const float4 a = __ldg(table + 2 * t), b = __ldg(table + 2 * t + 1);
  out[2 * j] = a;
  out[2 * j + 1] = b;
}

// episode-ordered steps -> transition rows
__global__ void k_build_transitions(const float2* __restrict__ obs, const float* __restrict__ act,
                                    const float* __restrict__ rew, const float* __restrict__ term, int64_t n,
                                    float4* __restrict__ table) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float2 o = obs[i];
  const float tm = term[i];
  float2 nx = make_float2(0.f, 0.f);
  if (tm == 0.f && i + 1 < n) nx = obs[i + 1];
  table[2 * i] = make_float4(o.x, o.y, act[i], rew[i]);
  table[2 * i + 1] = make_float4(nx.x, nx.y, tm, 0.f);
}

// Synthetic replay table of a BASELINE shape generated in place (bench / stress configuration: 1e9 rows = 32 GB would
// not fit through the host).  Episodes are user-major with a fixed length L = ceil(n / n_users); item ~ Zipf(1)-like
// (inverse-CDF of 1/x on [1, n_items]), action = rating in {1..5} (ML-like pmf) + N(0, 1e-3), reward = 1 on ~10 rows
// per episode, terminal on the episode's last row.  Row i depends only on (seed, i): reproducible.
__device__ __forceinline__ float2 synth_obs(int64_t i, int64_t L, int64_t n_users, int64_t n_items, uint64_t seed, uint32_t (&r)[4]) {
  Philox::gen(seed ^ 0x53594E5448ull, 0x7ab1eull, (uint64_t)i, r);
  const int64_t u = i / L < n_users ? i / L : n_users - 1;
  const float z = expf(u01(r[0]) * logf((float)n_items));          // in [1, n_items]
  int64_t it = (int64_t)z - 1;
  it = it < 0 ? 0 : (it >= n_items ? n_items - 1 : it);
  return make_float2((float)u, (float)it);
}
__global__ void k_synth_table(float4* __restrict__ table, int64_t n, int64_t n_users, int64_t n_items, uint64_t seed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t L = (n + n_users - 1) / n_users;
  uint32_t r[4], r2[4];
  const float2 o = synth_obs(i, L, n_users, n_items, seed, r);
  const bool last = (i == n - 1) || ((i + 1) / L != i / L && i / L < n_users - 1) ;
  const float u = u01(r[1]);
  const float rating = u < 0.06f ? 1.f : (u < 0.17f ? 2.f : (u < 0.43f ? 3.f : (u < 0.78f ? 4.f : 5.f)));
  const float nz = sqrtf(-2.f * logf(u01(r[2]))) * cospif(2.f * u01(r[3])) * 1e-3f;
  const float rew = (r[3] % (uint32_t)L) < 10u ? 1.f : 0.f;
  float2 nx = make_float2(0.f, 0.f);
  if (!last) nx = synth_obs(i + 1, L, n_users, n_items, seed, r2);
  table[2 * i] = make_float4(o.x, o.y, rating + nz, rew);
  table[2 * i + 1] = make_float4(nx.x, nx.y, last ? 1.f : 0.f, 0.f);
}

// One-step rows -> n-step rows (d3rlpy n_steps, DESIGN.md section 1), out of place: row t reads rows t .. t + n_steps - 1.
// k = min(n_steps, steps from t to its episode's end, t included); an episode ends at a terminal row or at the table's end.
// R and the discount g are accumulated in float64 in the pinned order (R += g * r, then g *= gamma) with explicit
// roundings, so k = 1 gives R = r and g = gamma exactly; s' and term are row t + k - 1's.  A block stages its
// NSTEP_TILE rows plus the n_steps - 1 halo rows in shared memory with coalesced 16-byte loads, then each thread walks
// its window there.
constexpr int NSTEP_TILE = 256;
__global__ void __launch_bounds__(NSTEP_TILE) k_nstep_rows(const float4* __restrict__ src, int64_t n, int n_steps,
                                                           double gamma, float4* __restrict__ dst) {
  extern __shared__ float4 tile[];           // [NSTEP_TILE + n_steps - 1][2]
  const int64_t base = (int64_t)blockIdx.x * NSTEP_TILE;
  const int rows = (int)min((int64_t)(NSTEP_TILE + n_steps - 1), n - base);
  for (int q = threadIdx.x; q < 2 * rows; q += NSTEP_TILE) tile[q] = src[2 * base + q];
  __syncthreads();
  const int t = threadIdx.x;
  if (base + t >= n) return;
  double R = 0.0, g = 1.0;
  int last = t;
  for (int j = 0; j < n_steps && t + j < rows; ++j) {
    last = t + j;
    R = __dadd_rn(R, __dmul_rn(g, (double)tile[2 * last].w));
    g = __dmul_rn(g, gamma);
    if (tile[2 * last + 1].z != 0.f) break;
  }
  const float4 a = tile[2 * t], b = tile[2 * last + 1];
  dst[2 * (base + t)] = make_float4(a.x, a.y, a.z, (float)R);
  dst[2 * (base + t) + 1] = make_float4(b.x, b.y, b.z, (float)g);
}

// Column statistics of one-step rows (d3rlpy's scaler fit, cql_get_table_stats): count, mean, M2, min, max of obs.x,
// obs.y, act and rew in float64.  Each thread runs Welford's update over its rows (j = t, t + 256, ... of the block's
// STATS_ROWS), the block merges its threads with Chan's formula in a fixed tree, and k_stats_final merges the block
// partials the same way: the order depends only on n, so the same rows always give the same bits.
struct Moments { double n, mean, m2, mn, mx; };
__device__ __forceinline__ Moments mom_merge(Moments a, const Moments& b) {
  if (b.n == 0.0) return a;
  if (a.n == 0.0) return b;
  const double n = a.n + b.n, d = b.mean - a.mean;
  a.mean = a.mean + d * (b.n / n);
  a.m2 = a.m2 + b.m2 + d * d * (a.n * b.n / n);
  a.mn = fmin(a.mn, b.mn);
  a.mx = fmax(a.mx, b.mx);
  a.n = n;
  return a;
}
constexpr int STATS_THREADS = 256, STATS_ROWS = 32 * STATS_THREADS;
// blocks of k_stats_partial: ceil(n / STATS_ROWS), at most STATS_MAX_BLOCKS (then each takes ceil(n / blocks) rows); the
// partials live in the handle's stats_dev, [(STATS_MAX_BLOCKS + 1) * 4] Moments (engine.cuh: STATS_DEV_DOUBLES)
static_assert(sizeof(Moments) == 5 * sizeof(double), "Moments is five doubles");
static_assert(STATS_DEV_DOUBLES == (STATS_MAX_BLOCKS + 1) * 4 * 5, "stats_dev holds the partials and the result");
__device__ void stats_block_store(Moments (&m)[4], Moments* __restrict__ out) {
  __shared__ Moments sm[STATS_THREADS];
  for (int c = 0; c < 4; ++c) {
    sm[threadIdx.x] = m[c];
    __syncthreads();
    for (int s = STATS_THREADS / 2; s > 0; s >>= 1) {
      if (threadIdx.x < s) sm[threadIdx.x] = mom_merge(sm[threadIdx.x], sm[threadIdx.x + s]);
      __syncthreads();
    }
    if (threadIdx.x == 0) out[c] = sm[0];
    __syncthreads();
  }
}
__global__ void __launch_bounds__(STATS_THREADS) k_stats_partial(const float4* __restrict__ rows, int64_t n,
                                                                  int64_t per_block, Moments* __restrict__ part) {
  Moments m[4];
  for (int c = 0; c < 4; ++c) m[c] = Moments{0.0, 0.0, 0.0, INFINITY, -INFINITY};
  const int64_t base = (int64_t)blockIdx.x * per_block;
  for (int64_t j = threadIdx.x; j < per_block && base + j < n; j += STATS_THREADS) {
    const float4 r = rows[2 * (base + j)];
    const float v[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const double x = v[c];
      m[c].n += 1.0;
      const double d = x - m[c].mean;
      m[c].mean += d / m[c].n;
      m[c].m2 += d * (x - m[c].mean);
      m[c].mn = fmin(m[c].mn, x);
      m[c].mx = fmax(m[c].mx, x);
    }
  }
  stats_block_store(m, part + 4 * (size_t)blockIdx.x);
}
__global__ void __launch_bounds__(STATS_THREADS) k_stats_final(const Moments* __restrict__ part, int64_t nb,
                                                                Moments* __restrict__ out) {
  Moments m[4];
  for (int c = 0; c < 4; ++c) m[c] = Moments{0.0, 0.0, 0.0, INFINITY, -INFINITY};
  for (int64_t b = threadIdx.x; b < nb; b += STATS_THREADS)
    for (int c = 0; c < 4; ++c) m[c] = mom_merge(m[c], part[4 * b + c]);
  stats_block_store(m, out);
}

// ---------------------------------------------------------------- noise (Philox)
__global__ void k_noise(float* __restrict__ noise, int64_t total, int B, int n, uint64_t seed,
                        const long long* __restrict__ step_dev, int rank) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  uint32_t r[4];
  Philox::gen(seed ^ 0x5851F42D4C957F2Dull, ((uint64_t)(*step_dev) << 8) | (uint64_t)(rank & 0xff), (uint64_t)i, r);
  const int64_t Bn = (int64_t)B * n;
  const int64_t a = i - B;  // position inside the six B*n blocks
  const bool uniform = a >= 0 && a < 6 * Bn && ((a / Bn) % 3 == 2);
  const float u1 = u01(r[0]), u2 = u01(r[1]);
  noise[i] = uniform ? fmaf(2.f, u1, -1.f) : sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
}

// ---------------------------------------------------------------- step bookkeeping
__global__ void k_step_begin(const long long* step_dev, StepInfo* info, float beta1, float beta2) {
  const long long t = *step_dev + 1;
  info->step = t;
  info->bc1 = 1.0 - pow((double)beta1, (double)t);
  info->bc2_sqrt = sqrt(1.0 - pow((double)beta2, (double)t));
}
__global__ void k_step_end(long long* step_dev) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  *step_dev += 1; }

// sampled-update prologue in one launch: Adam bias corrections, replay gather (+ actor input rows), Philox noise
__global__ void k_step_head(const float4* __restrict__ table, int64_t n_trans, const long long* __restrict__ step_dev,
                            StepInfo* __restrict__ info, float beta1, float beta2, int B, int n, int rank, int world,
                            uint64_t seed, float4* __restrict__ batch, float4* __restrict__ XA,
                            float* __restrict__ noise, int64_t noise_total, int prank, int pworld, const Prep prep) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const long long done = *step_dev;
  if (i == 0) {
    const long long t = done + 1;
    info->step = t;
    info->bc1 = 1.0 - pow((double)beta1, (double)t);
    info->bc2_sqrt = sqrt(1.0 - pow((double)beta2, (double)t));
  }
  if (i < B) {
    // position in the epoch permutation: (rank, world) of the data-parallel job for a replicated table, (0, 1) when this
    // rank holds only its own user shard (prank / pworld); the Philox stream below always uses the job's rank
    const int64_t p = ((int64_t)done * pworld + prank) * B + i;
    const int64_t t = stream_index(p, n_trans, (int64_t)B * pworld, seed);
    float4 a = __ldg(table + 2 * t), b = __ldg(table + 2 * t + 1);
    if (prep.any()) { a = prep_row0(prep, a); b = prep_row1(prep, b); }   // the table stays raw: scaled at gather
    batch[2 * i] = a;
    batch[2 * i + 1] = b;
    XA[i] = make_float4(a.x, a.y, 0.f, 0.f);
    XA[B + i] = make_float4(b.x, b.y, 0.f, 0.f);
  }
  if (i < noise_total) {
    uint32_t r[4];
    Philox::gen(seed ^ 0x5851F42D4C957F2Dull, ((uint64_t)done << 8) | (uint64_t)(rank & 0xff), (uint64_t)i, r);
    const int64_t Bn = (int64_t)B * n;
    const int64_t a = i - B;
    const bool uniform = a >= 0 && a < 6 * Bn && ((a / Bn) % 3 == 2);
    const float u1 = u01(r[0]), u2 = u01(r[1]);
    noise[i] = uniform ? fmaf(2.f, u1, -1.f) : sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
  }
}

// ---------------------------------------------------------------- squashed Gaussian
struct Sample { float a, logp, raw, t, std_; };
__device__ __forceinline__ float softplus_t(float x) { return x > 20.f ? x : log1pf(expf(x)); }
// Mirrors the oracle op by op (separately rounded mul/add, no FMA contraction): the
// log(1 - a^2 + 1e-6) term is ill-conditioned near |a| -> 1, so even the rounding of a*a matters.
__device__ __forceinline__ Sample policy_sample(float mu, float ls, float eps, int squash) {
  Sample s;
  s.std_ = expf(ls);
  s.raw = __fadd_rn(mu, __fmul_rn(s.std_, eps));
  s.a = (float)tanh((double)s.raw);   // correctly rounded: log(1-a^2+1e-6) amplifies tanh's last ulp ~1e6x
  s.t = __fdiv_rn(__fsub_rn(s.raw, mu), s.std_);
  const float normal_logp =
      __fsub_rn(__fsub_rn(__fmul_rn(-0.5f, __fmul_rn(s.t, s.t)), ls), 0.91893853320467274f);
  float logdet;
  if (squash == CQL_SQUASH_EPS) {
    logdet = logf(__fadd_rn(__fsub_rn(1.f, __fmul_rn(s.a, s.a)), 1e-6f));
  } else {
    logdet = __fmul_rn(2.f, __fsub_rn(__fsub_rn(0.69314718055994531f, s.raw), softplus_t(__fmul_rn(-2.f, s.raw))));
  }
  s.logp = __fsub_rn(normal_logp, logdet);
  return s;
}
__device__ __forceinline__ float clamp_ls(float x) { return fminf(fmaxf(x, -20.f), 2.f); }

// Where the layer-3 outputs of a forward job live: final values [n_nets][rows][OUT] (n_parts == 0: FP32 path, or after
// k_sum_partials_multi) or the tensor-core kernels' partial sums [n_nets][n_parts][rows][OUT] with the bias b3 still to
// add.  The consumers of a forward (k_prep, k_lse, k_actor_dq) read through q_at(), which adds the parts in the order
// k_sum_partials_multi does -- the separate summation launch (three per update) is gone, the results are bit-identical.
struct QSrc {
  const float* q;
  const float* params;     // first net slot (b3), used when n_parts > 0
  int n_parts, rows, in_dim, out_dim;
};
// (all parts and the bias are REQUESTED before the first addition: a `v += q[p]` loop with a run-time trip count walks
// through n_parts dependent L2 round trips -- the top stall sites of k_lse and k_prep in the r02 ncu capture; the order
// of the additions is unchanged)
constexpr int Q_MAX_PARTS = 8;
__device__ __forceinline__ float q_at(const QSrc& s, int net, int r, int o = 0) {
  if (s.n_parts == 0) return s.q[((size_t)net * s.rows + r) * s.out_dim + o];
  float part[Q_MAX_PARTS];
#pragma unroll
  for (int p = 0; p < Q_MAX_PARTS; ++p)
    if (p < s.n_parts) part[p] = s.q[(((size_t)net * s.n_parts + p) * s.rows + r) * s.out_dim + o];
  const float bias = s.params[(size_t)net * NET_STRIDE + off_b3(s.in_dim, s.out_dim) + o];
  float v = 0.f;
#pragma unroll
  for (int p = 0; p < Q_MAX_PARTS; ++p)
    if (p < s.n_parts) v += part[p];
  return v + bias;
}

// Actor input rows of a staged minibatch.  With preprocessing the minibatch is staged in `in` (Handle::batch_in) and
// its scaled rows are written to `batch` (thread i < B owns half-row 2i, thread B + i half-row 2i + 1); the staged rows
// stay raw, so replaying phase 4 on one upload scales the same rows again.  Without preprocessing `in` == `batch`
// and nothing is written there.
__global__ void k_actor_rows(const float4* in, int B, float4* batch, float4* __restrict__ XA, const Prep prep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * B) return;
  if (i < B) {
    float4 a = in[2 * i];
    if (prep.any()) { a = prep_row0(prep, a); batch[2 * i] = a; }
    XA[i] = make_float4(a.x, a.y, 0.f, 0.f);
  } else {
    float4 b = in[2 * (i - B) + 1];
    if (prep.any()) { b = prep_row1(prep, b); batch[2 * (i - B) + 1] = b; }
    XA[i] = make_float4(b.x, b.y, 0.f, 0.f);
  }
}

// Builds every critic input row of the update from the shared actor outputs.
// thread (b, l): rows j = l, l+64, ... of batch element b; j in [0, 6n+4).
__global__ void __launch_bounds__(256) k_prep(const float4* __restrict__ batch, const QSrc srcS, const QSrc srcN, float* __restrict__ outA,
                       const float* __restrict__ noise, int B, int n, int squash,
                       float4* __restrict__ XAl, float* __restrict__ offAl,
                       float4* __restrict__ XC, float* __restrict__ offC,
                       float4* __restrict__ XT, float4* __restrict__ XP, float4* __restrict__ perb) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */

  __shared__ float sv[4][4];                 // per batch element of this block: mu(s), logstd(s), mu(s'), logstd(s')
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = g >> 6, l = g & 63, bl = threadIdx.x >> 6;
  if (b < B && l < 4) {                      // actor outputs of the s rows (srcS) and the s' rows (srcN), summed ONCE per element
    const float v = q_at(l < 2 ? srcS : srcN, 0, b, l & 1);
    sv[bl][l] = v;
    outA[2 * ((l < 2 ? 0 : B) + b) + (l & 1)] = v;          // k_actor_dout reads these
  }
  __syncthreads();
  if (b >= B) return;
  const float4 r0 = batch[2 * b], r1 = batch[2 * b + 1];
  const float mu_s = sv[bl][0], ls_s = clamp_ls(sv[bl][1]);
  const float mu_n = sv[bl][2], ls_n = clamp_ls(sv[bl][3]);
  const int64_t Bn = (int64_t)B * n;
  const int n3 = 3 * n;
  for (int j = l; j < 2 * n3 + 4; j += 64) {
    if (j < 2 * n3) {
      const int job = j / n3, jj = j % n3, kind = jj / n, i = jj % n;
      const float* nz = noise + B + (int64_t)job * 3 * Bn + (int64_t)kind * Bn + (int64_t)b * n + i;
      float a, off;
      if (kind == 2) {
        a = *nz;
        off = -0.69314718055994531f * CQL_ACT_DIM;  // log(0.5^act_dim)
      } else {
        const Sample s = policy_sample(kind == 0 ? mu_s : mu_n, kind == 0 ? ls_s : ls_n, *nz, squash);
        a = s.a;
        off = s.logp;
      }
      const float4 x = make_float4(r0.x, r0.y, a, 0.f);  // value observation is ALWAYS s
      if (job == 0) { XAl[(int64_t)b * n3 + jj] = x; offAl[(int64_t)b * n3 + jj] = off; }
      else { XC[(int64_t)b * (n3 + 1) + jj] = x; offC[(int64_t)b * (n3 + 1) + jj] = off; }
    } else if (j == 2 * n3) {       // data row (s, a)
      XC[(int64_t)b * (n3 + 1) + n3] = make_float4(r0.x, r0.y, r0.z, 0.f);
      offC[(int64_t)b * (n3 + 1) + n3] = 0.f;
    } else if (j == 2 * n3 + 1) {   // TD target row (s', best_action(s'))
      XT[b] = make_float4(r1.x, r1.y, (float)tanh((double)mu_n), 0.f);
    } else if (j == 2 * n3 + 2) {   // actor-step row (s, a_pi)
      const Sample s = policy_sample(mu_s, ls_s, noise[B + 6 * Bn + b], squash);
      XP[b] = make_float4(r0.x, r0.y, s.a, 0.f);
      perb[b].y = s.logp;
    } else {                        // temperature step: logp - action_size
      const Sample s = policy_sample(mu_s, ls_s, noise[b], squash);
      perb[b].x = s.logp - (float)CQL_ACT_DIM;
    }
  }
}

// ---------------------------------------------------------------- block reductions (fixed order)
template <int NTHREADS>
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  if (warp == 0) {
    t = lane < NTHREADS / 32 ? red[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) red[0] = t;
  }
  __syncthreads();
  t = red[0];
  return t;
}

__device__ __forceinline__ float lse_rows(const float* __restrict__ q, const float* __restrict__ off, int cnt,
                                          float& m_out, float& s_out) {
  float m = -INFINITY;
  for (int j = 0; j < cnt; ++j) m = fmaxf(m, q[j] - off[j]);
  float s = 0.f;
  for (int j = 0; j < cnt; ++j) s += expf(q[j] - off[j] - m);
  m_out = m; s_out = s;
  return m + logf(s);
}

struct LossConsts {
  int B, n, C;
  float gamma, cw, thr, temp_lr, alpha_lr, beta1, beta2, eps;
  int nstep;               // 1: the rows carry their own TD discount in slot 7 (n_steps > 1), else gamma applies
};

// ---- loss glue, split so that nothing heavy runs in a single CTA -------------------------------
// (1) k_lse: one warp per (critic, batch element): logsumexp of the alpha-step rows and of the
//     critic-step rows, unscaled softmax weights (into dQ), TD target / error.   -> pairv[c][b]
// (2) k_scalar_reduce: one CTA sums the C*B pair values in a fixed order -> temp/alpha gradients
//     [data-parallel: the host all-reduces the two scalar gradients here]
// (3) k_scalar_adam: one thread: Adam on log_temp/log_alpha, conservative coefficient, loss metrics
// (4) k_dq: every critic-job row: dQ = coef * softmax (samples) or 2(q-y)/B - coef (data row)
struct PairVals { float lse_a, lse_c, qd, err; };

__device__ __forceinline__ float warp_lse(const float* __restrict__ q, const float* __restrict__ off, int cnt, int lane,
                                          float& m_out, float& v_out) {
  const float v = lane < cnt ? q[lane] - off[lane] : -INFINITY;
  const float m = warp_max(v);
  const float e = lane < cnt ? expf(v - m) : 0.f;
  const float s = warp_sum(e);
  m_out = m;
  v_out = e / s;         // softmax weight of this lane's row
  return m + logf(s);
}

// logsumexp over the lanes' values v (lane < cnt valid); m_out = max, v_out = softmax weight of this lane's value
__device__ __forceinline__ float warp_lse_v(float v, int cnt, int lane, float& m_out, float& v_out) {
  v = lane < cnt ? v : -INFINITY;
  const float m = warp_max(v);
  const float e = lane < cnt ? expf(v - m) : 0.f;
  const float s = warp_sum(e);
  m_out = m;
  v_out = e / s;
  return m + logf(s);
}

// The same over a row of up to 32 * T values (3n + 1 > 32: n_action_samples 11..CQL_MAX_ACTION_SAMPLES), lane l holding
// values l, l + 32, ..., l + 32 (T - 1) (value j < cnt valid).  Fixed order: each lane takes the max of its values, then
// the sum of their exponentials, in t order; warp_max / warp_sum combine the lanes in their fixed butterfly -- the
// same row always gives the same bits.  w_out[t] = softmax weight of value l + 32 t.
template <int T>
__device__ __forceinline__ float warp_lse_strided(const float (&v)[T], int cnt, int lane, float (&w_out)[T]) {
  float m = -INFINITY;
#pragma unroll
  for (int t = 0; t < T; ++t)
    if (lane + 32 * t < cnt) m = fmaxf(m, v[t]);
  m = warp_max(m);
  float e[T], s = 0.f;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    e[t] = lane + 32 * t < cnt ? expf(v[t] - m) : 0.f;
    s += e[t];
  }
  s = warp_sum(s);
#pragma unroll
  for (int t = 0; t < T; ++t) w_out[t] = e[t] / s;
  return m + logf(s);
}
// values per lane in k_lse's wide path: 3n + 1 <= 32 * LSE_STRIDE for every n the API accepts
constexpr int LSE_STRIDE = (3 * CQL_MAX_ACTION_SAMPLES + 1 + 31) / 32;

struct ScalarReduceArgs {
  const float4* perb; const float* scalars; const float* sc_m; const float* sc_v;
  float* g_scalars; float* sums; float* metrics; unsigned int* ticket;
  DpPeer dp;
};
__device__ void scalar_reduce_tail(const PairVals* __restrict__ pairv, const LossConsts& k, const ScalarReduceArgs& a);

// WIDE = false: 3n + 1 <= 32 (n_action_samples <= 10), lane i holds row i, lane 3n the data row.  WIDE = true: up to
// 3 * CQL_MAX_ACTION_SAMPLES + 1 rows, lane l holds rows l, l + 32, ... (warp_lse_strided); the data row is row 3n.
template <bool WIDE>
__global__ void __launch_bounds__(256) k_lse(const float4* __restrict__ batch, const QSrc srcAl,
                                             const float* __restrict__ offAl, const QSrc srcC,
                                             const float* __restrict__ offC, const QSrc srcT, LossConsts k,
                                             float* __restrict__ dQ, PairVals* __restrict__ pairv, const ScalarReduceArgs ra) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */

  const int p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (p < k.C * k.B) {
    const int c = p / k.B, b = p % k.B;
    const int n3 = 3 * k.n, rsC = n3 + 1;
    PairVals pv;
    float qd;
    if constexpr (!WIDE) {
      float m, w;
      const float va = lane < n3 ? q_at(srcAl, c, b * n3 + lane) - offAl[(int64_t)b * n3 + lane] : 0.f;
      pv.lse_a = warp_lse_v(va, n3, lane, m, w);
      const float qc = lane < rsC ? q_at(srcC, c, b * rsC + lane) : 0.f;       // lane n3 = the data row (s, a)
      const float vc = lane < n3 ? qc - offC[(int64_t)b * rsC + lane] : 0.f;
      pv.lse_c = warp_lse_v(vc, n3, lane, m, w);
      if (lane < n3) dQ[((int64_t)c * k.B + b) * rsC + lane] = w;
      qd = __shfl_sync(0xffffffffu, qc, n3 & 31);
    } else {
      float va[LSE_STRIDE], qc[LSE_STRIDE], vc[LSE_STRIDE], w[LSE_STRIDE];
#pragma unroll
      for (int t = 0; t < LSE_STRIDE; ++t) {
        const int j = lane + 32 * t;
        va[t] = j < n3 ? q_at(srcAl, c, b * n3 + j) - offAl[(int64_t)b * n3 + j] : 0.f;
        qc[t] = j < rsC ? q_at(srcC, c, b * rsC + j) : 0.f;
        vc[t] = j < n3 ? qc[t] - offC[(int64_t)b * rsC + j] : 0.f;
      }
      pv.lse_a = warp_lse_strided(va, n3, lane, w);
      pv.lse_c = warp_lse_strided(vc, n3, lane, w);
#pragma unroll
      for (int t = 0; t < LSE_STRIDE; ++t)
        if (lane + 32 * t < n3) dQ[((int64_t)c * k.B + b) * rsC + lane + 32 * t] = w[t];
      float qdt = qc[0];                        // the data row: row n3 = lane n3 % 32 of stride n3 / 32
#pragma unroll
      for (int t = 1; t < LSE_STRIDE; ++t)
        if (t == n3 / 32) qdt = qc[t];
      qd = __shfl_sync(0xffffffffu, qdt, n3 & 31);
    }
    if (lane == 0) {
      float qt = q_at(srcT, 0, b);
      for (int c2 = 1; c2 < k.C; ++c2) qt = fminf(qt, q_at(srcT, c2, b));
      const float4 r0 = batch[2 * b], r1 = batch[2 * b + 1];
      const float disc = k.nstep ? r1.w : k.gamma;
      const float y = r0.w + disc * qt * (1.f - r1.z);
      pv.qd = qd;
      pv.err = pv.qd - y;
      pairv[p] = pv;
    }
  }
  // The block that finishes LAST sums the pair values (what the one-CTA k_scalar_reduce launch did: one launch boundary
  // less on the critical path, 3.4 us per update by the r02 skip test) -- in exactly that kernel's order.
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ra.ticket, 1u);
    last = t == gridDim.x - 1;
    if (last) *ra.ticket = 0;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  scalar_reduce_tail(pairv, k, ra);
}

// sums[0]=sum td err^2  [1]=sum lse_c  [2]=sum qd.  Runs in ONE block of 256 threads; every thread stands for four
// threads t, t + 256, t + 512, t + 768 of the former 1024-thread launch and the partial sums are combined in that launch's
// order (lanes, then the 32 warp sums), so the results are bit-identical to it.
__device__ __forceinline__ float block_sum_as_1024(const float (&v)[4], float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float w = warp_sum(v[j]);
    if (lane == 0) red[warp + 8 * j] = w;
  }
  __syncthreads();
  float t = 0.f;
  if (warp == 0) {
    t = warp_sum(red[lane]);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}
__device__ void scalar_reduce_tail(const PairVals* __restrict__ pairv, const LossConsts& k, const ScalarReduceArgs& a) {
  __shared__ float red[33];
  float st[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j)
    for (int b = threadIdx.x + 256 * j; b < k.B; b += 1024) st[j] += a.perb[b].x;
  const float s_t = block_sum_as_1024(st, red);
  float sa[4] = {0.f, 0.f, 0.f, 0.f}, sc[4] = {0.f, 0.f, 0.f, 0.f}, sd[4] = {0.f, 0.f, 0.f, 0.f}, se[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j)
    for (int p = threadIdx.x + 256 * j; p < k.C * k.B; p += 1024) {
      const PairVals pv = pairv[p];
      sa[j] += pv.lse_a; sc[j] += pv.lse_c; sd[j] += pv.qd; se[j] += pv.err * pv.err;
    }
  const float s_a = block_sum_as_1024(sa, red);
  const float s_c = block_sum_as_1024(sc, red);
  const float s_d = block_sum_as_1024(sd, red);
  const float s_e = block_sum_as_1024(se, red);
  if (threadIdx.x == 0) {
    const float lt = a.scalars[0], la = a.scalars[1];
    const float temp_loss = -expf(lt) * (s_t / (float)k.B);
    const float inv = 1.f / ((float)k.C * (float)k.B);
    const float raw = s_a * inv - s_d * inv;
    const float e = expf(la), clipped = fminf(fmaxf(e, 0.f), 1e6f);
    const float alpha_loss = -clipped * (k.cw * raw - k.thr);
    a.g_scalars[0] = temp_loss;                 // d/d log_temp of -exp(lt)*mean = the loss itself
    a.g_scalars[1] = e <= 1e6f ? alpha_loss : 0.f;
    a.metrics[0] = temp_loss;
    a.metrics[2] = alpha_loss;
    a.sums[0] = s_e; a.sums[1] = s_c; a.sums[2] = s_d;
    // snapshot for k_scalar_adam_dq (every block of which recomputes the scalar Adam steps from these)
    a.sums[8] = lt; a.sums[9] = la;
    a.sums[10] = a.sc_m[0]; a.sums[11] = a.sc_v[0]; a.sums[12] = a.sc_m[1]; a.sums[13] = a.sc_v[1];
    // fused data-parallel exchange: the two scalar gradients travel inside the signal words (group 0)
    if (a.dp.world > 1) dp_signal_scalars(a.dp, temp_loss, e <= 1e6f ? alpha_loss : 0.f);
  }
}

__device__ __forceinline__ float adam_scalar(float p, float g, float& m, float& v, float lr, const LossConsts& k,
                                             const StepInfo& si) {
  m = m + (g - m) * (1.f - k.beta1);
  v = v * k.beta2 + (1.f - k.beta2) * g * g;
  const float denom = sqrtf(v) / (float)si.bc2_sqrt + k.eps;
  return p - (float)((double)lr / si.bc1) * (m / denom);
}

// Adam on log_temp / log_alpha, conservative coefficient, loss metrics -- and, in the same launch, dQ of every
// critic-job row: coef * softmax (samples) or 2 (q - y) / B - coef (data row).  Every thread recomputes the two scalar
// Adam steps (a few dozen flops, bit-identical everywhere) from the SNAPSHOT of (log_temp, log_alpha, their moments)
// that k_scalar_reduce left in sums[8..13]; thread 0 of block 0 stores the results into the live locations, which no
// other thread of this launch reads.
__global__ void __launch_bounds__(256) k_scalar_adam_dq(float* __restrict__ scalars, float* __restrict__ sc_m, float* __restrict__ sc_v,
                                 const float* __restrict__ g_scalars, const StepInfo* __restrict__ si, LossConsts k,
                                 float* __restrict__ sums, float* __restrict__ metrics, const PairVals* __restrict__ pairv,
                                 float* __restrict__ dQ, const DpPeer dp, long long dp_off) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */

  float lt = sums[8], la = sums[9];
  float mt = sums[10], vt = sums[11], ma = sums[12], va = sums[13];
  float g_t = g_scalars[0], g_a = g_scalars[1];
  if (dp.world > 1) {                // fused data-parallel exchange: mean of the ranks' scalar gradients (group 0)
    __shared__ float gsh[2];
    if (threadIdx.x == 0) dp_wait_scalars(dp, g_t, g_a, gsh[0], gsh[1]);      // polls this rank's own signal pad
    __syncthreads();
    g_t = gsh[0];
    g_a = gsh[1];
  }
  if (k.temp_lr > 0.f) lt = adam_scalar(lt, g_t, mt, vt, k.temp_lr, k, *si);
  if (k.alpha_lr > 0.f) la = adam_scalar(la, g_a, ma, va, k.alpha_lr, k, *si);
  const float alpha = fminf(fmaxf(expf(la), 0.f), 1e6f);
  const float inv = 1.f / ((float)k.C * (float)k.B);
  const float coef = alpha * k.cw * inv;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int rsC = 3 * k.n + 1;
  if (i < (int64_t)k.C * k.B * rsC) {
    const int j = (int)(i % rsC);
    dQ[i] = j < rsC - 1 ? coef * dQ[i] : 2.f * pairv[i / rsC].err / (float)k.B - coef;
  }
  if (i == 0) {
    if (k.temp_lr > 0.f) { scalars[0] = lt; sc_m[0] = mt; sc_v[0] = vt; }
    if (k.alpha_lr > 0.f) { scalars[1] = la; sc_m[1] = ma; sc_v[1] = va; }
    sums[3] = coef;
    metrics[1] = expf(lt);
    metrics[3] = expf(la);
    const float td = sums[0] / (float)k.B;
    const float cons = alpha * (k.cw * (sums[1] * inv - sums[2] * inv) - k.thr);
    metrics[4] = td + cons;
    metrics[6] = td;
  }
  if (dp.world > 1) dp_consume_done(dp, 0, gridDim.x);
}

// actor loss + d/dQ through the min over critics (one CTA)
__global__ void __launch_bounds__(1024) k_actor_dq(const QSrc srcP, const float4* __restrict__ perb,
                                                   const float* __restrict__ scalars, int B, int C,
                                                   float* __restrict__ dQP, float* __restrict__ metrics) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
 
  __shared__ float red[32];
  const float T = expf(scalars[0]);
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += 1024) {
    int arg = 0;
    float qm = q_at(srcP, 0, b);
    for (int c = 1; c < C; ++c) {
      const float q = q_at(srcP, c, b);
      if (q < qm) { qm = q; arg = c; }
    }
    for (int c = 0; c < C; ++c) dQP[(int64_t)c * B + b] = c == arg ? -1.f / (float)B : 0.f;
    s += T * perb[b].y - qm;
  }
  s = block_sum<1024>(s, red);
  if (threadIdx.x == 0) metrics[5] = s / (float)B;
}

// d actor_loss / d (mu, raw logstd): mirrors autograd through rsample, tanh, log-prob, clamp.
// With srcP.q set (f16x3 path, where the dx-only bwd1 takes dQ itself) it also produces the actor-loss metric that the
// one-CTA k_actor_dq launch used to: warp sums into part[], the block that finishes last adds them in that launch's order.
__global__ void k_actor_dout(const float* __restrict__ outA, const float* __restrict__ noise_actor,
                             const float4* __restrict__ dXP, const float* __restrict__ scalars, int B, int n_parts,
                             int squash, float* __restrict__ dOutA, const QSrc srcP, const float4* __restrict__ perb,
                             int C, float* __restrict__ part, unsigned int* __restrict__ ticket, float* __restrict__ metrics) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
 
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (srcP.q != nullptr) {
    float v = 0.f;
    if (b < B) {
      float qm = q_at(srcP, 0, b);
      for (int c = 1; c < C; ++c) qm = fminf(qm, q_at(srcP, c, b));
      v = expf(scalars[0]) * perb[b].y - qm;
    }
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) part[b >> 5] = v;
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int t = atomicAdd(ticket, 1u);
      last = t == gridDim.x - 1;
      if (last) *ticket = 0;
    }
    __syncthreads();
    if (last && threadIdx.x < 32) {
      __threadfence();
      const int n_w = (gridDim.x * blockDim.x) >> 5;
      float s = 0.f;
      for (int i = threadIdx.x; i < n_w; i += 32) s += part[i];
      s = warp_sum(s);
      if (threadIdx.x == 0) metrics[5] = s / (float)B;
    }
  }
  if (b >= B) return;
  float da = 0.f;
  for (int c = 0; c < n_parts; ++c) da += dXP[(int64_t)c * B + b].z;   // parts = critics (x column slices)
  const float mu = outA[2 * b], ls_raw = outA[2 * b + 1], ls = clamp_ls(ls_raw);
  const float eps = noise_actor[b];
  const Sample s = policy_sample(mu, ls, eps, squash);
  const float w = __fdiv_rn(expf(scalars[0]), (float)B);   // d loss / d logp
  // Every product and sum below is rounded separately (no FMA contraction), in autograd's order.  With raw indices
  // as observations the policy saturates: a = +-1 exactly, 1 - a^2 = 0, and the reference's gradient through the mean
  // head is EXACTLY zero because -dt/std and +dt/std cancel bit for bit.  A contracted fma(w, t/std, g_raw) leaves the
  // product's rounding residue (~1e-7 of the batch gradient) instead, which the first Adam steps normalise to full
  // +-lr moves on weights whose true gradient is zero.
  const float one_m_a2 = __fsub_rn(1.f, __fmul_rn(s.a, s.a));
  const float dt_std = __fmul_rn(w, __fdiv_rn(s.t, s.std_));     // -(d loss / d t) / std = w t / std
  float g_tanh;                                                  // d loss / d raw through the squashing terms
  if (squash == CQL_SQUASH_EPS) {
    const float g_a = __fadd_rn(da, __fmul_rn(w, __fdiv_rn(__fmul_rn(2.f, s.a), __fadd_rn(one_m_a2, 1e-6f))));
    g_tanh = __fmul_rn(g_a, one_m_a2);
  } else {
    const float sig = __fdiv_rn(1.f, __fadd_rn(1.f, expf(__fmul_rn(2.f, s.raw))));  // sigmoid(-2 raw)
    g_tanh = __fadd_rn(__fmul_rn(w, __fsub_rn(2.f, __fmul_rn(4.f, sig))), __fmul_rn(da, one_m_a2));
  }
  const float g_raw = __fadd_rn(g_tanh, -dt_std);                // tanh branch + (raw - mu) / std branch
  const float g_mu = __fadd_rn(g_raw, dt_std);                   // raw = mu + std eps  and  -(raw - mu) / std
  const float g_std = __fadd_rn(__fmul_rn(g_raw, eps), __fmul_rn(w, __fdiv_rn(__fmul_rn(s.t, s.t), s.std_)));
  const float g_ls = __fsub_rn(__fmul_rn(g_std, s.std_), w);
  dOutA[2 * b] = g_mu;
  dOutA[2 * b + 1] = (ls_raw >= -20.f && ls_raw <= 2.f) ? g_ls : 0.f;
}

// ---------------------------------------------------------------- gradient reduction, Adam, Polyak
// grads[net][idx] = sum of the per-tile "small" partials / per-split dW2 partials, in fixed order.
__global__ void k_reduce_grads(const float* __restrict__ small, const float* __restrict__ pw2, int in_dim, int out_dim,
                               int tiles, int splits, float* __restrict__ grads) {
  const int net = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= NET_STRIDE) return;
  const int w2_lo = off_W2(in_dim), w2_hi = w2_lo + H * H, total = net_floats(in_dim, out_dim);
  float s = 0.f;
  if (idx >= w2_lo && idx < w2_hi) {
    const float* p = pw2 + (size_t)net * splits * H * H + (idx - w2_lo);
    for (int i = 0; i < splits; ++i) s += p[(size_t)i * H * H];
  } else if (idx < total) {
    const int sidx = idx < w2_lo ? idx : idx - H * H;
    const float* p = small + (size_t)net * tiles * SMALL_STRIDE + sidx;
    for (int i = 0; i < tiles; ++i) s += p[(size_t)i * SMALL_STRIDE];
  }
  grads[(size_t)net * NET_STRIDE + idx] = s;
}

// torch.optim.Adam (defaults) fused with the Polyak update of the target copy.
__global__ void k_adam_polyak(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v,
                              const float* __restrict__ g, float* __restrict__ targ, int64_t count, float lr,
                              float beta1, float beta2, float eps, float tau, const StepInfo* __restrict__ si) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
 
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float step_size = (float)((double)lr / si->bc1);
  const float bc2s = (float)si->bc2_sqrt;
  const float gi = g[i];
  const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
  const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float pn = p[i] - step_size * (mi / (sqrtf(vi) / bc2s + eps));
  p[i] = pn;
  if (targ) targ[i] = targ[i] * (1.f - tau) + tau * pn;
}

// ---------------------------------------------------------------- launches
// How a kernel is launched.  pdl: with programmatic dependent launch -- the kernel may start (barrier init, TMEM
// allocation) while its predecessor in the stream drains; it executes `griddepcontrol.wait` before touching anything the
// predecessor wrote, and only kernels that contain that wait are launched this way.  skip: the CQL_SKIP bit that leaves
// the launch out (timing experiments only: results wrong).
struct LaunchMode { bool pdl; int skip; };
constexpr LaunchMode PLAIN{false, 0}, PDL{true, 0};
constexpr LaunchMode pdl_skip(int bit) { return LaunchMode{true, bit}; }

// Every launch of the update goes through here: counted in Handle::launches and error-checked.  PDL is off under
// CQL_NO_PDL=1 and while Handle::pdl_off is set (cql_timed_update: with PDL a kernel's prologue starts under its
// predecessor, so a CUDA event recorded between two kernels no longer separates their durations -- r01: bwd1 0.118 ms /
// bwd2 0.003 ms).
template <typename... KArgs, typename... Args>
inline void launch(Handle* h, cudaStream_t st, LaunchMode mode, void (*kernel)(KArgs...), dim3 grid, dim3 block,
                   size_t smem, Args&&... args) {
  if (switches().skip & mode.skip) return;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = mode.pdl && !switches().no_pdl && !h->pdl_off ? 1 : 0;
  CQL_CUDA(cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...));
  CQL_LAUNCH_CHECK(h);
}

// ---------------------------------------------------------------- precision
// cfg.precision as a compile-time parameter of the schedule; with_precision is the one place that maps the one to the other
enum class Prec { FP32, TF32X3, BF16, F16X3 };
template <typename F>
inline void with_precision(const Handle* h, F&& f) {
  switch (h->cfg.precision) {
    case CQL_PREC_FP32: f(std::integral_constant<Prec, Prec::FP32>{}); break;
    case CQL_PREC_TF32X3: f(std::integral_constant<Prec, Prec::TF32X3>{}); break;
    case CQL_PREC_BF16: f(std::integral_constant<Prec, Prec::BF16>{}); break;
    case CQL_PREC_F16X3: f(std::integral_constant<Prec, Prec::F16X3>{}); break;
    default: throw Error{"internal: bad precision"};
  }
}
// the tensor-core kernel configuration of a precision (f16x3: fp16 hi/lo split; tf32x3 and bf16: mlp_tc.cuh)
template <Prec P>
using TcCfg = std::conditional_t<P == Prec::F16X3, tc::HCfg, tc::Cfg<P != Prec::BF16>>;

// The critic forward over a job list (fp32: CUDA cores; else tensor cores, W2 from the packed copy).  src[i] tells the
// consumer kernels where job i's outputs are (see QSrc): f16x3 leaves the layer-3 partial sums to them (q_at); tf32x3
// and bf16 sum the partials in one more launch.  `part` / `part_floats`: scratch for those partials other than the
// update's own (Handle::part), for a caller whose row counts are not the update's (cql_offline_eval).
template <Prec P, int IN, int OUT>
inline void launch_fwd(Handle* h, FwdJobs& jobs, cudaStream_t st, QSrc* src, float* part = nullptr, size_t part_floats = 0) {
  if constexpr (P == Prec::FP32) {
    int t = 0;
    for (int i = 0; i < jobs.n; ++i) {
      jobs.j[i].tile_begin = t;
      t += tiles_of(jobs.j[i].rows) * jobs.j[i].n_nets;
    }
    jobs.total_tiles = t;
    if (t > 0) launch(h, st, PLAIN, mlp_fwd_kernel<IN, OUT>, dim3(t), dim3(NT), FWD_SMEM, jobs);
    for (int i = 0; i < jobs.n; ++i) src[i] = QSrc{jobs.j[i].out, jobs.j[i].params, 0, jobs.j[i].rows, IN, OUT};
  } else {
    constexpr bool F16X3 = P == Prec::F16X3;
    const Switches& sw = switches();
    tc::TcFwdJobs tj{};
    tj.n = jobs.n;
    // big launches of the f16x3 path run on CTA pairs (one H1 tile feeds all 256 output columns).  Critics only: the
    // actor has no CTA-pair operand copy (pack_slots, adam_pack), so its forward stays on one-CTA kernels at any batch
    // size, as its backward does in launch_bwd.
    int pair_items = 0, items128 = 0;
    for (int i = 0; i < jobs.n; ++i) {
      pair_items += jobs.j[i].n_nets * ((jobs.j[i].rows + 2 * tc::TM - 1) / (2 * tc::TM));
      items128 += jobs.j[i].n_nets * tc::HCfg::SLICES * ((jobs.j[i].rows + tc::TM - 1) / tc::TM);
    }
    const bool pair = F16X3 && !sw.no_pair && IN == 3 && pair_items >= h->num_sms / 2;
    // small launches (the B-row passes of the actor step: 16-32 work items of 128 columns) run on 32-column work items
    // instead -- four times as many CTAs, a quarter of the operand load each
    const bool small = F16X3 && !pair && !sw.no_small && items128 * 2 <= h->num_sms;
    const int n_slices = small ? tc::HCfgS::SLICES : TcCfg<P>::SLICES;
    const int n_parts = pair ? tc::H2Cfg::PARTS : n_slices;       // layer-3 partial sums per row
    size_t part_off = 0;
    int items = 0;
    float* part_of[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int i = 0; i < jobs.n; ++i) {
      const FwdJob& j = jobs.j[i];
      const int slot = (int)((j.params - h->params) / NET_STRIDE);
      tj.item_begin[i] = items;
      items += j.n_nets * n_slices * ((j.rows + tc::TM - 1) / tc::TM);
      part_of[i] = (part ? part : h->part) + part_off;
      part_off += (size_t)j.n_nets * n_parts * j.rows * OUT;
      tj.j[i] = tc::TcFwdJob{j.X, j.params,
                             pair ? h->packed_fwd2 + (size_t)slot * h->packed_net_bytes2 : h->packed_fwd + (size_t)slot * h->packed_net_bytes,
                             part_of[i], j.h2, j.rows, j.n_nets};
    }
    tj.item_begin[jobs.n] = items;
    tj.h2_cost = sw.h2_cost;
    CQL_REQUIRE(part_off <= (part ? part_floats : h->part_floats), "internal: partial-sum scratch too small");
    if (items == 0) return;
    const int grid = items < h->num_sms ? items : h->num_sms;
    if constexpr (F16X3) {
      if (pair)
        launch(h, st, PDL, tc::tc_fwd_h2_kernel<IN, OUT>, dim3(2 * (h->num_sms / 2)), dim3(tc::H2Cfg::THREADS),
               tc::H2Cfg::SMEM_BYTES, tj, h->pair_swap_b);
      else if (small)
        launch(h, st, PDL, tc::tc_fwd_h_kernel<IN, OUT, tc::HCfgS>, dim3(grid), dim3(tc::HCfgS::THREADS), tc::HCfgS::SMEM_BYTES, tj);
      else
        launch(h, st, PDL, tc::tc_fwd_h_kernel<IN, OUT>, dim3(grid), dim3(tc::HCfg::THREADS), tc::HCfg::SMEM_BYTES, tj);
      for (int i = 0; i < jobs.n; ++i) src[i] = QSrc{part_of[i], jobs.j[i].params, n_parts, jobs.j[i].rows, IN, OUT};
    } else {
      if constexpr (P == Prec::TF32X3)
        launch(h, st, PLAIN, tc::tc_fwd_ts_kernel<IN, OUT>, dim3(grid), dim3(tc::TsCfg::THREADS), tc::TsCfg::SMEM_BYTES, tj);
      else
        launch(h, st, PLAIN, tc::tc_fwd_kernel<false, IN, OUT>, dim3(grid), dim3(tc::Pipe<false, tc::FWD_NPW>::THREADS),
               tc::FwdSmem<false, tc::FWD_NPW>::BYTES, tj);
      tc::SumJobs sj{};
      sj.n = jobs.n;
      int max_n = 0;
      for (int i = 0; i < jobs.n; ++i) {
        const FwdJob& j = jobs.j[i];
        sj.j[i] = {part_of[i], j.params, j.out, j.rows, j.n_nets};
        max_n = std::max(max_n, j.n_nets * j.rows * OUT);
        src[i] = QSrc{j.out, j.params, 0, j.rows, IN, OUT};
      }
      launch(h, st, PDL, tc::k_sum_partials_multi<IN, OUT>, dim3((max_n + 255) / 256, jobs.n), dim3(256), 0, sj, n_parts);
    }
  }
}

// refresh the packed (tensor-core operand layout) copies of W2 -- forward orientation for every listed slot,
// plus W2^T for the trainable ones (slot <= C) -- in ONE launch (f16x3: one more for the critics' CTA-pair layout)
template <Prec P>
inline void pack_slots(Handle* h, const int* slots, int n_slots, cudaStream_t st) {
  if (P == Prec::FP32 || n_slots == 0) return;
  tc::PackJobs jobs{};
  for (int i = 0; i < n_slots; ++i) {
    const int slot = slots[i];
    const bool is_actor = slot == slot_actor() || slot == slot_targ_actor(h->C);
    const int in_dim = is_actor ? 2 : 3;
    jobs.j[jobs.n++] = {h->net_params(slot), h->packed_fwd + (size_t)slot * h->packed_net_bytes, in_dim, 0};
    if (slot <= h->C) jobs.j[jobs.n++] = {h->net_params(slot), h->packed_bwd + (size_t)slot * h->packed_net_bytes_bwd, in_dim, 1};
  }
  if constexpr (P == Prec::F16X3) {    // the fp16 hi|lo layout
    launch(h, st, PDL, tc::k_pack_multi_h, dim3(H * 32 / 256, jobs.n), dim3(256), 0, jobs, 2);
    tc::PackJobs jp{};                // the same operands in the CTA-pair layout
    for (int i = 0; i < n_slots; ++i) {
      const int slot = slots[i];
      const bool is_actor = slot == slot_actor() || slot == slot_targ_actor(h->C);
      if (is_actor) continue;         // the actor's launches are small: one-CTA kernels only
      jp.j[jp.n++] = {h->net_params(slot), h->packed_fwd2 + (size_t)slot * h->packed_net_bytes2, 3, 0};
      if (slot <= h->C) jp.j[jp.n++] = {h->net_params(slot), h->packed_bwd2 + (size_t)slot * h->packed_net_bytes2, 3, 1};
    }
    if (jp.n) launch(h, st, PDL, tc::k_pack_pair_h, dim3(H * 32 / 256, jp.n), dim3(256), 0, jp, 2);
  } else {
    constexpr bool TF32 = P == Prec::TF32X3;
    const int chunks = H * (H / tc::Cfg<TF32>::EPC);
    launch(h, st, PLAIN, tc::k_pack_multi<TF32>, dim3((chunks + 255) / 256, jobs.n), dim3(256), 0, jobs);
  }
}
template <Prec P>
inline void pack_weights(Handle* h, int slot, int n_slots, cudaStream_t st) {
  int slots[CQL_MAX_CRITICS];
  for (int i = 0; i < n_slots; ++i) slots[i] = slot + i;
  pack_slots<P>(h, slots, n_slots, st);
}

template <Prec P>
inline void pack_all_weights(Handle* h, cudaStream_t st) {
  if constexpr (P == Prec::F16X3)
    launch(h, st, PLAIN, tc::k_w2max_init, dim3(2 + 2 * h->C), dim3(256), 0, h->params, 2 + 2 * h->C, h->w2max);
  pack_weights<P>(h, slot_actor(), 1, st);
  pack_weights<P>(h, slot_critic(0), h->C, st);
  pack_weights<P>(h, slot_targ_actor(h->C), 1, st);
  pack_weights<P>(h, slot_targ_critic(h->C, 0), h->C, st);
}

// f16x3 at world size 1: k_adam_pack sums the backward's gradient partials itself and the weight-gradient bwd1 kernels
// zero their own partial slots -- no k_reduce_grads_tc launch and no memset node per gradient group, so every edge of
// the backward chain is a programmatic one.  Data-parallel runs keep the separate reduction: it is where their gradient
// exchange starts (phase A of dp_peer.cuh, or the exchange between cql_step_phase calls).
template <Prec P>
inline bool fold_grads(const Handle* h) {
  const Switches& sw = switches();
  return P == Prec::F16X3 && !sw.no_fold && !sw.no_fused_adam && h->cfg.world_size <= 1 && h->dp.world <= 1;
}

// The backward jobs of an update.  The critic and actor jobs are built in one phase and their gradients consumed by the
// optimizer step of the next, which re-derives the job's BwdPlan from the same job.
inline BwdJob critic_bwd_job(Handle* h) {
  return BwdJob{h->XC, h->dQ, h->h2C, h->net_params(slot_critic(0)), h->smallC, nullptr, h->pw2C, h->B * (3 * h->n + 1),
                h->C, h->splitsC};
}
inline BwdJob actor_bwd_job(Handle* h) {
  return BwdJob{h->XA, h->dOutA, h->h2A, h->net_params(slot_actor()), h->smallA, nullptr, h->pw2A, h->B, 1, h->splitsA};
}

// Launch geometry of one backward job and the partial counts its consumers sum: k_reduce_grads_tc or k_adam_pack
// (slots1 bwd1 partials, splits bwd2 partials per net) and k_actor_dout (dx_parts partials of dx).  A function of the
// job and the handle alone.
struct BwdPlan {
  bool pair = false, small = false, pair2 = false, fork = false, fold = false;
  int clusters1 = 0, grid1 = 0, slots1 = 0, splits = 0;
  const float4* dx = nullptr;
  int dx_parts = 0;
};
template <Prec P, int IN, int OUT, bool WGRADS, bool DX>
inline BwdPlan bwd_plan(const Handle* h, const BwdJob& jb) {
  BwdPlan p{};
  if constexpr (P == Prec::FP32) {
    p.splits = jb.splits;
    p.dx = jb.dX;
    p.dx_parts = jb.n_nets;            // parts = critics (x column slices)
  } else {
    constexpr bool F16X3 = P == Prec::F16X3;
    const Switches& sw = switches();
    const int tiles = (jb.rows + tc::TM - 1) / tc::TM;
    const int items = jb.n_nets * TcCfg<P>::SLICES * tiles;
    // big launches of the f16x3 path run on CTA pairs (mlp_tc_h2.cuh): one dZ2 tile feeds all 256 columns of dH1
    p.pair = F16X3 && !sw.no_pair && !sw.no_pair_bwd1 && IN == 3 &&
             jb.n_nets * ((jb.rows + 2 * tc::TM - 1) / (2 * tc::TM)) >= h->num_sms / 2;
    p.small = F16X3 && !p.pair && !sw.no_small && items * 2 <= h->num_sms;
    const int n_slices = p.small ? tc::HCfgS::SLICES : TcCfg<P>::SLICES;
    const int items_s = jb.n_nets * n_slices * tiles;
    // The big launch's bwd1 and bwd2 are independent too and run SIDE BY SIDE: bwd1 on 30 of the 74 CTA pairs, bwd2 on
    // the other 44 (22 splits per critic).  Back to back on all SMs each, the fixed cost of either kernel -- prologue,
    // accumulator dump (half as many dW2 partials now), tail -- was serial: with the main loop skipped bwd2 still took
    // 16 of its 44 us.  Measured sweep of the bwd1 share (pairs -> us per update): 74 (serial) 222.4, 46 238, 42 229,
    // 38 222.5, 34 216.5, 32 213.1, 30 212.7, 28 212.9, 26 219, 22 230.  CQL_BIG_FORK=<pairs> overrides (0 = serial).
    const bool may_fork = WGRADS && !sw.no_fork && !h->timing && h->side_stream != nullptr;
    const int fork_pairs = sw.big_fork >= 0 ? sw.big_fork : (h->num_sms / 2) * 30 / 74;
    p.clusters1 = (p.pair && may_fork && fork_pairs > 0 && fork_pairs < h->num_sms / 2) ? fork_pairs : h->num_sms / 2;
    p.grid1 = p.pair ? 2 * p.clusters1 : (items_s < h->num_sms ? items_s : h->num_sms);
    p.slots1 = (F16X3 ? 2 : 4) * p.grid1;      // f16x3: one slot per (CTA, epilogue group)
    p.dx = h->dX_part;
    p.dx_parts = jb.n_nets * (p.pair ? (int)tc::H2Cfg::PARTS : n_slices);
    p.fold = WGRADS && fold_grads<P>(h);
    // bwd1 and bwd2 of one job are independent (both only read X, dOut, H2).  For the small jobs (the actor's B rows:
    // a few dozen CTAs each) they run side by side on a forked branch -- the fork/join is captured into the step graph.
    constexpr int RS2 = F16X3 ? tc::B2HCfg::RS : tc::B2Cfg<P != Prec::BF16>::RS;
    const int n_stage = (jb.rows + RS2 - 1) / RS2;
    int splits = h->num_sms / jb.n_nets;
    if (splits > n_stage) splits = n_stage;      // (fewer, longer splits for the small jobs were measured: slower)
    if (splits > h->splits_tc) splits = h->splits_tc;
    if (splits < 1) splits = 1;
    if constexpr (F16X3) {                       // dW2 on CTA pairs (A operand in tensor memory): the big launches
      p.pair2 = !sw.no_pair && !sw.no_pair_bwd2 && (p.pair || !sw.no_pair_bwd2_small);   // also the small (actor)
      if (p.pair2) splits = std::max(1, std::min(n_stage, (h->num_sms / 2) / jb.n_nets));   // launch: a pair CTA dumps
      if (p.pair2 && p.pair && p.clusters1 < h->num_sms / 2)                                // half an accumulator
        splits = std::max(1, (h->num_sms / 2 - p.clusters1) / jb.n_nets);
    }
    p.splits = splits;
    p.fork = may_fork && p.grid1 + (p.pair2 ? 2 : 1) * splits * jb.n_nets <= h->num_sms;
  }
  return p;
}

// event marks of cql_timed_update inside a backward job (-1: none): mid after bwd1, end after bwd2, done after the job
// (fp32 records `done` ahead of its reduction launch, so the actor-backward duration leaves that launch out there)
struct BwdMarks { int mid = -1, end = -1, done = -1; };

// The backward of one job: bwd1 (dH1, dW1, db1, dx), with WGRADS bwd2 (dW2, db2, dW3, db3) and the reduction of their
// partials into grads_out -- unless k_adam_pack sums them (plan.fold).
template <Prec P, int IN, int OUT, bool WGRADS, bool DX>
inline BwdPlan launch_bwd(Handle* h, const BwdJob& jb, float* grads_out, cudaStream_t st, BwdMarks mk = {}) {
  auto mark_at = [&](int i) { if (i >= 0) mark(h, st, i); };
  const BwdPlan p = bwd_plan<P, IN, OUT, WGRADS, DX>(h, jb);
  if constexpr (P == Prec::FP32) {
    launch(h, st, PLAIN, mlp_bwd1_kernel<IN, OUT, WGRADS, DX>, dim3(tiles_of(jb.rows) * jb.n_nets), dim3(NT), BWD1_SMEM, jb);
    mark_at(mk.mid);
    if (!WGRADS) return p;
    launch(h, st, PLAIN, mlp_bwd2_kernel<IN, OUT>, dim3(4, jb.splits, jb.n_nets), dim3(NT), BWD2_SMEM, jb);
    mark_at(mk.end);
    mark_at(mk.done);
    launch(h, st, PLAIN, k_reduce_grads, dim3((NET_STRIDE + 255) / 256, jb.n_nets), dim3(256), 0, jb.small, jb.pw2, IN, OUT,
           tiles_of(jb.rows), jb.splits, grads_out);
  } else {
    constexpr bool F16X3 = P == Prec::F16X3;
    const int slot = (int)((jb.params - h->params) / NET_STRIDE);
    if (WGRADS && !p.fold) CQL_CUDA(cudaMemsetAsync(h->small1, 0, (size_t)jb.n_nets * p.slots1 * SMALL_STRIDE * sizeof(float), st));
    tc::Bwd1Job j1{jb.X, jb.dOut, jb.h2, jb.params,
                   p.pair ? h->packed_bwd2 + (size_t)slot * h->packed_net_bytes2 : h->packed_bwd + (size_t)slot * h->packed_net_bytes_bwd,
                   h->small1, DX ? h->dX_part : nullptr, jb.rows, jb.n_nets, p.slots1};
    j1.q_part = jb.q_part; j1.q_parts = jb.q_parts; j1.dq_scale = jb.dq_scale;
    j1.zero_small1 = p.fold ? 1 : 0;
    cudaStream_t st2 = st;
    if (p.fork) {
      CQL_CUDA(cudaEventRecord(h->ev_fork, st));
      CQL_CUDA(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
      st2 = h->side_stream;
    }
    if constexpr (F16X3) {
      if (p.pair)
        launch(h, st, PDL, tc::tc_bwd1_h2_kernel<IN, OUT, WGRADS, DX>, dim3(2 * p.clusters1), dim3(tc::H2Cfg::THREADS),
               tc::H2B1Cfg::SMEM_BYTES, j1, h->pair_swap_b);
      else if (p.small)
        launch(h, st, PDL, tc::tc_bwd1_h_kernel<IN, OUT, WGRADS, DX, tc::HCfgS>, dim3(p.grid1), dim3(tc::HCfgS::THREADS),
               tc::HCfgS::SMEM_BYTES, j1);
      else
        launch(h, st, PDL, tc::tc_bwd1_h_kernel<IN, OUT, WGRADS, DX>, dim3(p.grid1), dim3(tc::HCfg::THREADS), tc::HCfg::SMEM_BYTES, j1);
    } else if constexpr (P == Prec::TF32X3) {
      launch(h, st, PLAIN, tc::tc_bwd1_ts_kernel<IN, OUT, WGRADS, DX>, dim3(p.grid1), dim3(tc::TsCfg::THREADS), tc::TsCfg::SMEM_BYTES, j1);
    } else {
      launch(h, st, PLAIN, tc::tc_bwd1_kernel<false, IN, OUT, WGRADS, DX>, dim3(p.grid1), dim3(tc::Pipe<false, tc::BWD1_NPW>::THREADS),
             tc::FwdSmem<false, tc::BWD1_NPW>::BYTES, j1);
    }
    mark_at(mk.mid);
    if (!WGRADS) return p;
    tc::Bwd2Job j2{jb.X, jb.dOut, jb.h2, jb.params, h->pw2_tc, h->small2, jb.rows, jb.n_nets, p.splits};
    if constexpr (F16X3) {
      if (p.pair2)
        launch(h, st2, PDL, tc::tc_bwd2_h2_kernel<IN, OUT>, dim3(2 * p.splits, jb.n_nets), dim3(tc::B2PCfg::THREADS), tc::B2PCfg::BYTES, j2);
      else
        launch(h, st2, PDL, tc::tc_bwd2_h_kernel<IN, OUT>, dim3(p.splits, jb.n_nets), dim3(tc::B2HCfg::THREADS), tc::B2HCfg::BYTES, j2);
    } else {
      constexpr bool TF32 = P == Prec::TF32X3;
      launch(h, st2, PLAIN, tc::tc_bwd2_kernel<TF32, IN, OUT>, dim3(p.splits, jb.n_nets), dim3(tc::B2_THREADS), tc::B2Cfg<TF32>::BYTES, j2);
    }
    if (p.fork) {
      CQL_CUDA(cudaEventRecord(h->ev_join, st2));
      CQL_CUDA(cudaStreamWaitEvent(st, h->ev_join, 0));
    }
    mark_at(mk.end);
    if (!p.fold)
      launch(h, st, pdl_skip(64), tc::k_reduce_grads_tc, dim3((NET_STRIDE / 4 + 31) / 32, jb.n_nets), dim3(256), 0, h->small1,
             p.slots1, h->small2, h->pw2_tc, p.splits, IN, OUT, grads_out, h->dp_fused ? h->dp : DpPeer{}, IN == 3 ? 1 : 2,
             (long long)(IN == 3 ? NET_STRIDE : 0));
    mark_at(mk.done);
  }
  return p;
}

// the networks one optimizer step updates: the critics or the actor, each with its Polyak-averaged target copy
struct NetGroup { int first_slot, n_nets, in_dim, out_dim; float lr; };
inline NetGroup critic_group(const Handle* h) { return NetGroup{slot_critic(0), h->C, 3, 1, h->cfg.critic_lr}; }
inline NetGroup actor_group(const Handle* h) { return NetGroup{slot_actor(), 1, 2, 2, h->cfg.actor_lr}; }

// Where an optimizer step may write the group's target copy instead of its target slots.  FQE's ordinary updates
// (fqe.cuh) leave the target slots and their packed copies as they are: k_adam_polyak then gets no target, the target
// slots are not repacked, and k_adam_pack -- which always writes a target copy -- writes it into this scratch.
struct TargetSink {
  float* params;     // [n_nets][NET_STRIDE]
  uint8_t* fwd;      // [n_nets][packed_net_bytes]
  uint8_t* fwd2;     // [n_nets][packed_net_bytes2] (f16x3)
};

// f16x3: Adam + Polyak + every operand copy of W2 (network and target, both orientations, both layouts) in one launch
inline void adam_pack(Handle* h, const NetGroup& g, const BwdPlan& plan, cudaStream_t st, bool last,
                      const TargetSink* sink = nullptr) {
  const cql_config& c = h->cfg;
  const bool critic = g.in_dim == 3;
  tc::AdamPackJobs j{};
  j.in_dim = g.in_dim; j.out_dim = g.out_dim;
  j.lr = g.lr; j.beta1 = c.beta1; j.beta2 = c.beta2; j.eps = c.adam_eps; j.tau = c.tau;
  j.step_inc = last ? h->step_dev : nullptr;
  j.dp = h->dp_fused ? h->dp : DpPeer{};
  j.dp_group = critic ? 1 : 2;
  j.dp_off = (long long)g.first_slot * NET_STRIDE;       // staging layout = gradient buffer layout [actor | critics | scalars]
  for (int i = 0; i < g.n_nets; ++i) {
    const int slot = g.first_slot + i, tslot = slot + 1 + h->C;       // [actor | critics | targ_actor | targ_critics]
    tc::AdamPackNet& n = j.n[i];
    n.p = h->net_params(slot);
    n.m = h->adam_m + (size_t)slot * NET_STRIDE;
    n.v = h->adam_v + (size_t)slot * NET_STRIDE;
    n.g = h->grads + (size_t)slot * NET_STRIDE;                      // grads: [actor | critics | scalars], same slot order
    n.targ = h->net_params(tslot);
    n.fwd = h->packed_fwd + (size_t)slot * h->packed_net_bytes;
    n.bwd = h->packed_bwd + (size_t)slot * h->packed_net_bytes_bwd;
    n.tfwd = h->packed_fwd + (size_t)tslot * h->packed_net_bytes;
    n.fwd2 = critic ? h->packed_fwd2 + (size_t)slot * h->packed_net_bytes2 : nullptr;
    n.bwd2 = critic ? h->packed_bwd2 + (size_t)slot * h->packed_net_bytes2 : nullptr;
    n.tfwd2 = critic ? h->packed_fwd2 + (size_t)tslot * h->packed_net_bytes2 : nullptr;
    n.w2max = h->w2max + slot * 4;
    if (sink) {
      n.targ = sink->params + (size_t)i * NET_STRIDE;
      n.tfwd = sink->fwd + (size_t)i * h->packed_net_bytes;
      n.tfwd2 = critic ? sink->fwd2 + (size_t)i * h->packed_net_bytes2 : nullptr;
    }
  }
  if (plan.fold) {                     // the partials of this group's backward (launch_bwd)
    j.small1 = h->small1; j.small2 = h->small2; j.pw2 = h->pw2_tc;
    j.slots1 = plan.slots1; j.splits = plan.splits;
    j.wmax_acc = h->ap_wmax;
  }
  const int blocks = tc::AP_W2_BLOCKS + (plan.fold ? tc::ap_small_blocks(g.in_dim, g.out_dim) : 1);
  launch(h, st, pdl_skip(128), tc::k_adam_pack, dim3(blocks, g.n_nets), dim3(1024), 0, j, h->stepinfo);
}

// Adam + Polyak of one group and the refresh of its packed W2 copies; `last`: the update's final launch, which also counts
// the step.  plan: the group's backward (launch_bwd), whose partials f16x3 sums here.  sink: the target slots stay as
// they are (TargetSink).
template <Prec P>
inline void optimizer_step(Handle* h, const NetGroup& g, const BwdPlan& plan, cudaStream_t st, bool last,
                           const TargetSink* sink = nullptr) {
  if (P == Prec::F16X3 && !switches().no_fused_adam) {
    adam_pack(h, g, plan, st, last, sink);
    return;
  }
  const cql_config& c = h->cfg;
  const int64_t cnt = (int64_t)g.n_nets * NET_STRIDE, off = (int64_t)g.first_slot * NET_STRIDE;
  const int tslot = g.first_slot + 1 + h->C;
  launch(h, st, PDL, k_adam_polyak, dim3((int)((cnt + 255) / 256)), dim3(256), 0, h->net_params(g.first_slot), h->adam_m + off,
         h->adam_v + off, h->grads + off, sink ? nullptr : h->net_params(tslot), cnt, g.lr, c.beta1, c.beta2, c.adam_eps, c.tau,
         h->stepinfo);
  int slots[2 * CQL_MAX_CRITICS], n = 0;
  for (int i = 0; i < g.n_nets; ++i) slots[n++] = g.first_slot + i;
  if (g.in_dim == 3 && !sink)          // the target critics' forward (TD target) reads the packed copy; the target actor's none
    for (int i = 0; i < g.n_nets; ++i) slots[n++] = tslot + i;
  pack_slots<P>(h, slots, n, st);
  if (last) launch(h, st, PDL, k_step_end, dim3(1), dim3(1), 0, h->step_dev);
}

inline LossConsts loss_consts(const Handle* h) {
  const cql_config& c = h->cfg;
  return LossConsts{h->B, h->n, h->C, c.gamma, c.conservative_weight, c.alpha_threshold,
                    c.temp_lr, c.alpha_lr, c.beta1, c.beta2, c.adam_eps, h->n_steps > 1 ? 1 : 0};
}

constexpr int TIMED_FWD_REPS = 4;
enum class BatchSource { Sampled, Provided };
enum class NoiseSource { Philox, Provided };

// phase 0: (sample, noise,) shared actor forward, all critic forwards, scalar gradients
template <Prec P>
inline void phase0(Handle* h, cudaStream_t st, BatchSource bs, NoiseSource ns) {
  NvtxRange nvtx("cql.update.phase0: sample, actor forward, critic forwards, temp/alpha gradients");
  const int B = h->B, C = h->C, n3 = 3 * h->n;
  const cql_config& c = h->cfg;
  mark(h, st, 0);
  const float4* batch4 = reinterpret_cast<const float4*>(h->batch);
  if (bs == BatchSource::Sampled && ns == NoiseSource::Philox) {
    CQL_REQUIRE(h->n_trans > 0, "cql_update: no transitions loaded (call cql_load_transitions first)");
    const int64_t nthr = h->noise_floats > B ? h->noise_floats : B;
    launch(h, st, pdl_skip(256), k_step_head, dim3((int)((nthr + 255) / 256)), dim3(256), 0, reinterpret_cast<const float4*>(h->table),
           h->n_trans, h->step_dev, h->stepinfo, c.beta1, c.beta2, B, h->n, c.rank, c.world_size, c.seed,
           reinterpret_cast<float4*>(h->batch), h->XA, h->noise, h->noise_floats, h->table_sharded ? 0 : c.rank,
           h->table_sharded ? 1 : c.world_size, h->prep);
  } else {
    launch(h, st, PLAIN, k_step_begin, dim3(1), dim3(1), 0, h->step_dev, h->stepinfo, c.beta1, c.beta2);
    if (bs == BatchSource::Sampled) {
      CQL_REQUIRE(h->n_trans > 0, "cql_update: no transitions loaded (call cql_load_transitions first)");
      launch(h, st, PLAIN, k_sample, dim3((B + 127) / 128), dim3(128), 0, reinterpret_cast<const float4*>(h->table), h->n_trans,
             nullptr, h->step_dev, 0, B, (int64_t)B * (h->table_sharded ? 1 : c.world_size), h->table_sharded ? 0 : c.rank,
             h->table_sharded ? 1 : c.world_size, c.seed, reinterpret_cast<float4*>(h->staged_batch()));
    }
    if (ns == NoiseSource::Philox)
      launch(h, st, PLAIN, k_noise, dim3((int)((h->noise_floats + 255) / 256)), dim3(256), 0, h->noise, h->noise_floats, B, h->n,
             c.seed, h->step_dev, c.rank);
    launch(h, st, PLAIN, k_actor_rows, dim3((2 * B + 255) / 256), dim3(256), 0, reinterpret_cast<const float4*>(h->staged_batch()),
           B, reinterpret_cast<float4*>(h->batch), h->XA, h->prep);
  }
  {
    FwdJobs jobs{};
    jobs.n = 2;
    jobs.j[0] = FwdJob{h->XA, h->net_params(slot_actor()), h->outA, h->h2A, B, 1, 0};
    jobs.j[1] = FwdJob{h->XA + B, h->net_params(slot_actor()), h->outA + 2 * (size_t)B, nullptr, B, 1, 0};
    mark(h, st, 1);
    QSrc srcA[2];
    launch_fwd<P, 2, 2>(h, jobs, st, srcA);
    mark(h, st, 2);
    launch(h, st, pdl_skip(1), k_prep, dim3((B * 64 + 255) / 256), dim3(256), 0, batch4, srcA[0], srcA[1], h->outA, h->noise, B,
           h->n, c.squash, h->XAl, h->offAl, h->XC, h->offC, h->XT, h->XP, reinterpret_cast<float4*>(h->perb));
  }
  {
    FwdJobs jobs{};
    jobs.n = 3;
    jobs.j[0] = FwdJob{h->XAl, h->net_params(slot_critic(0)), h->QAl, nullptr, B * n3, C, 0};
    jobs.j[1] = FwdJob{h->XC, h->net_params(slot_critic(0)), h->QC, h->h2C, B * (n3 + 1), C, 0};
    jobs.j[2] = FwdJob{h->XT, h->net_params(slot_targ_critic(C, 0)), h->QT, nullptr, B, C, 0};
    mark(h, st, 3);
    QSrc srcQ[3];
    // cql_timed_update: the launch is repeated back to back between the two events (same inputs, same outputs), so that
    // the reported duration is the kernel's steady-state launch-to-launch time, not one launch plus its launch latency
    // (the repeats are launched the way the step graph launches this kernel -- with programmatic dependent launch -- so a
    //  repeat's prologue overlaps its predecessor's drain exactly as it overlaps k_prep's in the product schedule; the
    //  events on either side still separate the four launches from their neighbours)
    const bool pdl_off = h->pdl_off;
    for (int rep = 0; rep < (h->timing ? TIMED_FWD_REPS : 1); ++rep) {
      h->pdl_off = pdl_off && rep == 0;
      launch_fwd<P, 3, 1>(h, jobs, st, srcQ);
    }
    h->pdl_off = pdl_off;
    mark(h, st, 4);
    // (the last block of k_lse also sums the pair values and publishes the two scalar gradients: the former k_scalar_reduce)
    const int64_t so = scalars_off(C);
    ScalarReduceArgs ra{reinterpret_cast<const float4*>(h->perb), h->scalars(), h->adam_m + so, h->adam_v + so, h->g_scalars(),
                        h->loss_sums, h->metrics, reinterpret_cast<unsigned int*>(h->loss_sums + 15), h->dp_fused ? h->dp : DpPeer{}};
    launch(h, st, pdl_skip(2), 3 * h->n + 1 <= 32 ? &k_lse<false> : &k_lse<true>, dim3((C * B * 32 + 255) / 256), dim3(256), 0,
           batch4, srcQ[0], h->offAl, srcQ[1], h->offC, srcQ[2], loss_consts(h), h->dQ, reinterpret_cast<PairVals*>(h->pairv), ra);
  }
}

// phase 1: temp/alpha Adam, critic backward -> critic gradients
template <Prec P>
inline void phase1(Handle* h, cudaStream_t st) {
  NvtxRange nvtx("cql.update.phase1: temp/alpha Adam, critic backward");
  const int B = h->B, C = h->C, rows = B * (3 * h->n + 1);
  const int64_t so = scalars_off(C);
  launch(h, st, pdl_skip(8), k_scalar_adam_dq, dim3((int)(((int64_t)C * rows + 255) / 256)), dim3(256), 0, h->scalars(),
         h->adam_m + so, h->adam_v + so, h->g_scalars(), h->stepinfo, loss_consts(h), h->loss_sums, h->metrics,
         reinterpret_cast<const PairVals*>(h->pairv), h->dQ, h->dp_fused ? h->dp : DpPeer{}, (long long)(1 + C) * NET_STRIDE);
  mark(h, st, 5);
  launch_bwd<P, 3, 1, true, false>(h, critic_bwd_job(h), h->g_critics(), st, BwdMarks{6, 7, -1});
}

// phase 2: critic Adam + Polyak, actor loss through the updated critics -> actor gradients
template <Prec P>
inline void phase2(Handle* h, cudaStream_t st) {
  NvtxRange nvtx("cql.update.phase2: critic Adam + Polyak + pack, actor step forward/backward");
  const int B = h->B, C = h->C;
  optimizer_step<P>(h, critic_group(h), bwd_plan<P, 3, 1, true, false>(h, critic_bwd_job(h)), st, false);
  FwdJobs jobs{};
  jobs.n = 1;
  jobs.j[0] = FwdJob{h->XP, h->net_params(slot_critic(0)), h->QP, h->h2P, B, C, 0};
  mark(h, st, 8);
  QSrc srcP;
  launch_fwd<P, 3, 1>(h, jobs, st, &srcP);
  mark(h, st, 9);
  // the forward left partial sums (f16x3): the dx-only bwd1 below takes dQ from them itself, k_actor_dout the metric
  const bool fold_dq = srcP.n_parts > 0;
  const float4* perb = reinterpret_cast<const float4*>(h->perb);
  if (!fold_dq)
    launch(h, st, pdl_skip(16), k_actor_dq, dim3(1), dim3(1024), 0, srcP, perb, h->scalars(), B, C, h->dQP, h->metrics);
  BwdJob jd{h->XP, h->dQP, h->h2P, h->net_params(slot_critic(0)), nullptr, h->dXP, nullptr, B, C, 1};
  if (fold_dq) { jd.q_part = srcP.q; jd.q_parts = srcP.n_parts; jd.dq_scale = -1.f / (float)B; }
  const BwdPlan dx = launch_bwd<P, 3, 1, false, true>(h, jd, nullptr, st);
  launch(h, st, pdl_skip(32), k_actor_dout, dim3((B + 127) / 128), dim3(128), 0, h->outA, h->noise + B + 6 * (int64_t)B * h->n,
         dx.dx, h->scalars(), B, dx.dx_parts, h->cfg.squash, h->dOutA, fold_dq ? srcP : QSrc{}, perb, C, h->actor_part,
         reinterpret_cast<unsigned int*>(h->loss_sums + 14), h->metrics);
  mark(h, st, 10);
  launch_bwd<P, 2, 2, true, false>(h, actor_bwd_job(h), h->g_actor(), st, BwdMarks{-1, -1, 11});
}

// phase 3: actor Adam + Polyak of the target policy, step counter
template <Prec P>
inline void phase3(Handle* h, cudaStream_t st) {
  NvtxRange nvtx("cql.update.phase3: actor Adam + Polyak + pack");
  optimizer_step<P>(h, actor_group(h), bwd_plan<P, 2, 2, true, false>(h, actor_bwd_job(h)), st, true);
  mark(h, st, 12);
}

}  // namespace cql
