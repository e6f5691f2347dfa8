// offline_eval.cuh -- d3rlpy's offline scorers over the one-step replay table (cql_offline_eval, DESIGN.md section 1).
//
// Per table row i = (s, a, r | s', term):  Q(s,a) = mean_c Q_c(s, a'), V(s) = mean_c Q_c(s, pi(s)) with
// pi = tanh(mu) in network space, sigma(s) = population std of Q_c(s, pi(s)) over the critics, the one-step TD error
// (Q(s,a) - y)^2 with y = r' + gamma * V(s') * (1 - term), and (a - reverse(pi(s)))^2.  V(s') of a non-terminal row is
// the next row's V(s) whenever s' is bit-equal to the next row's s -- the same forward of the same input -- so only
// rows where that fails (a table end without a terminal row, verbatim tables) get an explicit s' actor and critic row.
//
// The forwards run in chunks of OE_CHUNK rows through the update's launch_fwd (one actor job, one critic job over the
// data rows and the policy rows) and leave five float32 values per row in whole-table arrays.  Whole-table passes then
// find each row's episode start (an inclusive max-scan), run d3rlpy's 1024-row advantage windows (one thread per
// window, backwards, float64) and each episode's raw return (one thread per episode start, window by window), and a
// fixed-tree float64 reduction sums everything: the order depends only on the row count (as k_stats_partial /
// k_stats_final), so the same table gives the same bits on any stream.
#pragma once
#include <cub/cub.cuh>
#include "update.cuh"

namespace cql {

constexpr int64_t OE_CHUNK = 1 << 18;                     // table rows per forward chunk
constexpr int OE_WINDOW = 1024;                           // d3rlpy metrics/scorer.py WINDOW_SIZE
constexpr int OE_THREADS = 256, OE_ROWS = 32 * OE_THREADS, OE_MAX_BLOCKS = 1024;
constexpr int OE_SUMS = 10;   // td, adv, V, sigma, V(s0), action diff, success Q, all-row Q, episodes, success rows

// a non-terminal row whose s' is not bit-equal to the next row's s needs its own s' forward
__device__ __forceinline__ bool oe_explicit_next(const float4* __restrict__ rows, int64_t n, int64_t i) {
  const float4 b = rows[2 * i + 1];
  if (b.z != 0.f) return false;
  if (i + 1 >= n) return true;
  const float4 a = rows[2 * (i + 1)];
  return __float_as_uint(b.x) != __float_as_uint(a.x) || __float_as_uint(b.y) != __float_as_uint(a.y);
}

__global__ void k_oe_count(const float4* __restrict__ rows, int64_t n, int* __restrict__ per_chunk) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && oe_explicit_next(rows, n, i)) atomicAdd(per_chunk + i / OE_CHUNK, 1);
}

// actor input rows of chunk [c0, c0 + m): the m rows' s, then row c0 + m's s when it exists (its V is the last row's
// V(s')), then the explicit s' rows in slots behind them (xslot[l] = slot, -1 = none).  The slot order comes from an
// atomic counter, but each row's forward does not depend on its position in the launch.
__global__ void k_oe_head(const float4* __restrict__ rows, int64_t n, int64_t c0, int m, int ma, const Prep prep,
                          float4* __restrict__ XA, int* __restrict__ xslot, int* __restrict__ counter) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= ma) return;
  const int64_t i = c0 + l;
  const float4 a = rows[2 * i];
  XA[l] = make_float4(prep_fwd(prep.obs[0], a.x), prep_fwd(prep.obs[1], a.y), 0.f, 0.f);
  if (l >= m) return;
  int slot = -1;
  if (oe_explicit_next(rows, n, i)) {
    const float4 b = rows[2 * i + 1];
    slot = atomicAdd(counter, 1);
    XA[ma + slot] = make_float4(prep_fwd(prep.obs[0], b.x), prep_fwd(prep.obs[1], b.y), 0.f, 0.f);
  }
  xslot[l] = slot;
}

// critic rows from the actor outputs: [0, m) = (s, a') of the data rows, [m, m + n_act) = (x, pi(x)) of every actor
// row; the action difference of the data rows against the reverse-transformed greedy action
__global__ void k_oe_prep(const float4* __restrict__ rows, int64_t c0, int m, int n_act, const float4* __restrict__ XA,
                          const QSrc srcA, const Prep prep, float4* __restrict__ XC, float* __restrict__ cad) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_act) return;
  const float pi = (float)tanh((double)q_at(srcA, 0, r, 0));   // as the update's TD-target row
  const float4 x = XA[r];
  XC[m + r] = make_float4(x.x, x.y, pi, 0.f);
  if (r < m) {
    const float a = rows[2 * (c0 + r)].z;
    XC[r] = make_float4(x.x, x.y, act_fwd(prep.act, a), 0.f);
    const float d = __fsub_rn(a, act_rev(prep.act, pi));
    cad[c0 + r] = __fmul_rn(d, d);
  }
}

__device__ __forceinline__ float oe_mean(const QSrc& s, int C, int r) {
  float v = 0.f;
  for (int c = 0; c < C; ++c) v = __fadd_rn(v, q_at(s, c, r));
  return __fdiv_rn(v, (float)C);
}

// mean_c Q_c of row r and, when sd is not null, the population std over the critics (numpy std, ddof 0; exactly 0 at
// C = 1): float32, critic order 0..C-1, separately rounded sums, a two-pass variance.  The offline scorers' V and
// sigma and cql_predict_value (infer.cuh) both come from here.
__device__ __forceinline__ float ens_mean_std(const QSrc& s, int C, int r, float* sd) {
  float qc[CQL_MAX_CRITICS];
  float sum = 0.f;
  for (int c = 0; c < C; ++c) { qc[c] = q_at(s, c, r); sum = __fadd_rn(sum, qc[c]); }
  const float mean = __fdiv_rn(sum, (float)C);
  if (sd) {
    float var = 0.f;
    for (int c = 0; c < C; ++c) { const float d = __fsub_rn(qc[c], mean); var = __fadd_rn(var, __fmul_rn(d, d)); }
    *sd = sqrtf(__fdiv_rn(var, (float)C));
  }
  return mean;
}

// per data row: Q(s,a), V(s), sigma(s), TD error
__global__ void k_oe_rows(const float4* __restrict__ rows, int64_t c0, int m, int ma, const int* __restrict__ xslot,
                          const QSrc srcQ, int C, float gamma, const Prep prep, float* __restrict__ qd,
                          float* __restrict__ v, float* __restrict__ sg, float* __restrict__ td) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= m) return;
  const int64_t i = c0 + l;
  const float q = oe_mean(srcQ, C, l);
  float sd;
  const float vs = ens_mean_std(srcQ, C, m + l, &sd);
  const float4 r0 = rows[2 * i], r1 = rows[2 * i + 1];
  float vn = 0.f;                                       // a terminal row's bootstrap is multiplied by 0
  if (r1.z == 0.f) vn = oe_mean(srcQ, C, xslot[l] >= 0 ? m + ma + xslot[l] : m + l + 1);
  const float y = __fadd_rn(prep_fwd(prep.rew, r0.w), __fmul_rn(__fmul_rn(gamma, vn), __fsub_rn(1.f, r1.z)));
  const float e = __fsub_rn(q, y);
  qd[i] = q;
  v[i] = vs;
  sg[i] = sd;
  td[i] = __fmul_rn(e, e);
}

// episode heads: row 0 and every row after a terminal one -> key = i (else 0); the max-scan gives each row's start
__global__ void k_oe_head_keys(const float4* __restrict__ rows, int64_t n, int64_t* __restrict__ key) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) key[i] = (i == 0 || rows[2 * (i - 1) + 1].z != 0.f) ? i : 0;
}
struct OeMax {
  __device__ __forceinline__ int64_t operator()(int64_t a, int64_t b) const { return a > b ? a : b; }
};

// one thread per window start (offset from the episode start a multiple of OE_WINDOW): the window's advantage
// recursion A = adv_last, A = adv_t + gamma * A backwards in float64 (sum of every A_t -> wA), its raw-reward sum, its
// Q(s,a) sum and its length
__global__ void k_oe_windows(const float4* __restrict__ rows, int64_t n, const int64_t* __restrict__ start,
                             const float* __restrict__ qd, const float* __restrict__ v, double gamma,
                             double* __restrict__ wA, double* __restrict__ wR, double* __restrict__ wQ,
                             int* __restrict__ wL) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if ((i - start[i]) % OE_WINDOW != 0) { wA[i] = 0.0; return; }
  int64_t e = i;
  double ret = 0.0, qs = 0.0;
  for (;;) {
    ret += (double)rows[2 * e].w;
    qs += (double)qd[e];
    if (rows[2 * e + 1].z != 0.f || e + 1 >= n || e + 1 - i >= OE_WINDOW) break;
    ++e;
  }
  double A = 0.0, sum = 0.0;
  for (int64_t j = e; j >= i; --j) {
    const double adv = (double)__fsub_rn(qd[j], v[j]);
    A = j == e ? adv : adv + gamma * A;
    sum += A;
  }
  wA[i] = sum; wR[i] = ret; wQ[i] = qs; wL[i] = (int)(e - i + 1);
}

// one thread per episode start: the episode's raw return over its windows in order; a successful episode
// (return >= threshold) leaves its Q(s,a) sum in wR[head] and its length in wQ[head], every other head 0, 0
__global__ void k_oe_episodes(int64_t n, const int64_t* __restrict__ start, double thr, int use_thr,
                              double* __restrict__ wR, double* __restrict__ wQ, const int* __restrict__ wL) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || start[i] != i) return;
  double ret = 0.0, qs = 0.0, len = 0.0;
  for (int64_t j = i; j < n && start[j] == i; j += OE_WINDOW) { ret += wR[j]; qs += wQ[j]; len += (double)wL[j]; }
  const bool ok = use_thr && ret >= thr;
  wR[i] = ok ? qs : 0.0;
  wQ[i] = ok ? len : 0.0;
}

struct OeRows {
  const float *td, *v, *sg, *cad, *qd;
  const double *wA, *wR, *wQ;
  const int64_t* start;
};
__device__ __forceinline__ void oe_row(const OeRows& a, int64_t i, double (&s)[OE_SUMS]) {
  const bool head = a.start[i] == i;
  s[0] += (double)a.td[i];
  s[1] += a.wA[i];
  s[2] += (double)a.v[i];
  s[3] += (double)a.sg[i];
  s[5] += (double)a.cad[i];
  s[7] += (double)a.qd[i];
  if (head) { s[4] += (double)a.v[i]; s[6] += a.wR[i]; s[8] += 1.0; s[9] += a.wQ[i]; }
}
__device__ void oe_block_store(double (&s)[OE_SUMS], double* __restrict__ out) {
  __shared__ double sm[OE_THREADS];
  for (int k = 0; k < OE_SUMS; ++k) {
    sm[threadIdx.x] = s[k];
    __syncthreads();
    for (int w = OE_THREADS / 2; w > 0; w >>= 1) {
      if (threadIdx.x < w) sm[threadIdx.x] += sm[threadIdx.x + w];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[k] = sm[0];
    __syncthreads();
  }
}
__global__ void __launch_bounds__(OE_THREADS) k_oe_partial(const OeRows a, int64_t n, int64_t per_block,
                                                           double* __restrict__ part) {
  double s[OE_SUMS] = {};
  const int64_t base = (int64_t)blockIdx.x * per_block;
  for (int64_t j = threadIdx.x; j < per_block && base + j < n; j += OE_THREADS) oe_row(a, base + j, s);
  oe_block_store(s, part + (size_t)OE_SUMS * blockIdx.x);
}
__global__ void __launch_bounds__(OE_THREADS) k_oe_final(const double* __restrict__ part, int64_t nb,
                                                         double* __restrict__ out) {
  double s[OE_SUMS] = {};
  for (int64_t b = threadIdx.x; b < nb; b += OE_THREADS)
    for (int k = 0; k < OE_SUMS; ++k) s[k] += part[(size_t)OE_SUMS * b + k];
  oe_block_store(s, out);
}

// the whole evaluation on `st`; returns the ten sums in `out` (host) after synchronising `st`
template <Prec P>
void offline_eval(Handle* h, float thr, double* out, cudaStream_t st) {
  const int64_t n = h->n_trans;
  const int C = h->C;
  const float4* rows = reinterpret_cast<const float4*>(h->table);
  const unsigned gb = (unsigned)((n + 255) / 256);
  DevTmp tmp(st);
  // explicit s' rows per chunk: the forward launches need their row counts on the host
  const int64_t n_chunks = (n + OE_CHUNK - 1) / OE_CHUNK;
  int* per_chunk = tmp.get<int>(n_chunks + 1);
  CQL_CUDA(cudaMemsetAsync(per_chunk, 0, (n_chunks + 1) * sizeof(int), st));
  k_oe_count<<<gb, 256, 0, st>>>(rows, n, per_chunk);
  CQL_LAUNCH_CHECK(h);
  std::vector<int> extra(n_chunks);
  CQL_CUDA(cudaMemcpyAsync(extra.data(), per_chunk, n_chunks * sizeof(int), cudaMemcpyDeviceToHost, st));
  CQL_CUDA(cudaStreamSynchronize(st));
  const int max_extra = *std::max_element(extra.begin(), extra.end());
  const int cm = (int)std::min<int64_t>(OE_CHUNK, n);
  const int ra_max = cm + 1 + max_extra, rc_max = cm + ra_max;
  float4* XA = tmp.get<float4>(ra_max);
  float* outA = tmp.get<float>(2 * (size_t)ra_max);
  float4* XC = tmp.get<float4>(rc_max);
  float* QC = tmp.get<float>((size_t)C * rc_max);
  const size_t part_floats = (size_t)Q_MAX_PARTS * std::max<size_t>(2 * (size_t)ra_max, (size_t)C * rc_max);
  float* part = tmp.get<float>(part_floats);
  int* xslot = tmp.get<int>(cm);
  float* qd = tmp.get<float>(n);
  float* v = tmp.get<float>(n);
  float* sg = tmp.get<float>(n);
  float* td = tmp.get<float>(n);
  float* cad = tmp.get<float>(n);
  for (int64_t k = 0; k < n_chunks; ++k) {
    const int64_t c0 = k * OE_CHUNK;
    const int m = (int)std::min<int64_t>(OE_CHUNK, n - c0);
    const int ma = c0 + m < n ? m + 1 : m;             // + the next chunk's first row
    const int n_act = ma + extra[k];
    int* counter = per_chunk + n_chunks;
    CQL_CUDA(cudaMemsetAsync(counter, 0, sizeof(int), st));
    k_oe_head<<<(unsigned)((ma + 255) / 256), 256, 0, st>>>(rows, n, c0, m, ma, h->prep, XA, xslot, counter);
    CQL_LAUNCH_CHECK(h);
    FwdJobs ja{};
    ja.n = 1;
    ja.j[0] = FwdJob{XA, h->net_params(slot_actor()), outA, nullptr, n_act, 1, 0};
    QSrc srcA;
    launch_fwd<P, 2, 2>(h, ja, st, &srcA, part, part_floats);
    launch(h, st, PDL, k_oe_prep, dim3((n_act + 255) / 256), dim3(256), 0, rows, c0, m, n_act, (const float4*)XA, srcA,
           h->prep, XC, cad);
    FwdJobs jc{};
    jc.n = 1;
    jc.j[0] = FwdJob{XC, h->net_params(slot_critic(0)), QC, nullptr, m + n_act, C, 0};
    QSrc srcQ;
    launch_fwd<P, 3, 1>(h, jc, st, &srcQ, part, part_floats);
    launch(h, st, PDL, k_oe_rows, dim3((m + 255) / 256), dim3(256), 0, rows, c0, m, ma, (const int*)xslot, srcQ, C,
           h->cfg.gamma, h->prep, qd, v, sg, td);
  }
  // episode starts
  int64_t* key = tmp.get<int64_t>(n);
  int64_t* start = tmp.get<int64_t>(n);
  k_oe_head_keys<<<gb, 256, 0, st>>>(rows, n, key);
  CQL_LAUNCH_CHECK(h);
  size_t scan_bytes = 0;
  CQL_CUDA(cub::DeviceScan::InclusiveScan(nullptr, scan_bytes, key, start, OeMax(), n, st));
  uint8_t* scan_tmp = tmp.get<uint8_t>(scan_bytes + 16);
  CQL_CUDA(cub::DeviceScan::InclusiveScan(scan_tmp, scan_bytes, key, start, OeMax(), n, st));
  h->launches++;
  // windows, episodes
  double* wA = tmp.get<double>(n);
  double* wR = tmp.get<double>(n);
  double* wQ = tmp.get<double>(n);
  int* wL = tmp.get<int>(n);
  k_oe_windows<<<gb, 256, 0, st>>>(rows, n, start, qd, v, (double)h->cfg.gamma, wA, wR, wQ, wL);
  CQL_LAUNCH_CHECK(h);
  k_oe_episodes<<<gb, 256, 0, st>>>(n, start, (double)thr, std::isnan(thr) ? 0 : 1, wR, wQ, wL);
  CQL_LAUNCH_CHECK(h);
  // fixed-tree reduction
  const int64_t nb = std::min<int64_t>((n + OE_ROWS - 1) / OE_ROWS, OE_MAX_BLOCKS);
  const int64_t per_block = (n + nb - 1) / nb;
  double* partials = tmp.get<double>((size_t)(nb + 1) * OE_SUMS);
  double* result = partials + (size_t)nb * OE_SUMS;
  OeRows ar{td, v, sg, cad, qd, wA, wR, wQ, start};
  k_oe_partial<<<(unsigned)nb, OE_THREADS, 0, st>>>(ar, n, per_block, partials);
  CQL_LAUNCH_CHECK(h);
  k_oe_final<<<1, OE_THREADS, 0, st>>>(partials, nb, result);
  CQL_LAUNCH_CHECK(h);
  CQL_CUDA(cudaMemcpyAsync(out, result, OE_SUMS * sizeof(double), cudaMemcpyDeviceToHost, st));
  CQL_CUDA(cudaStreamSynchronize(st));
}

}  // namespace cql
