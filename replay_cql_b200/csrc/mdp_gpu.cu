// mdp_gpu.cu -- MDP builder on the GPU (SURVEY.md section 8 row a7 / "next" item 1).
//
// Replaces the wrapper's two Spark window sorts + global orderBy + toPandas ([EXT] MdpDatasetBuilder.build) with
// stable LSD radix sorts on the device (CUB: library code, like cuBLAS -- sorting is not the hot path's arithmetic):
//   order      = stable sort by (user, timestamp)                 : sort by ts, then by user
//   rank order = stable sort by (user, relevance desc, ts desc)   : sort by ts desc, rel desc, user
// followed by one pass that writes the 32-byte transition rows (reward = rank-in-user < top_k, terminal = last
// row of the user, action = relevance + noise, next_obs = next row of the same user).  Ties keep input order,
// exactly like the host builder (replay_cql_b200/mdp.py), which the tests hold it bit-exact against.
#include <algorithm>
#include <cmath>
#include <initializer_list>
#include <vector>
#include <cstring>
#include <memory>
#include <thread>
#include <cub/cub.cuh>
#include "engine.cuh"

using namespace cql;

namespace {

__global__ void k_iota(uint32_t* p, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (uint32_t)i;
}
template <typename T>
__global__ void k_gather(const T* __restrict__ src, const uint32_t* __restrict__ idx, int64_t n, T* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}
// head position of every run of equal users in a user-sorted sequence (0 elsewhere) -> max-scan = group start
__global__ void k_heads(const int32_t* __restrict__ u_sorted, int64_t n, int64_t* __restrict__ head) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) head[i] = (i == 0 || u_sorted[i] != u_sorted[i - 1]) ? i : 0;
}
__global__ void k_rewarded(const uint32_t* __restrict__ rank_order, const int64_t* __restrict__ group_start, int64_t n,
                           int top_k, uint8_t* __restrict__ rewarded) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) rewarded[rank_order[i]] = (i - group_start[i]) < top_k ? 1 : 0;
}
struct MaxOp {
  __device__ __forceinline__ int64_t operator()(int64_t a, int64_t b) const { return a > b ? a : b; }
};

__global__ void k_emit(const uint32_t* __restrict__ order, const int32_t* __restrict__ user, const int32_t* __restrict__ item,
                       const double* __restrict__ rel, const double* __restrict__ noise, const uint8_t* __restrict__ rewarded,
                       int64_t n, float noise_scale, uint64_t seed, float4* __restrict__ table, float* __restrict__ obs_o,
                       float* __restrict__ act_o, float* __restrict__ rew_o, float* __restrict__ term_o) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t row = order[i];
  const int32_t u = user[row];
  const bool last = (i == n - 1) || user[order[i + 1]] != u;
  double nz;
  if (noise) {
    nz = noise[row];
  } else {                                   // seeded N(0,1) * scale per ORIGINAL row
    uint32_t r[4];
    Philox::gen(seed ^ 0xA0761D6478BD642Full, 0x4D4450ull, (uint64_t)row, r);
    nz = (double)(sqrtf(-2.f * logf(u01(r[0]))) * cospif(2.f * u01(r[1])) * noise_scale);
  }
  const float act = (float)((double)(float)rel[row] + nz);
  const float rw = rewarded[row] ? 1.f : 0.f;
  const float uf = (float)u, itf = (float)item[row];
  float nu = 0.f, ni = 0.f;
  if (!last) { nu = uf; ni = (float)item[order[i + 1]]; }
  table[2 * i] = make_float4(uf, itf, act, rw);
  table[2 * i + 1] = make_float4(nu, ni, last ? 1.f : 0.f, 0.f);
  if (obs_o) { obs_o[2 * i] = uf; obs_o[2 * i + 1] = itf; act_o[i] = act; rew_o[i] = rw; term_o[i] = last ? 1.f : 0.f; }
}

// Session scratch comes from the stream-ordered pool (keep_pool_cached, engine.cuh); the caller synchronises `st`
// before the pointers are used on another stream.
template <typename T>
T* dmalloc(size_t n, std::vector<void*>& pool, cudaStream_t st) {
  keep_pool_cached();
  void* p = nullptr;
  CQL_CUDA(cudaMallocAsync(&p, std::max<size_t>(1, n) * sizeof(T), st));
  pool.push_back(p);
  return reinterpret_cast<T*>(p);
}

// raw column chunk (any accepted dtype) -> the builder's column type
template <typename S, typename D>
__global__ void k_convert(const S* __restrict__ src, D* __restrict__ dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (D)src[i];
}

void parallel_memcpy(uint8_t* dst, const uint8_t* src, size_t bytes) {
  constexpr size_t MIN_PER_THREAD = 2u << 20;
  const int n_thr = (int)std::min<size_t>(4, std::max<size_t>(1, bytes / MIN_PER_THREAD));
  if (n_thr <= 1) { std::memcpy(dst, src, bytes); return; }
  std::vector<std::thread> th;
  const size_t per = (bytes / n_thr + 63) & ~(size_t)63;
  for (int t = 1; t < n_thr; ++t) {
    const size_t lo = std::min(bytes, per * t), hi = std::min(bytes, per * (t + 1));
    if (hi > lo) th.emplace_back([=] { std::memcpy(dst + lo, src + lo, hi - lo); });
  }
  std::memcpy(dst, src, std::min(bytes, per));
  for (auto& x : th) x.join();
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Ingestion session (SURVEY.md 8f-1): Arrow record batches / Parquet row groups / pandas columns arrive as CHUNKS of
// host memory in their own dtype.  Each chunk is copied -- by up to four host threads -- into a slot of a pinned ring and
// goes to the device with cudaMemcpyAsync on a copy stream (pageable memory handed to cudaMemcpy directly is staged by
// the driver in small pieces: r01 measured 0.14 - 1.3 s for the 480 MB of an ML-20M log); a one-line kernel converts the
// dtype where it differs from the builder's.  As soon as the TIMESTAMP column is complete the first two radix sorts (by
// timestamp, ascending and descending) start on the compute stream while the other columns are still in flight.
struct cql::MdpSession {
  int64_t n = 0;
  int32_t *user = nullptr, *item = nullptr;
  int64_t* ts = nullptr;
  double *rel = nullptr, *noise = nullptr;
  int64_t filled[5] = {0, 0, 0, 0, 0};
  uint32_t *ia = nullptr, *ib = nullptr, *perm_desc = nullptr, *order = nullptr;
  int64_t *k64a = nullptr, *k64b = nullptr;
  double *kda = nullptr, *kdb = nullptr;
  int32_t *k32a = nullptr, *k32b = nullptr;
  uint8_t* rewarded = nullptr;
  void* temp = nullptr;
  size_t tbytes = 0;
  static constexpr int SLOTS = 4;
  static constexpr size_t SLOT_BYTES = 16u << 20;
  uint8_t* ring = nullptr;          // pinned [SLOTS][SLOT_BYTES] (owned by the handle: allocated once, 64 MB of page-locking is not free)
  uint8_t* raw = nullptr;           // device [SLOTS][SLOT_BYTES] (chunks whose dtype needs converting)
  cudaEvent_t slot_ev[SLOTS] = {};
  int next_slot = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_ts = nullptr, ev_all = nullptr;
  bool stage_a = false;
  int64_t launches = 0;
  std::vector<void*> pool;

  cudaStream_t alloc_stream = nullptr;      // the handle's stream: every session buffer is allocated and released on it

  ~MdpSession() {
    if (alloc_stream) cudaStreamSynchronize(alloc_stream);
    if (copy_stream) cudaStreamSynchronize(copy_stream);
    for (void* p : pool) cudaFreeAsync(p, alloc_stream);
    for (auto& e : slot_ev) if (e) cudaEventDestroy(e);
    if (ev_ts) cudaEventDestroy(ev_ts);
    if (ev_all) cudaEventDestroy(ev_all);
    if (copy_stream) cudaStreamDestroy(copy_stream);
  }
};

namespace {
size_t dtype_bytes(int dt) { return dt == CQL_DT_I32 || dt == CQL_DT_F32 ? 4 : 8; }

template <typename D>
void convert_chunk(int dtype, const void* raw, D* dst, int64_t cnt, cudaStream_t st) {
  const unsigned nb = (unsigned)((cnt + 255) / 256);
  switch (dtype) {
    case CQL_DT_I32: k_convert<int32_t, D><<<nb, 256, 0, st>>>((const int32_t*)raw, dst, cnt); break;
    case CQL_DT_I64: k_convert<int64_t, D><<<nb, 256, 0, st>>>((const int64_t*)raw, dst, cnt); break;
    case CQL_DT_F32: k_convert<float, D><<<nb, 256, 0, st>>>((const float*)raw, dst, cnt); break;
    default: k_convert<double, D><<<nb, 256, 0, st>>>((const double*)raw, dst, cnt); break;
  }
  CQL_CUDA(cudaGetLastError());
}

// the two timestamp sorts: need nothing but the timestamp column
void mdp_stage_a(Handle& h, MdpSession& m) {
  cudaStream_t st = h.own_stream;
  const int64_t n = m.n;
  const unsigned nb = (unsigned)((n + 255) / 256);
  size_t tb;
  CQL_CUDA(cudaStreamWaitEvent(st, m.ev_ts, 0));
  k_iota<<<nb, 256, 0, st>>>(m.ia, n);
  tb = m.tbytes; CQL_CUDA(cub::DeviceRadixSort::SortPairs(m.temp, tb, m.ts, m.k64a, m.ia, m.ib, (int)n, 0, 64, st));            // ib = by ts asc
  tb = m.tbytes; CQL_CUDA(cub::DeviceRadixSort::SortPairsDescending(m.temp, tb, m.ts, m.k64a, m.ia, m.perm_desc, (int)n, 0, 64, st));   // by ts desc
  m.launches += 7;
  m.stage_a = true;
}
}  // namespace

void cql::mdp_session_free(MdpSession* m) { delete m; }

void cql::mdp_begin(Handle& h, int64_t n) {
  CQL_REQUIRE(n >= 1 && n < (1ll << 31), "cql_mdp_begin: n must be in 1..2^31-1");
  if (h.mdp) { delete h.mdp; h.mdp = nullptr; }
  auto* m = new MdpSession();
  h.mdp = m;
  m->n = n;
  m->alloc_stream = h.own_stream;
  m->user = dmalloc<int32_t>(n, m->pool, m->alloc_stream);
  m->item = dmalloc<int32_t>(n, m->pool, m->alloc_stream);
  m->ts = dmalloc<int64_t>(n, m->pool, m->alloc_stream);
  m->rel = dmalloc<double>(n, m->pool, m->alloc_stream);
  m->ia = dmalloc<uint32_t>(n, m->pool, m->alloc_stream);
  m->ib = dmalloc<uint32_t>(n, m->pool, m->alloc_stream);
  m->perm_desc = dmalloc<uint32_t>(n, m->pool, m->alloc_stream);
  m->order = dmalloc<uint32_t>(n, m->pool, m->alloc_stream);
  m->k64a = dmalloc<int64_t>(n, m->pool, m->alloc_stream);
  m->k64b = dmalloc<int64_t>(n, m->pool, m->alloc_stream);
  m->kda = dmalloc<double>(n, m->pool, m->alloc_stream);
  m->kdb = dmalloc<double>(n, m->pool, m->alloc_stream);
  m->k32a = dmalloc<int32_t>(n, m->pool, m->alloc_stream);
  m->k32b = dmalloc<int32_t>(n, m->pool, m->alloc_stream);
  m->rewarded = dmalloc<uint8_t>(n, m->pool, m->alloc_stream);
  size_t t1 = 0, t2 = 0, t3 = 0, t4 = 0, t5 = 0;
  cudaStream_t st = h.own_stream;
  cub::DeviceRadixSort::SortPairs(nullptr, t1, m->ts, m->k64a, m->ia, m->ib, (int)n, 0, 64, st);
  cub::DeviceRadixSort::SortPairs(nullptr, t2, m->k32a, m->k32b, m->ia, m->ib, (int)n, 0, 32, st);
  cub::DeviceRadixSort::SortPairsDescending(nullptr, t3, m->ts, m->k64a, m->ia, m->ib, (int)n, 0, 64, st);
  cub::DeviceRadixSort::SortPairsDescending(nullptr, t4, m->kda, m->kdb, m->ia, m->ib, (int)n, 0, 64, st);
  cub::DeviceScan::InclusiveScan(nullptr, t5, m->k64a, m->k64b, MaxOp(), (int)n, st);
  m->tbytes = t1;
  for (size_t t : {t2, t3, t4, t5}) m->tbytes = t > m->tbytes ? t : m->tbytes;
  m->temp = dmalloc<uint8_t>(m->tbytes, m->pool, m->alloc_stream);
  if (h.mdp_ring == nullptr) CQL_CUDA(cudaMallocHost(&h.mdp_ring, MdpSession::SLOTS * MdpSession::SLOT_BYTES));
  m->ring = h.mdp_ring;
  m->raw = dmalloc<uint8_t>(MdpSession::SLOTS * MdpSession::SLOT_BYTES, m->pool, m->alloc_stream);
  CQL_CUDA(cudaStreamSynchronize(m->alloc_stream));          // the buffers are used on the copy stream as well
  for (auto& e : m->slot_ev) CQL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CQL_CUDA(cudaEventCreateWithFlags(&m->ev_ts, cudaEventDisableTiming));
  CQL_CUDA(cudaEventCreateWithFlags(&m->ev_all, cudaEventDisableTiming));
  CQL_CUDA(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
}

void cql::mdp_append(Handle& h, int col, int dtype, const void* host, int64_t count) {
  CQL_REQUIRE(h.mdp != nullptr, "cql_mdp_append: call cql_mdp_begin first");
  NvtxRange nvtx("cql.mdp.append: host chunk -> pinned ring -> device");
  MdpSession& m = *h.mdp;
  CQL_REQUIRE(col >= 0 && col <= 4, "cql_mdp_append: column must be 0 user, 1 item, 2 timestamp, 3 relevance, 4 action noise");
  CQL_REQUIRE(dtype >= CQL_DT_I32 && dtype <= CQL_DT_F64, "cql_mdp_append: dtype must be one of CQL_DT_*");
  CQL_REQUIRE(count >= 0 && m.filled[col] + count <= m.n, "cql_mdp_append: more rows than cql_mdp_begin announced");
  CQL_REQUIRE(host != nullptr || count == 0, "cql_mdp_append: NULL chunk");
  CQL_REQUIRE(col != 2 || dtype == CQL_DT_I32 || dtype == CQL_DT_I64,
              "cql_mdp_append: timestamps must be int32 or int64 keys (convert float timestamps to an order-preserving key)");
  if (col == 4 && m.noise == nullptr) {
    m.noise = dmalloc<double>(m.n, m.pool, m.alloc_stream);
    CQL_CUDA(cudaStreamSynchronize(m.alloc_stream));
  }
  const int native = (col <= 1) ? CQL_DT_I32 : (col == 2 ? CQL_DT_I64 : CQL_DT_F64);
  const size_t eb = dtype_bytes(dtype);
  const int64_t per_slot = (int64_t)(MdpSession::SLOT_BYTES / eb);
  const uint8_t* src = (const uint8_t*)host;
  for (int64_t done = 0; done < count;) {
    const int64_t cnt = std::min(per_slot, count - done);
    const int slot = m.next_slot;
    m.next_slot = (m.next_slot + 1) % MdpSession::SLOTS;
    CQL_CUDA(cudaEventSynchronize(m.slot_ev[slot]));                        // the slot's previous copy (and conversion) is done
    uint8_t* pin = m.ring + (size_t)slot * MdpSession::SLOT_BYTES;
    parallel_memcpy(pin, src + (size_t)done * eb, (size_t)cnt * eb);
    const int64_t at = m.filled[col] + done;
    void* dst = col == 0 ? (void*)(m.user + at) : col == 1 ? (void*)(m.item + at) : col == 2 ? (void*)(m.ts + at)
              : col == 3 ? (void*)(m.rel + at) : (void*)(m.noise + at);
    if (dtype == native) {
      CQL_CUDA(cudaMemcpyAsync(dst, pin, (size_t)cnt * eb, cudaMemcpyHostToDevice, m.copy_stream));
    } else {
      uint8_t* rawd = m.raw + (size_t)slot * MdpSession::SLOT_BYTES;
      CQL_CUDA(cudaMemcpyAsync(rawd, pin, (size_t)cnt * eb, cudaMemcpyHostToDevice, m.copy_stream));
      if (col <= 1) convert_chunk<int32_t>(dtype, rawd, (int32_t*)dst, cnt, m.copy_stream);
      else if (col == 2) convert_chunk<int64_t>(dtype, rawd, (int64_t*)dst, cnt, m.copy_stream);
      else convert_chunk<double>(dtype, rawd, (double*)dst, cnt, m.copy_stream);
      m.launches += 1;
    }
    CQL_CUDA(cudaEventRecord(m.slot_ev[slot], m.copy_stream));
    done += cnt;
  }
  m.filled[col] += count;
  if (col == 2 && m.filled[2] == m.n && !m.stage_a) {                        // timestamps complete: sort while the rest uploads
    CQL_CUDA(cudaEventRecord(m.ev_ts, m.copy_stream));
    mdp_stage_a(h, m);
  }
}

// returns the number of kernels launched (for the handle's launch counter)
int64_t cql::mdp_finish(Handle& h, int top_k, float noise_scale, float* obs_out, float* act_out, float* rew_out, float* term_out,
                        int64_t* order_out) {
  CQL_REQUIRE(h.mdp != nullptr, "cql_mdp_finish: call cql_mdp_begin first");
  NvtxRange nvtx("cql.mdp.finish: radix sorts + replay table");
  std::unique_ptr<MdpSession> guard(h.mdp);
  h.mdp = nullptr;
  MdpSession& m = *guard;
  const int64_t n = m.n;
  for (int c = 0; c < 4; ++c) CQL_REQUIRE(m.filled[c] == n, "cql_mdp_finish: a column is incomplete (user, item, timestamp, relevance need n rows each)");
  CQL_REQUIRE(m.noise == nullptr || m.filled[4] == n, "cql_mdp_finish: the action-noise column is incomplete");
  cudaStream_t st = h.own_stream;
  if (!m.stage_a) { CQL_CUDA(cudaEventRecord(m.ev_ts, m.copy_stream)); mdp_stage_a(h, m); }
  CQL_CUDA(cudaEventRecord(m.ev_all, m.copy_stream));
  CQL_CUDA(cudaStreamWaitEvent(st, m.ev_all, 0));
  const unsigned nb = (unsigned)((n + 255) / 256);
  size_t tb;
  int64_t* head = m.k64a;            // reused after the timestamp sorts
  int64_t* gstart = m.k64b;
  // ---- order: (user, ts, input order): stable sort by user of the ts-ascending permutation
  k_gather<int32_t><<<nb, 256, 0, st>>>(m.user, m.ib, n, m.k32a);
  tb = m.tbytes; CQL_CUDA(cub::DeviceRadixSort::SortPairs(m.temp, tb, m.k32a, m.k32b, m.ib, m.order, (int)n, 0, 32, st));
  // ---- rank order: (user, rel desc, ts desc, input order)
  k_gather<double><<<nb, 256, 0, st>>>(m.rel, m.perm_desc, n, m.kda);
  tb = m.tbytes; CQL_CUDA(cub::DeviceRadixSort::SortPairsDescending(m.temp, tb, m.kda, m.kdb, m.perm_desc, m.ia, (int)n, 0, 64, st));
  k_gather<int32_t><<<nb, 256, 0, st>>>(m.user, m.ia, n, m.k32a);
  tb = m.tbytes; CQL_CUDA(cub::DeviceRadixSort::SortPairs(m.temp, tb, m.k32a, m.k32b, m.ia, m.ib, (int)n, 0, 32, st));   // ib = rank order
  k_heads<<<nb, 256, 0, st>>>(m.k32b, n, head);
  tb = m.tbytes; CQL_CUDA(cub::DeviceScan::InclusiveScan(m.temp, tb, head, gstart, MaxOp(), (int)n, st));
  k_rewarded<<<nb, 256, 0, st>>>(m.ib, gstart, n, top_k, m.rewarded);
  m.launches += 13;

  // ---- emit transition rows straight into the replay table (n_steps > 1: into session scratch, expanded from there)
  ensure_table(h, n);
  float4* rows = reinterpret_cast<float4*>(h.table);
  if (h.n_steps > 1) rows = dmalloc<float4>(2 * (size_t)n, m.pool, m.alloc_stream);
  float *d_obs = nullptr, *d_act = nullptr, *d_rew = nullptr, *d_term = nullptr;
  if (obs_out) {
    CQL_REQUIRE(act_out && rew_out && term_out, "cql_build_mdp: give all four output columns or none");
    d_obs = dmalloc<float>(2 * n, m.pool, m.alloc_stream); d_act = dmalloc<float>(n, m.pool, m.alloc_stream);
    d_rew = dmalloc<float>(n, m.pool, m.alloc_stream); d_term = dmalloc<float>(n, m.pool, m.alloc_stream);
  }
  k_emit<<<nb, 256, 0, st>>>(m.order, m.user, m.item, m.rel, m.noise, m.rewarded, n, noise_scale, h.cfg.seed,
                             rows, d_obs, d_act, d_rew, d_term);
  CQL_CUDA(cudaGetLastError());
  m.launches += 1;
  m.launches += table_stats(h, reinterpret_cast<const float*>(rows), n, true, st);
  if (h.n_steps > 1) {
    expand_n_steps(h, reinterpret_cast<const float*>(rows), n, st);
    m.launches += 1;
  }
  if (obs_out) {
    CQL_CUDA(cudaMemcpyAsync(obs_out, d_obs, 2 * n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaMemcpyAsync(act_out, d_act, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaMemcpyAsync(rew_out, d_rew, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaMemcpyAsync(term_out, d_term, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  }
  if (order_out) {
    std::vector<uint32_t> tmp((size_t)n);          // widen on the host: order is uint32 on the device
    CQL_CUDA(cudaMemcpyAsync(tmp.data(), m.order, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < n; ++i) order_out[i] = tmp[(size_t)i];
  }
  CQL_CUDA(cudaStreamSynchronize(st));
  // A NaN or infinite relevance (or action noise) gives a non-finite action, which would make every critic gradient
  // NaN.  The action column's statistics (table_stats above: count, mean, M2, min, max, copied to the pinned
  // stats_host before this synchronise) are finite exactly when every action is: no extra device work or copy.
  const double* act_stats = h.stats_host + 5 * 2;
  if (!(std::isfinite(act_stats[1]) && std::isfinite(act_stats[2]) && std::isfinite(act_stats[3]) && std::isfinite(act_stats[4]))) {
    h.stats = cql_table_stats{};                    // no table is left: ensure_table set n_trans = 0
    h.stats_pending = false;
    CQL_REQUIRE(false, "cql_mdp_finish: relevance column has a non-finite value (or the action noise has)");
  }
  h.n_trans = n;
  return m.launches;
}

// one-call form (cql_build_mdp): whole columns in the builder's own dtypes
int64_t mdp_build_on_device(Handle& h, const int32_t* user_h, const int32_t* item_h, const int64_t* ts_h, const double* rel_h,
                            const double* noise_h, int64_t n, int top_k, float noise_scale, float* obs_out, float* act_out,
                            float* rew_out, float* term_out, int64_t* order_out) {
  CQL_REQUIRE(user_h && item_h && ts_h && rel_h, "cql_build_mdp: NULL column");
  mdp_begin(h, n);
  try {
    mdp_append(h, 2, CQL_DT_I64, ts_h, n);          // timestamps first: their sorts overlap the other uploads
    mdp_append(h, 0, CQL_DT_I32, user_h, n);
    mdp_append(h, 1, CQL_DT_I32, item_h, n);
    mdp_append(h, 3, CQL_DT_F64, rel_h, n);
    if (noise_h) mdp_append(h, 4, CQL_DT_F64, noise_h, n);
    return mdp_finish(h, top_k, noise_scale, obs_out, act_out, rew_out, term_out, order_out);
  } catch (...) {
    if (h.mdp) { delete h.mdp; h.mdp = nullptr; }
    throw;
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Seen-items CSR of an interaction log, built on the device (the data the lazy seen filter of the scorer searches;
// reference: the joins inside `_filter_seen`, replay/models/base_rec.py:417-464).  Host: one 64-bit key per log row +
// an introsort of 2e7 keys + masks = 1.1 s for the ML-20M shape; here: two column uploads, one LSD radix sort over the
// significant bits, one unique pass, one emit pass.
namespace {
__global__ void k_seen_keys(const int32_t* __restrict__ user, const int32_t* __restrict__ item, const uint8_t* __restrict__ wanted,
                            int64_t n, int64_t n_users, unsigned long long* __restrict__ key) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t u = user[i];
  const bool keep = u >= 0 && u < n_users && item[i] >= 0 && (wanted == nullptr || wanted[u] != 0);
  key[i] = keep ? ((unsigned long long)u << 32) | (unsigned int)item[i] : (unsigned long long)n_users << 32;   // dropped rows sort last
}
// unique, sorted keys -> seen items + CSR row pointers (a thread fills the pointers of the users between its
// predecessor's user and its own: users without rows get empty ranges)
__global__ void k_seen_emit(const unsigned long long* __restrict__ key, int64_t num, int64_t n_users,
                            int32_t* __restrict__ seen, int64_t* __restrict__ indptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  const int64_t u = (int64_t)(key[i] >> 32), prev = i == 0 ? -1 : (int64_t)(key[i - 1] >> 32);
  if (u < n_users) seen[i] = (int32_t)(key[i] & 0xffffffffull);
  for (int64_t x = prev + 1; x <= (u < n_users ? u : n_users); ++x) indptr[x] = i;
  if (i == num - 1 && u < n_users)
    for (int64_t x = u + 1; x <= n_users; ++x) indptr[x] = num;
}
}  // namespace

int64_t cql::seen_csr_on_device(Handle& h, const int32_t* users_h, const int32_t* items_h, int64_t n, int64_t n_users,
                                const uint8_t* wanted_h, int64_t* indptr_d, int32_t* seen_d, cudaStream_t st) {
  CQL_REQUIRE(n >= 0 && n_users >= 1 && n_users < (1ll << 31), "cql_seen_csr: bad sizes");
  CQL_REQUIRE(indptr_d != nullptr && (n == 0 || (users_h && items_h && seen_d)), "cql_seen_csr: NULL pointer");
  if (n == 0) {
    CQL_CUDA(cudaMemsetAsync(indptr_d, 0, (size_t)(n_users + 1) * sizeof(int64_t), st));
    CQL_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  DevTmp tmp(st);
  int32_t* u_d = tmp.get<int32_t>(n);
  int32_t* i_d = tmp.get<int32_t>(n);
  unsigned long long* k0 = tmp.get<unsigned long long>(n);
  unsigned long long* k1 = tmp.get<unsigned long long>(n);
  int64_t* num_d = tmp.get<int64_t>(1);
  uint8_t* w_d = nullptr;
  CQL_CUDA(cudaMemcpyAsync(u_d, users_h, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  CQL_CUDA(cudaMemcpyAsync(i_d, items_h, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  if (wanted_h) {
    w_d = tmp.get<uint8_t>(n_users);
    CQL_CUDA(cudaMemcpyAsync(w_d, wanted_h, (size_t)n_users, cudaMemcpyHostToDevice, st));
  }
  const unsigned blocks = (unsigned)((n + 255) / 256);
  k_seen_keys<<<blocks, 256, 0, st>>>(u_d, i_d, w_d, n, n_users, k0);
  int ubits = 1;
  while ((1ll << ubits) <= n_users) ++ubits;                    // user ids 0 .. n_users (n_users = the dropped rows)
  size_t sort_bytes = 0, uniq_bytes = 0;
  CQL_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, k0, k1, n, 0, 32 + ubits, st));
  CQL_CUDA(cub::DeviceSelect::Unique(nullptr, uniq_bytes, k1, k0, num_d, n, st));
  uint8_t* cub_tmp = tmp.get<uint8_t>(std::max(sort_bytes, uniq_bytes) + 16);
  CQL_CUDA(cub::DeviceRadixSort::SortKeys(cub_tmp, sort_bytes, k0, k1, n, 0, 32 + ubits, st));
  CQL_CUDA(cub::DeviceSelect::Unique(cub_tmp, uniq_bytes, k1, k0, num_d, n, st));
  int64_t num = 0;
  CQL_CUDA(cudaMemcpyAsync(&num, num_d, sizeof(num), cudaMemcpyDeviceToHost, st));
  CQL_CUDA(cudaStreamSynchronize(st));
  k_seen_emit<<<(unsigned)((num + 255) / 256), 256, 0, st>>>(k0, num, n_users, seen_d, indptr_d);
  int64_t n_seen = 0;
  CQL_CUDA(cudaMemcpyAsync(&n_seen, indptr_d + n_users, sizeof(n_seen), cudaMemcpyDeviceToHost, st));
  CQL_CUDA(cudaStreamSynchronize(st));
  CQL_CUDA(cudaGetLastError());
  return n_seen;
}
