// engine.cuh -- the per-GPU handle: configuration, HBM-resident state, scratch.
#pragma once
#include <algorithm>
#include <cstdlib>
#include <vector>
#include <string>
#include "common.cuh"
#include "mlp_simt.cuh"
#include "dp_peer.cuh"
#include <nvtx3/nvToolsExt.h>

namespace cql {

constexpr int N_NOISE_PARTS = 8;

struct StepInfo {          // written by k_step_begin, read by the Adam kernels
  double bc1, bc2_sqrt;    // 1 - beta1^t, sqrt(1 - beta2^t)
  long long step;          // t (1-based) of the update in flight
};

// NVTX range (SURVEY.md section 5 "Tracing / profiling"): the phases of an update, scoring and ingestion show up by name
// on an Nsight Systems / ncu --nvtx timeline.  Header-only NVTX3: a no-op unless a tool is attached.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

// d3rlpy's scalers as the kernels apply them (cql_set_preprocessing, DESIGN.md section 1): x' = (x - off) / den with
// den = max - min or std + 1e-3 already rounded on the host; every operation rounded separately (no FMA contraction).
// on == 0: the value passes untouched.  Passed by value: a change destroys the captured graphs.
struct Affine {
  int on;
  float off, den;
};
struct Prep {
  Affine obs[2];   // user, item
  Affine act;      // min_max: off = min, den = max - min; forward maps onto [-1, 1]
  Affine rew;
  __host__ __device__ bool any() const { return obs[0].on | obs[1].on | act.on | rew.on; }
};
__device__ __forceinline__ float prep_fwd(const Affine& p, float x) {
  return p.on ? __fdiv_rn(__fsub_rn(x, p.off), p.den) : x;
}
__device__ __forceinline__ float act_fwd(const Affine& p, float a) {
  return p.on ? __fsub_rn(__fmul_rn(__fdiv_rn(__fsub_rn(a, p.off), p.den), 2.f), 1.f) : a;
}
__device__ __forceinline__ float act_rev(const Affine& p, float a) {
  return p.on ? __fadd_rn(__fmul_rn(__fdiv_rn(__fadd_rn(a, 1.f), 2.f), p.den), p.off) : a;
}
// transition row (s.x s.y a r | s'.x s'.y term discount) in the network's coordinates; term and discount untouched
__device__ __forceinline__ float4 prep_row0(const Prep& p, float4 r) {
  return make_float4(prep_fwd(p.obs[0], r.x), prep_fwd(p.obs[1], r.y), act_fwd(p.act, r.z), prep_fwd(p.rew, r.w));
}
__device__ __forceinline__ float4 prep_row1(const Prep& p, float4 r) {
  return make_float4(prep_fwd(p.obs[0], r.x), prep_fwd(p.obs[1], r.y), r.z, r.w);
}

constexpr int STATS_MAX_BLOCKS = 1024;                               // table_stats (update.cuh)
constexpr size_t STATS_DEV_DOUBLES = (STATS_MAX_BLOCKS + 1) * 4 * 5;

// A/B switches of the update schedule, read from the environment once per process.  Each selects the path a measurement
// in DESIGN.md compared against; unset, the library runs its default schedule.
struct Switches {
  int skip;                   // CQL_SKIP=<mask>: leave the launches with these bits out (timing experiments; results wrong)
  bool no_pdl;                // CQL_NO_PDL: no programmatic dependent launch
  bool no_pair;               // CQL_NO_PAIR: no CTA-pair kernels (forward, bwd1, bwd2)
  bool no_pair_bwd1;          // CQL_NO_PAIR_BWD1: no CTA-pair bwd1
  bool no_pair_bwd2;          // CQL_NO_PAIR_BWD2: no CTA-pair bwd2
  bool no_pair_bwd2_small;    // CQL_NO_PAIR_BWD2_SMALL: the small (actor) bwd2 on one-CTA kernels
  bool no_small;              // CQL_NO_SMALL: no 32-column work items for the small f16x3 launches
  bool no_fold;               // CQL_NO_FOLD: separate gradient reduction launch instead of k_adam_pack summing the partials
  bool no_fused_adam;         // CQL_NO_FUSED_ADAM: k_adam_polyak + pack kernels instead of k_adam_pack (implies CQL_NO_FOLD)
  bool no_fork;               // CQL_NO_FORK: bwd1 and bwd2 of a job back to back on one stream
  int big_fork;               // CQL_BIG_FORK=<pairs>: CTA pairs of the big forked bwd1 (0 = serial); -1 = default
  int h2_cost;                // CQL_H2_COST=<cost>: f16x3 forward's relative cost of an item that stores H2 (0 = default)
  int pair_swap;              // CQL_PAIR_SWAP=<rank>: cluster rank holding the first half of the CTA-pair operand rows
  int dp_debug;               // CQL_DP_DEBUG=<mask>: data-parallel exchange timing experiments (dp_peer.cuh; results wrong)
  bool no_fused_dp;           // CQL_NO_FUSED_DP: data-parallel gradient exchange by cql_dp_allreduce, not inside the kernels
};
inline const Switches& switches() {
  static const Switches s = [] {
    auto set = [](const char* name) { return std::getenv(name) != nullptr; };
    auto num = [](const char* name, int unset) { const char* v = std::getenv(name); return v ? std::atoi(v) : unset; };
    Switches w{};
    w.skip = num("CQL_SKIP", 0);
    w.no_pdl = set("CQL_NO_PDL");
    w.no_pair = set("CQL_NO_PAIR");
    w.no_pair_bwd1 = set("CQL_NO_PAIR_BWD1");
    w.no_pair_bwd2 = set("CQL_NO_PAIR_BWD2");
    w.no_pair_bwd2_small = set("CQL_NO_PAIR_BWD2_SMALL");
    w.no_small = set("CQL_NO_SMALL");
    w.no_fold = set("CQL_NO_FOLD");
    w.no_fused_adam = set("CQL_NO_FUSED_ADAM");
    w.no_fork = set("CQL_NO_FORK");
    w.big_fork = num("CQL_BIG_FORK", -1);
    w.h2_cost = num("CQL_H2_COST", 0);
    w.pair_swap = num("CQL_PAIR_SWAP", 0);
    w.dp_debug = num("CQL_DP_DEBUG", 0);
    w.no_fused_dp = set("CQL_NO_FUSED_DP");
    return w;
  }();
  return s;
}

struct MdpSession;                   // chunked ingestion session (mdp_gpu.cu)
// seen-items CSR of a log on the device (mdp_gpu.cu); returns the number of (user, item) entries written
int64_t seen_csr_on_device(struct Handle& h, const int32_t* users_h, const int32_t* items_h, int64_t n, int64_t n_users,
                           const uint8_t* wanted_h, int64_t* indptr_d, int32_t* seen_d, cudaStream_t st);
void mdp_session_free(MdpSession*);

struct Handle {
  cql_config cfg{};
  std::string err;
  cudaStream_t own_stream = nullptr;
  cudaStream_t side_stream = nullptr;            // fork/join branch for independent small launches (captured into the graphs)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int num_sms = 148;
  int64_t launches = 0;

  // ---- learner state (flat layout, see common.cuh) ----
  float* params = nullptr;   // state_floats(C)
  float* adam_m = nullptr;   // same layout (trainable part used)
  float* adam_v = nullptr;
  float* grads = nullptr;    // grad_floats(C): [actor | critics | scalars]
  long long* step_dev = nullptr;   // completed updates
  StepInfo* stepinfo = nullptr;
  float* metrics = nullptr;  // 8 floats: temp_loss,temp,alpha_loss,alpha,critic_loss,actor_loss,td_loss,-
  float* metrics_host = nullptr;   // pinned

  // ---- replay table ----
  float* table = nullptr;    // [n_trans][8]: obs.x obs.y act rew nobs.x nobs.y term discount (0 when n_steps == 1)
  int64_t n_trans = 0;
  int n_steps = 1;           // TD horizon of the tables built from now on and of the TD target (cql_set_n_steps)
  int64_t table_cap = 0;     // rows the table allocation can hold (re-ingesting a log of the same size re-uses it)
  bool table_sharded = false;   // data parallel: this rank holds only its own users' episodes (cql_set_table_sharded)
  int64_t sample_pos_host = 0;  // position in the epoch stream for the stand-alone sampler
  long long* sample_pos = nullptr;   // device: next position in the permutation stream
  cql_table_stats stats{};   // column statistics of the table's one-step rows (table_stats; filled from stats_host)
  double* stats_dev = nullptr;    // [STATS_DEV_DOUBLES] k_stats_partial / k_stats_final partials and result
  double* stats_host = nullptr;   // pinned [4][5]: the result (count, mean, m2, min, max per column), copied async
  bool stats_pending = false;     // stats_host holds the current table's statistics, not yet moved into `stats`
  bool stats_rew_ok = false;
  cql_preprocessing prep_cfg{};   // as given to cql_set_preprocessing
  Prep prep{};               // ... as the kernels apply it

  // ---- per-step scratch (B = batch, n = action samples, C = critics) ----
  int B = 0, n = 0, C = 0;
  int rsA = 0, rsC = 0;      // rows per batch element: alpha job (3n), critic job (3n+1)
  float* batch = nullptr;    // [B][8] sampled transition rows (same row format as table)
  float* batch_host = nullptr;   // pinned staging for cql_update_batch
  float* batch_in = nullptr;     // [B][8] the provided / k_sample minibatch as staged, when preprocessing is on
                                 // (k_actor_rows writes its scaled rows to `batch`; the staged rows stay raw)
  float* noise = nullptr;    // packed, see header
  float* noise_host = nullptr;
  int64_t noise_floats = 0;
  float4* XA = nullptr;      // [2B] actor inputs: s rows then s' rows
  float* outA = nullptr;     // [2B][2] mu, raw logstd
  float* h2A = nullptr;      // [tiles(B)][256][64] actor H2 of the s rows
  float4* XAl = nullptr;     // [B*rsA] alpha-step critic rows
  float* offAl = nullptr;    // [B*rsA] log-prob offsets
  float* QAl = nullptr;      // [C][B*rsA]
  float4* XC = nullptr;      // [B*rsC] critic-step rows (3n samples + data row)
  float* offC = nullptr;     // [B*rsC]
  float* QC = nullptr;       // [C][B*rsC]
  float* h2C = nullptr;      // [C][tiles][256][64]
  float* dQ = nullptr;       // [C][B*rsC]
  float4* XT = nullptr;      // [B] target rows (s', tanh(mu(s')))
  float* QT = nullptr;       // [C][B]
  float4* XP = nullptr;      // [B] actor-step rows (s, a_pi)
  float* QP = nullptr;       // [C][B]
  float* h2P = nullptr;      // [C][tiles(B)][256][64]
  float* dQP = nullptr;      // [C][B]
  float4* dXP = nullptr;     // [C][B]
  float* dOutA = nullptr;    // [B][2]
  float* perb = nullptr;     // [B][4]: temp term, logp_pi, a_pi raw, -
  float* pairv = nullptr;    // [C][B] PairVals {lse_alpha, lse_critic, q_data, td_err}
  float* loss_sums = nullptr;  // [16] reduced sums / conservative coefficient; [14], [15] = block tickets (k_actor_dout, k_lse)
  float* actor_part = nullptr; // [ceil(B / 128) * 4] warp sums of the actor-loss metric (k_actor_dout)
  float* smallC = nullptr;   // [C][tilesC][SMALL_STRIDE]
  float* smallA = nullptr;   // [tilesB][SMALL_STRIDE]
  float* pw2C = nullptr;     // [C][splitsC][H*H]
  float* pw2A = nullptr;     // [splitsA][H*H]
  int splitsC = 1, splitsA = 1;

  // ---- tensor-core path (precision != FP32): packed W2 per slot, layer-3 partial sums ----
  uint8_t* packed_fwd = nullptr;   // [(2+2C) slots][PACKED_NET_BYTES]  B[n][k] = W2[n][k]
  size_t packed_net_bytes = 0;     // stride of packed_fwd
  size_t packed_net_bytes_bwd = 0; // stride of packed_bwd
  float* part = nullptr;           // scratch for [n_nets][SLICES][rows][OUT] partials
  size_t part_floats = 0;
  uint8_t* packed_bwd = nullptr;   // [(1+C) slots: actor, critics][PACKED_NET_BYTES]  B[n][k] = W2[k][n]
  float* small1 = nullptr;         // [C][slots1][SMALL_STRIDE] bwd1 partials (W1 | b1), slots1 = 4 * num_sms
  float* small2 = nullptr;         // [C][splits_tc][SMALL_STRIDE] bwd2 partials (b2 | W3 | b3)
  float* pw2_tc = nullptr;         // [C][splits_tc][H*H]
  float4* dX_part = nullptr;       // [C*SLICES][B]
  int slots1 = 0, splits_tc = 0, tc_slices = 1;
  // CTA-pair (cta_group::2) f16x3 kernels: W2 of every slot in the pair layout (mlp_tc_h2.cuh)
  uint8_t* packed_fwd2 = nullptr;  // [(2+2C) slots][H2Cfg::PACKED_NET_BYTES]  B[n][k] = W2[n][k]
  uint8_t* packed_bwd2 = nullptr;  // [(1+C) slots]                           B[n][k] = W2[k][n]
  size_t packed_net_bytes2 = 0;
  DpPeer dp;                       // data-parallel peers (cql_dp_attach); world <= 1: single GPU
  bool dp_fused = false;           // the gradient exchange happens INSIDE the update kernels (f16x3 path, dp_peer.cuh)
  int* w2max = nullptr;            // [(2+2C) slots][4]: rotating max|W2| slots of the fused Adam + pack kernel (adam_pack.cuh)
  int* ap_wmax = nullptr;          // k_adam_pack's layer maxima across its small-tensor CTAs + tickets (AdamPackJobs::wmax_acc)
  int pair_swap_b = 0;             // which cluster rank holds the first half of the operand rows (probed at create)

  // optional event marks for cql_timed_update
  bool timing = false;
  bool pdl_off = false;            // cql_timed_update: launches without PDL, so the events separate their kernels' durations
  cudaEvent_t ev[16] = {};

  MdpSession* mdp = nullptr;       // between cql_mdp_begin and cql_mdp_finish
  uint8_t* mdp_ring = nullptr;     // pinned staging ring of the ingestion sessions
  std::vector<void*> allocs;

  template <typename T>
  T* dalloc(size_t count) {
    void* p = nullptr;
    CQL_CUDA(cudaMalloc(&p, count * sizeof(T)));
    CQL_CUDA(cudaMemset(p, 0, count * sizeof(T)));
    allocs.push_back(p);
    return reinterpret_cast<T*>(p);
  }
  void free_all() {
    for (void* p : allocs) cudaFree(p);
    allocs.clear();
    if (mdp) { mdp_session_free(mdp); mdp = nullptr; }
    if (mdp_ring) { cudaFreeHost(mdp_ring); mdp_ring = nullptr; }
    if (table) { cudaFree(table); table = nullptr; table_cap = 0; }
    if (metrics_host) { cudaFreeHost(metrics_host); metrics_host = nullptr; }
    if (batch_host) { cudaFreeHost(batch_host); batch_host = nullptr; }
    if (stats_host) { cudaFreeHost(stats_host); stats_host = nullptr; }
    if (noise_host) { cudaFreeHost(noise_host); noise_host = nullptr; }
    if (own_stream) { cudaStreamDestroy(own_stream); own_stream = nullptr; }
    if (side_stream) { cudaStreamDestroy(side_stream); side_stream = nullptr; }
    if (ev_fork) { cudaEventDestroy(ev_fork); ev_fork = nullptr; }
    if (ev_join) { cudaEventDestroy(ev_join); ev_join = nullptr; }
    for (auto& e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
  }

  // where a minibatch is staged before k_actor_rows: `batch` itself without preprocessing, else batch_in (the captured
  // graphs bake this address in; cql_set_preprocessing destroys them)
  float* staged_batch() const { return prep.any() ? batch_in : batch; }
  float* net_params(int slot) const { return params + (size_t)slot * NET_STRIDE; }
  float* scalars() const { return params + scalars_off(C); }
  // grads buffer parts
  float* g_actor() const { return grads; }
  float* g_critics() const { return grads + NET_STRIDE; }
  float* g_scalars() const { return grads + (size_t)(1 + C) * NET_STRIDE; }
};

void mdp_begin(Handle& h, int64_t n);
void mdp_append(Handle& h, int col, int dtype, const void* host, int64_t count);
int64_t mdp_finish(Handle& h, int top_k, float noise_scale, float* obs_out, float* act_out, float* rew_out, float* term_out,
                   int64_t* order_out);

// replay table for n rows: the existing allocation is kept when it is large enough (a 640 MB cudaFree + cudaMalloc per
// ingestion synchronises the device and costs milliseconds to tens of milliseconds)
inline void ensure_table(Handle& h, int64_t n) {
  h.n_trans = 0;
  h.stats = cql_table_stats{};
  h.stats_pending = false;
  if (h.table != nullptr && h.table_cap >= n) return;
  if (h.table) { CQL_CUDA(cudaFree(h.table)); h.table = nullptr; h.table_cap = 0; }
  CQL_CUDA(cudaMalloc(&h.table, (size_t)n * 8 * sizeof(float)));
  h.table_cap = n;
}

// n_steps > 1: one-step rows (device [n][8], not h.table) -> n-step rows in h.table, on `st` (capi.cu)
void expand_n_steps(Handle& h, const float* one_step, int64_t n, cudaStream_t st);
// column statistics of one-step rows (device [n][8]), enqueued on `st` into the handle's buffers (no allocation, no
// synchronisation; cql_get_table_stats reads them).  rew_ok = false: the reward slot holds n-step returns, the reward
// statistics are marked unavailable.  Returns the launches it made (capi.cu).
int table_stats(Handle& h, const float* rows, int64_t n, bool rew_ok, cudaStream_t st);

// Call scratch comes from the stream-ordered pool (cudaMallocAsync), which keeps up to 4 GB cached between calls:
// the ~1.9 GB of cudaMalloc / cudaFree pairs per 20 M-row ingestion session synchronise the device and made ingestion
// (and `fit`) wall clocks erratic on shared hosts -- 0.05 .. 1.2 s for the same call (r02 bench lines).
inline void keep_pool_cached() {
  static unsigned long long done_mask = 0;          // per device (engines on several GPUs may live in one process)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || (done_mask >> dev) & 1ull) return;
  done_mask |= 1ull << dev;
  cudaMemPool_t mp = nullptr;
  unsigned long long keep = 4ull << 30;
  if (cudaDeviceGetDefaultMemPool(&mp, dev) == cudaSuccess)
    cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
}

// device scratch from the stream-ordered pool, released on every exit path: cudaMalloc / cudaFree pairs per call
// synchronise the device and made `predict` wall clocks erratic (0.05 .. 1.4 s for the same ML-1M call)
struct DevTmp {
  cudaStream_t st;
  std::vector<void*> p;
  explicit DevTmp(cudaStream_t s) : st(s) { keep_pool_cached(); }
  ~DevTmp() { for (void* x : p) cudaFreeAsync(x, st); }
  DevTmp(const DevTmp&) = delete;
  DevTmp& operator=(const DevTmp&) = delete;
  template <typename T>
  T* get(size_t count) {
    void* q = nullptr;
    CQL_CUDA(cudaMallocAsync(&q, std::max<size_t>(1, count) * sizeof(T), st));
    p.push_back(q);
    return (T*)q;
  }
};

inline void mark(Handle* h, cudaStream_t st, int i) {
  if (h->timing) CQL_CUDA(cudaEventRecord(h->ev[i], st));
}

inline cudaStream_t pick_stream(Handle* h, void* stream) {
  return stream ? reinterpret_cast<cudaStream_t>(stream) : h->own_stream;
}

#define CQL_LAUNCH_CHECK(h)                 \
  do {                                      \
    (h)->launches++;                        \
    CQL_CUDA(cudaGetLastError());           \
  } while (0)

}  // namespace cql
