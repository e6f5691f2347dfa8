// capi.cu -- the extern "C" surface declared in include/cql_b200.h.
#include <cmath>
#include <cstring>
#include <cstdio>
#include <algorithm>
#include "engine.cuh"
#include "update.cuh"
#include "score.cuh"
#include "tc_selftest.cuh"
#include "score_tc.cuh"
#include "score_tc_h.cuh"
#include "topk_staged.cuh"
#include "metrics.cuh"
#include "dp_peer.cuh"
#include "mma_bench.cuh"
#include "offline_eval.cuh"

using namespace cql;

// A CUDA graph of one update, captured from an enqueue function on first use and again when the stream changes.  A
// replay counts the launches the capture made.
struct StepGraph {
  cudaGraphExec_t exec = nullptr;
  cudaStream_t stream = nullptr;
  int64_t launches = 0;

  void reset() {
    if (exec) cudaGraphExecDestroy(exec);
    exec = nullptr;
  }
  // capture `enqueue` if needed, then replay the graph n times on st
  template <typename F>
  void run(Handle& h, cudaStream_t st, int64_t n, F&& enqueue) {
    if (!exec || stream != st) {
      reset();
      cudaGraph_t g = nullptr;
      const int64_t before = h.launches;
      CQL_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      try {
        enqueue();
      } catch (...) {
        cudaStreamEndCapture(st, &g);
        if (g) cudaGraphDestroy(g);
        throw;
      }
      CQL_CUDA(cudaStreamEndCapture(st, &g));
      launches = h.launches - before;
      h.launches = before;
      CQL_CUDA(cudaGraphInstantiate(&exec, g, 0));
      CQL_CUDA(cudaGraphDestroy(g));
      stream = st;
    }
    for (int64_t i = 0; i < n; ++i) CQL_CUDA(cudaGraphLaunch(exec, st));
    h.launches += launches * n;
  }
};

struct cql_handle {
  Handle h;
  StepGraph update_graph;            // one sampled update (phases 0-3): cql_update
  StepGraph batch_graph[2];          // the host-minibatch entry (cql_update_batch): [0] Philox noise, [1] caller-provided noise
  // grow-only device scratch for the host-pointer scoring entry points
  void* sbuf[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  size_t sbuf_bytes[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  float* part_s = nullptr;
  int* part_i = nullptr;
  size_t part_elems = 0;
  uint8_t* packed_score = nullptr;   // tf32-packed W2 of actor + critics for the tensor-core scorer
  // cql_update_batches: the bare step (minibatch already on the device) as a graph, pinned staging ring, metrics rows
  StepGraph step_graph;
  float* ring = nullptr;             // pinned [8][B*8]
  cudaEvent_t ring_ev[8] = {};
  float* metrics_rows = nullptr;     // pinned [metrics_rows_cap][8]
  int64_t metrics_rows_cap = 0;
  // ... and its copy pipeline: a second stream moves minibatch i + 1 host -> device ring and the metrics of step i - 1
  // device -> host while step i computes
  cudaStream_t copy_stream = nullptr, copy_stream_out = nullptr;      // one per direction: neither queues behind the other
  float* dev_ring = nullptr;         // device [8][B*8]
  float* dev_metrics = nullptr;      // device [8][8]
  cudaEvent_t ev_used[8] = {};       // compute stream: slot's minibatch has been copied into h.batch
  cudaEvent_t ev_met[8] = {};        // compute stream: slot's metrics are in dev_metrics
  cudaEvent_t ev_met_out[8] = {};    // copy stream: slot's metrics have left dev_metrics
  void* dp_local = nullptr;          // epochs | tickets | error flag
};

static thread_local std::string g_create_error;

// mdp_gpu.cu
int64_t mdp_build_on_device(Handle& h, const int32_t* user_h, const int32_t* item_h, const int64_t* ts_h, const double* rel_h,
                            const double* noise_h, int64_t n, int top_k, float noise_scale, float* obs_out, float* act_out,
                            float* rew_out, float* term_out, int64_t* order_out);

namespace {

void* scratch(cql_handle* ch, int slot, size_t bytes) {
  if (bytes > ch->sbuf_bytes[slot]) {
    if (ch->sbuf[slot]) CQL_CUDA(cudaFree(ch->sbuf[slot]));
    ch->sbuf[slot] = nullptr;
    ch->sbuf_bytes[slot] = 0;
    const size_t cap = bytes + bytes / 4 + 256;
    CQL_CUDA(cudaMalloc(&ch->sbuf[slot], cap));
    ch->sbuf_bytes[slot] = cap;
  }
  return ch->sbuf[slot];
}

void set_kernel_attrs() {
  CQL_CUDA(cudaFuncSetAttribute(mlp_fwd_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(mlp_fwd_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(mlp_bwd1_kernel<3, 1, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD1_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(mlp_bwd1_kernel<3, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD1_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(mlp_bwd1_kernel<2, 2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD1_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(mlp_bwd2_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD2_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(mlp_bwd2_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD2_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(k_score_topk, cudaFuncAttributeMaxDynamicSharedMemorySize, score_smem(CQL_MAX_TOPK)));
  CQL_CUDA(cudaFuncSetAttribute(k_score_pairs, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(k_topk_filter_staged, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TKS_SMEM));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_kernel<false, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::FwdSmem<false, tc::FWD_NPW>::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_kernel<false, 3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::FwdSmem<false, tc::FWD_NPW>::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::ScoreSmem::bytes(CQL_MAX_TOPK)));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_score_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::ScoreSmemH::bytes(CQL_MAX_TOPK)));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_h_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2HCfg::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_h_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2HCfg::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_h2_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2PCfg::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_h2_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2PCfg::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_h_kernel<3, 1, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_h_kernel<3, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_h_kernel<2, 2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_h_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_h_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute((tc::tc_fwd_h_kernel<3, 1, tc::HCfgS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfgS::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute((tc::tc_fwd_h_kernel<2, 2, tc::HCfgS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfgS::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute((tc::tc_bwd1_h_kernel<3, 1, true, false, tc::HCfgS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfgS::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute((tc::tc_bwd1_h_kernel<3, 1, false, true, tc::HCfgS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfgS::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute((tc::tc_bwd1_h_kernel<2, 2, true, false, tc::HCfgS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::HCfgS::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_h2_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::H2Cfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_h2_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::H2Cfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_h2_kernel<3, 1, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::H2B1Cfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_h2_kernel<3, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::H2B1Cfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_h2_kernel<2, 2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::H2B1Cfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_ts_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::TsCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_fwd_ts_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::TsCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_ts_kernel<3, 1, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::TsCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_ts_kernel<3, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::TsCfg::SMEM_BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_ts_kernel<2, 2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::TsCfg::SMEM_BYTES));
  const int f0 = (int)tc::FwdSmem<false, tc::BWD1_NPW>::BYTES;
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_kernel<false, 3, 1, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, f0));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_kernel<false, 3, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, f0));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd1_kernel<false, 2, 2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, f0));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_kernel<true, 3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2Cfg<true>::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_kernel<true, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2Cfg<true>::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_kernel<false, 3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2Cfg<false>::BYTES));
  CQL_CUDA(cudaFuncSetAttribute(tc::tc_bwd2_kernel<false, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::B2Cfg<false>::BYTES));
}

void create_impl(const cql_config* cfg, cql_handle* ch) {
  Handle& h = ch->h;
  CQL_REQUIRE(cfg != nullptr, "cql_create: cfg is NULL");
  CQL_REQUIRE(cfg->struct_size == (int32_t)sizeof(cql_config), "cql_create: cql_config size mismatch (ABI)");
  CQL_REQUIRE(cfg->batch_size >= 1 && cfg->batch_size <= (1 << 20), "cql_create: batch_size out of range");
  CQL_REQUIRE(cfg->n_critics >= 1 && cfg->n_critics <= CQL_MAX_CRITICS, "cql_create: n_critics must be 1..4");
  CQL_REQUIRE(cfg->n_action_samples >= 1 && cfg->n_action_samples <= 10, "cql_create: n_action_samples must be 1..10");
  CQL_REQUIRE(cfg->precision == CQL_PREC_FP32 || cfg->precision == CQL_PREC_TF32X3 || cfg->precision == CQL_PREC_BF16 ||
                  cfg->precision == CQL_PREC_F16X3,
              "cql_create: bad precision");
  CQL_REQUIRE(cfg->squash == CQL_SQUASH_EPS || cfg->squash == CQL_SQUASH_SOFTPLUS, "cql_create: bad squash");
  CQL_REQUIRE(cfg->world_size >= 1 && cfg->rank >= 0 && cfg->rank < cfg->world_size, "cql_create: bad rank/world_size");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    throw Error{std::string("cql_create: no CUDA device available (") + cudaGetErrorString(e) +
                "); this library has no CPU fallback"};
  CQL_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "cql_create: device ordinal out of range");
  CQL_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop{};
  CQL_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  CQL_REQUIRE(prop.major >= 10, "cql_create: built for sm_100a (B200); found an older GPU");
  h.cfg = *cfg;
  h.num_sms = prop.multiProcessorCount;
  h.B = cfg->batch_size; h.n = cfg->n_action_samples; h.C = cfg->n_critics;
  const int B = h.B, n = h.n, C = h.C, n3 = 3 * n;
  h.rsA = n3; h.rsC = n3 + 1;
  CQL_CUDA(cudaStreamCreateWithFlags(&h.own_stream, cudaStreamNonBlocking));
  CQL_CUDA(cudaStreamCreateWithFlags(&h.side_stream, cudaStreamNonBlocking));
  CQL_CUDA(cudaEventCreateWithFlags(&h.ev_fork, cudaEventDisableTiming));
  CQL_CUDA(cudaEventCreateWithFlags(&h.ev_join, cudaEventDisableTiming));
  set_kernel_attrs();

  const int64_t S = state_floats(C);
  h.params = h.dalloc<float>(S);
  h.adam_m = h.dalloc<float>(S);
  h.adam_v = h.dalloc<float>(S);
  h.grads = h.dalloc<float>(grad_floats(C));
  h.step_dev = h.dalloc<long long>(1);
  h.sample_pos = h.dalloc<long long>(1);
  h.stepinfo = h.dalloc<StepInfo>(1);
  h.metrics = h.dalloc<float>(8);
  h.stats_dev = h.dalloc<double>(STATS_DEV_DOUBLES);
  CQL_CUDA(cudaMallocHost(&h.stats_host, 4 * 5 * sizeof(double)));
  CQL_CUDA(cudaMallocHost(&h.metrics_host, 8 * sizeof(float)));
  h.batch = h.dalloc<float>((size_t)B * 8);
  h.batch_in = h.dalloc<float>((size_t)B * 8);
  CQL_CUDA(cudaMallocHost(&h.batch_host, (size_t)B * 8 * sizeof(float)));
  h.noise_floats = 2 * (int64_t)B + 6 * (int64_t)B * n;
  h.noise = h.dalloc<float>(h.noise_floats);
  CQL_CUDA(cudaMallocHost(&h.noise_host, h.noise_floats * sizeof(float)));
  const int tB = tiles_of(B), rowsC = B * (n3 + 1), tC = tiles_of(rowsC);
  h.XA = h.dalloc<float4>(2 * (size_t)B);
  h.outA = h.dalloc<float>(4 * (size_t)B);
  h.h2A = h.dalloc<float>((size_t)tB * H * BM);
  h.XAl = h.dalloc<float4>((size_t)B * n3);
  h.offAl = h.dalloc<float>((size_t)B * n3);
  h.QAl = h.dalloc<float>((size_t)C * B * n3);
  h.XC = h.dalloc<float4>((size_t)rowsC);
  h.offC = h.dalloc<float>((size_t)rowsC);
  h.QC = h.dalloc<float>((size_t)C * rowsC);
  h.h2C = h.dalloc<float>((size_t)C * tC * H * BM);
  h.dQ = h.dalloc<float>((size_t)C * rowsC);
  h.XT = h.dalloc<float4>(B);
  h.QT = h.dalloc<float>((size_t)C * B);
  h.XP = h.dalloc<float4>(B);
  h.QP = h.dalloc<float>((size_t)C * B);
  h.h2P = h.dalloc<float>((size_t)C * tB * H * BM);
  h.dQP = h.dalloc<float>((size_t)C * B);
  h.dXP = h.dalloc<float4>((size_t)C * B);
  h.dOutA = h.dalloc<float>(2 * (size_t)B);
  h.perb = h.dalloc<float>(4 * (size_t)B);
  h.pairv = h.dalloc<float>(4 * (size_t)C * B);
  h.loss_sums = h.dalloc<float>(16);
  h.actor_part = h.dalloc<float>((size_t)((B + 127) / 128) * 4 + 4);
  h.splitsC = std::max(1, std::min(tC, (2 * h.num_sms) / (4 * C)));
  h.splitsA = std::max(1, std::min(tB, (2 * h.num_sms) / 4));
  h.smallC = h.dalloc<float>((size_t)C * tC * SMALL_STRIDE);
  h.smallA = h.dalloc<float>((size_t)tB * SMALL_STRIDE);
  h.pw2C = h.dalloc<float>((size_t)C * h.splitsC * H * H);
  h.pw2A = h.dalloc<float>((size_t)h.splitsA * H * H);
  if (cfg->precision != CQL_PREC_FP32) {
    const bool bf = cfg->precision == CQL_PREC_BF16, f16 = cfg->precision == CQL_PREC_F16X3;
    h.packed_net_bytes = f16 ? tc::HCfg::PACKED_NET_BYTES : (bf ? tc::Cfg<false>::PACKED_NET_BYTES : tc::Cfg<true>::PACKED_NET_BYTES);
    h.packed_net_bytes_bwd = f16 ? tc::HCfg::PACKED_NET_BYTES : (bf ? tc::Cfg<false>::PACKED_NET_BYTES : tc::Cfg<true>::PACKED_NET_BYTES);
    h.packed_fwd = h.dalloc<uint8_t>((size_t)(2 + 2 * C) * h.packed_net_bytes);
    const int slices = f16 ? tc::HCfg::SLICES : (bf ? tc::Cfg<false>::SLICES : tc::Cfg<true>::SLICES);
    h.part_floats = (size_t)C * std::max(slices, (int)tc::H2Cfg::PARTS) * ((size_t)B * (2 * n3 + 2)) * 2 + 4096;
    h.part = h.dalloc<float>(h.part_floats);
    h.tc_slices = slices;
    h.packed_bwd = h.dalloc<uint8_t>((size_t)(1 + C) * h.packed_net_bytes_bwd);
    if (f16) {
      h.packed_net_bytes2 = tc::H2Cfg::PACKED_NET_BYTES;
      h.packed_fwd2 = h.dalloc<uint8_t>((size_t)(2 + 2 * C) * h.packed_net_bytes2);
      h.packed_bwd2 = h.dalloc<uint8_t>((size_t)(1 + C) * h.packed_net_bytes2);
      h.w2max = h.dalloc<int>((size_t)(2 + 2 * C) * 4);
      h.ap_wmax = h.dalloc<int>((size_t)CQL_MAX_CRITICS * 17);
      h.pair_swap_b = switches().pair_swap;
    }
    h.slots1 = (f16 ? tc::HCfg::NEW : 4) * h.num_sms;
    h.splits_tc = h.num_sms;
    h.small1 = h.dalloc<float>((size_t)C * h.slots1 * SMALL_STRIDE);
    h.small2 = h.dalloc<float>((size_t)C * h.splits_tc * SMALL_STRIDE);
    h.pw2_tc = h.dalloc<float>((size_t)(h.num_sms + C) * H * H);
    h.dX_part = h.dalloc<float4>((size_t)C * std::max(slices, 8) * B);
  }
  // scalars start at the configured initial values; networks are set by cql_set_weights
  float sc[SCALAR_SLOT] = {0};
  sc[0] = logf(cfg->initial_temperature);
  sc[1] = logf(cfg->initial_alpha);
  CQL_CUDA(cudaMemcpy(h.scalars(), sc, sizeof(sc), cudaMemcpyHostToDevice));
}

void destroy_graph(cql_handle* ch) {
  ch->update_graph.reset();
  for (auto& g : ch->batch_graph) g.reset();
  ch->step_graph.reset();
}

template <typename F>
int guarded(cql_handle* ch, F&& f) {
  if (!ch) { g_create_error = "NULL handle"; return 1; }
  // the caller's current device is restored on every exit path (the handle's device is only current inside the call)
  struct DeviceScope {
    int prev = -1;
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
  } scope;
  try {
    int cur = -1;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != ch->h.cfg.device) scope.prev = cur;
    CQL_CUDA(cudaSetDevice(ch->h.cfg.device));
    f();
    return 0;
  } catch (const ArgError& e) {
    ch->h.err = e.msg;
    return 3;
  } catch (const Error& e) {
    ch->h.err = e.msg;
    return 1;
  } catch (const std::exception& e) {
    ch->h.err = e.what();
    return 2;
  }
}

void run_full_step(Handle* h, cudaStream_t st, BatchSource bs, NoiseSource ns) {
  with_precision(h, [&](auto p) {
    constexpr Prec P = decltype(p)::value;
    phase0<P>(h, st, bs, ns);
    phase1<P>(h, st);
    phase2<P>(h, st);
    phase3<P>(h, st);
  });
}

// a host minibatch (obs [B][2], act, rew, next_obs [B][2], term) -> B rows of the table's format in `rows`; the discount
// slot holds gamma in n-step mode (these are one-step transitions) and 0 otherwise
void pack_rows(const Handle& h, const float* obs, const float* act, const float* rew, const float* next_obs,
               const float* term, float* rows) {
  const float disc = h.n_steps > 1 ? h.cfg.gamma : 0.f;
  for (int b = 0; b < h.B; ++b) {
    float* r = rows + (size_t)b * 8;
    r[0] = obs[2 * b]; r[1] = obs[2 * b + 1]; r[2] = act[b]; r[3] = rew[b];
    r[4] = next_obs[2 * b]; r[5] = next_obs[2 * b + 1]; r[6] = term[b]; r[7] = disc;
  }
}

// obs scaler on: the candidate items' scaled coordinates (k_scale_items) in scratch slot 7; off: nullptr (the scorers
// convert the ids themselves, as without preprocessing)
const float* scaled_items(cql_handle* ch, const int32_t* items, int64_t I, cudaStream_t st) {
  Handle* h = &ch->h;
  if (!h->prep.obs[1].on) return nullptr;
  float* out = static_cast<float*>(scratch(ch, 7, (size_t)I * sizeof(float)));
  k_scale_items<<<(unsigned)((I + 255) / 256), 256, 0, st>>>(items, I, h->prep.obs[1], out);
  CQL_LAUNCH_CHECK(h);
  return out;
}

void score_topk_dev_impl(cql_handle* ch, const int32_t* users, int64_t U, const int32_t* items, int64_t I,
                         const int64_t* seen_indptr, const int32_t* seen_items, int k, int mode, int32_t* out_items,
                         float* out_scores, cudaStream_t st) {
  Handle* h = &ch->h;
  CQL_REQUIRE(k >= 1 && k <= CQL_MAX_TOPK, "cql_score_topk: k must be 1..1024");
  CQL_REQUIRE(mode == CQL_SCORE_Q || mode == CQL_SCORE_POLICY, "cql_score_topk: bad mode");
  CQL_REQUIRE(U >= 0 && I >= 0 && U < (1ll << 31), "cql_score_topk: bad sizes");
  if (U == 0) return;
  const int64_t tiles = (I + BM - 1) / BM;
  if (tiles == 0) {  // no candidates: pad
    CQL_CUDA(cudaMemsetAsync(out_items, 0xff, (size_t)U * k * sizeof(int32_t), st));
    std::vector<float> ninf((size_t)U * k, -INFINITY);
    CQL_CUDA(cudaMemcpyAsync(out_scores, ninf.data(), ninf.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaStreamSynchronize(st));
    return;
  }
  if (h->cfg.precision != CQL_PREC_FP32) {   // tensor-core scorer, FP32-grade: fp16 hi/lo split (f16x3) or tf32 split (other modes)
    using TC = tc::Cfg<true>;
    const bool f16 = h->cfg.precision == CQL_PREC_F16X3;
    if (!ch->packed_score)
      CQL_CUDA(cudaMalloc(&ch->packed_score, (size_t)(1 + h->C) * std::max<size_t>(TC::PACKED_NET_BYTES, tc::HCfg::PACKED_NET_BYTES)));
    if (f16) {
      tc::PackJobs pj{};
      pj.j[pj.n++] = {h->net_params(slot_actor()), ch->packed_score, 2, 0};
      for (int c = 0; c < h->C; ++c)
        pj.j[pj.n++] = {h->net_params(slot_critic(c)), ch->packed_score + (size_t)(1 + c) * tc::HCfg::PACKED_NET_BYTES, 3, 0};
      tc::k_pack_multi_h<<<dim3(H * 32 / 256, pj.n), 256, 0, st>>>(pj, 2);
      CQL_LAUNCH_CHECK(h);
    } else {
      const int chunks16 = H * (H / TC::EPC);
      tc::k_pack_w2<true, false><<<dim3((chunks16 + 255) / 256, 1), 256, 0, st>>>(h->net_params(slot_actor()), 2, 1, ch->packed_score);
      CQL_LAUNCH_CHECK(h);
      tc::k_pack_w2<true, false><<<dim3((chunks16 + 255) / 256, h->C), 256, 0, st>>>(h->net_params(slot_critic(0)), 3, h->C,
                                                                                     ch->packed_score + TC::PACKED_NET_BYTES);
      CQL_LAUNCH_CHECK(h);
    }
    const int64_t tiles128 = (I + tc::TM - 1) / tc::TM;
    const int chunks = (int)((tiles128 + tc::SC_CH - 1) / tc::SC_CH);
    const size_t need = (size_t)U * chunks * k;
    float* ps = out_scores;
    int* pi = out_items;
    if (chunks > 1) {
      if (need > ch->part_elems) {
        if (ch->part_s) CQL_CUDA(cudaFree(ch->part_s));
        if (ch->part_i) CQL_CUDA(cudaFree(ch->part_i));
        ch->part_s = nullptr; ch->part_i = nullptr; ch->part_elems = 0;
        CQL_CUDA(cudaMalloc(&ch->part_s, need * sizeof(float)));
        CQL_CUDA(cudaMalloc(&ch->part_i, need * sizeof(int)));
        ch->part_elems = need;
      }
      ps = ch->part_s;
      pi = ch->part_i;
    }
    tc::ScoreTcArgs a{h->params, ch->packed_score, users, items, seen_indptr, seen_items, U, I, h->C, k, mode, chunks, ps, pi,
                      scaled_items(ch, items, I, st), h->prep};
    const int64_t n_blocks = U * chunks;
    const int grid = (int)std::min<int64_t>(n_blocks, h->num_sms);
    if (f16) tc::tc_score_h_kernel<<<grid, tc::HCfg4::THREADS, tc::ScoreSmemH::bytes(k), st>>>(a);
    else tc::tc_score_kernel<<<grid, tc::TsCfg::THREADS, tc::ScoreSmem::bytes(k), st>>>(a);
    CQL_LAUNCH_CHECK(h);
    if (chunks > 1) {
      const int wpb = 4;
      k_topk_merge<<<(unsigned)((U + wpb - 1) / wpb), wpb * 32, wpb * 2 * k * sizeof(float), st>>>(ps, pi, U, chunks, k,
                                                                                                  out_scores, out_items);
      CQL_LAUNCH_CHECK(h);
    }
    return;
  }
  // enough CTAs to fill the machine a few times over, at most one chunk per tile
  int64_t want = (8ll * h->num_sms + U - 1) / U;
  int chunks = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, want));
  int tpc = (int)((tiles + chunks - 1) / chunks);
  chunks = (int)((tiles + tpc - 1) / tpc);
  CQL_REQUIRE(chunks <= 65535 * 32, "cql_score_topk: too many chunks");
  ScoreArgs a{};
  a.params = h->params; a.users = users; a.items = items;
  a.seen_indptr = seen_indptr; a.seen_items = seen_items;
  a.n_users = U; a.n_items = I; a.C = h->C; a.k = k; a.mode = mode; a.chunks = chunks; a.tiles_per_chunk = tpc;
  a.item_x = scaled_items(ch, items, I, st);
  a.prep = h->prep;
  // users go on grid.y (max 65535): process in slabs
  const int64_t slab = 65535;
  for (int64_t u0 = 0; u0 < U; u0 += slab) {
    const int64_t nu = std::min(slab, U - u0);
    ScoreArgs s = a;
    s.users = users + u0;
    s.n_users = nu;
    if (chunks == 1) {
      s.part_s = out_scores + u0 * k;
      s.part_i = out_items + u0 * k;
    } else {
      const size_t need = (size_t)nu * chunks * k;
      if (need > ch->part_elems) {
        if (ch->part_s) CQL_CUDA(cudaFree(ch->part_s));
        if (ch->part_i) CQL_CUDA(cudaFree(ch->part_i));
        ch->part_s = nullptr; ch->part_i = nullptr; ch->part_elems = 0;
        CQL_CUDA(cudaMalloc(&ch->part_s, need * sizeof(float)));
        CQL_CUDA(cudaMalloc(&ch->part_i, need * sizeof(int)));
        ch->part_elems = need;
      }
      s.part_s = ch->part_s;
      s.part_i = ch->part_i;
    }
    k_score_topk<<<dim3(chunks, (unsigned)nu), NT, score_smem(k), st>>>(s);
    CQL_LAUNCH_CHECK(h);
    if (chunks > 1) {
      const int wpb = 4;
      k_topk_merge<<<(unsigned)((nu + wpb - 1) / wpb), wpb * 32, wpb * 2 * k * sizeof(float), st>>>(
          ch->part_s, ch->part_i, nu, chunks, k, out_scores + u0 * k, out_items + u0 * k);
      CQL_LAUNCH_CHECK(h);
    }
  }
}

// n_steps > 1: a device buffer for the one-step rows a table producer writes before the n-step expansion
// (finish_n_steps expands and frees it); n_steps == 1: the table itself
float* one_step_rows(Handle& h, int64_t n) {
  if (h.n_steps == 1) return h.table;
  float* p = nullptr;
  CQL_CUDA(cudaMalloc(&p, (size_t)n * 8 * sizeof(float)));
  return p;
}
void finish_n_steps(Handle& h, float* one_step, int64_t n, cudaStream_t st) {
  if (one_step == h.table) return;
  expand_n_steps(h, one_step, n, st);
  h.launches++;
  CQL_CUDA(cudaStreamSynchronize(st));
  CQL_CUDA(cudaFree(one_step));
}

// the host minibatch in h.batch_host -> one update (cql_update_batch, cql_update_batch_rows)
void update_staged_batch(cql_handle* ch, const float* noise, float* metrics6, float* grads_out, cudaStream_t st) {
  Handle& h = ch->h;
  const int B = h.B;
  if (noise) std::memcpy(h.noise_host, noise, h.noise_floats * sizeof(float));
  // pinned staging -> device, the 26 launches of the step and the metrics read-back replay as ONE CUDA graph
  // (26 runtime launches + 3 copies cost ~100 us of host time per step)
  auto enqueue = [&] {
    CQL_CUDA(cudaMemcpyAsync(h.staged_batch(), h.batch_host, (size_t)B * 8 * sizeof(float), cudaMemcpyHostToDevice, st));
    if (noise) CQL_CUDA(cudaMemcpyAsync(h.noise, h.noise_host, h.noise_floats * sizeof(float), cudaMemcpyHostToDevice, st));
    run_full_step(&h, st, BatchSource::Provided, noise ? NoiseSource::Provided : NoiseSource::Philox);
    CQL_CUDA(cudaMemcpyAsync(h.metrics_host, h.metrics, 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
  };
  ch->batch_graph[noise ? 1 : 0].run(h, st, 1, enqueue);
  if (grads_out)
    CQL_CUDA(cudaMemcpyAsync(grads_out, h.grads, grad_floats(h.C) * sizeof(float), cudaMemcpyDeviceToHost, st));
  CQL_CUDA(cudaStreamSynchronize(st));
  if (metrics6) std::memcpy(metrics6, h.metrics_host, 6 * sizeof(float));
}

}  // namespace

void cql::expand_n_steps(Handle& h, const float* one_step, int64_t n, cudaStream_t st) {
  const size_t smem = (size_t)(NSTEP_TILE + h.n_steps - 1) * 2 * sizeof(float4);
  k_nstep_rows<<<(unsigned)((n + NSTEP_TILE - 1) / NSTEP_TILE), NSTEP_TILE, smem, st>>>(
      reinterpret_cast<const float4*>(one_step), n, h.n_steps, (double)h.cfg.gamma, reinterpret_cast<float4*>(h.table));
  CQL_CUDA(cudaGetLastError());
}

int cql::table_stats(Handle& h, const float* rows, int64_t n, bool rew_ok, cudaStream_t st) {
  const int64_t nb = std::min<int64_t>((n + STATS_ROWS - 1) / STATS_ROWS, STATS_MAX_BLOCKS);
  const int64_t per_block = (n + nb - 1) / nb;
  Moments* part = reinterpret_cast<Moments*>(h.stats_dev);
  k_stats_partial<<<(unsigned)nb, STATS_THREADS, 0, st>>>(reinterpret_cast<const float4*>(rows), n, per_block, part);
  CQL_CUDA(cudaGetLastError());
  Moments* result = part + 4 * STATS_MAX_BLOCKS;
  k_stats_final<<<1, STATS_THREADS, 0, st>>>(part, nb, result);
  CQL_CUDA(cudaGetLastError());
  CQL_CUDA(cudaMemcpyAsync(h.stats_host, result, 4 * sizeof(Moments), cudaMemcpyDeviceToHost, st));
  h.stats_pending = true;
  h.stats_rew_ok = rew_ok;
  return 2;
}

extern "C" {

int cql_abi_version(void) { return CQL_ABI_VERSION; }

int cql_create(const cql_config* cfg, cql_handle** out) {
  if (!out) { g_create_error = "cql_create: out is NULL"; return 1; }
  *out = nullptr;
  cql_handle* ch = new cql_handle();
  try {
    create_impl(cfg, ch);
  } catch (const Error& e) {
    g_create_error = e.msg;
    ch->h.free_all();
    delete ch;
    return 1;
  }
  *out = ch;
  return 0;
}

void cql_destroy(cql_handle* ch) {
  if (!ch) return;
  cudaSetDevice(ch->h.cfg.device);
  cudaDeviceSynchronize();
  destroy_graph(ch);
  for (int i = 0; i < 8; ++i) if (ch->sbuf[i]) cudaFree(ch->sbuf[i]);
  if (ch->part_s) cudaFree(ch->part_s);
  if (ch->part_i) cudaFree(ch->part_i);
  if (ch->packed_score) cudaFree(ch->packed_score);
  if (ch->dp_local) cudaFree(ch->dp_local);
  if (ch->ring) cudaFreeHost(ch->ring);
  if (ch->metrics_rows) cudaFreeHost(ch->metrics_rows);
  for (auto& e : ch->ring_ev) if (e) cudaEventDestroy(e);
  for (auto& e : ch->ev_used) if (e) cudaEventDestroy(e);
  for (auto& e : ch->ev_met) if (e) cudaEventDestroy(e);
  for (auto& e : ch->ev_met_out) if (e) cudaEventDestroy(e);
  if (ch->dev_ring) cudaFree(ch->dev_ring);
  if (ch->dev_metrics) cudaFree(ch->dev_metrics);
  if (ch->copy_stream) cudaStreamDestroy(ch->copy_stream);
  if (ch->copy_stream_out) cudaStreamDestroy(ch->copy_stream_out);
  ch->h.free_all();
  delete ch;
}

const char* cql_last_error(const cql_handle* ch) { return ch ? ch->h.err.c_str() : g_create_error.c_str(); }

int64_t cql_state_floats(const cql_handle* ch) { return ch ? state_floats(ch->h.C) : 0; }
int64_t cql_num_transitions(const cql_handle* ch) { return ch ? ch->h.n_trans : 0; }
int64_t cql_launch_count(const cql_handle* ch) { return ch ? ch->h.launches : 0; }

int cql_set_weights(cql_handle* ch, const float* host_flat, int64_t n) {
  return guarded(ch, [&] {
    CQL_REQUIRE(host_flat && n == state_floats(ch->h.C), "cql_set_weights: n must equal cql_state_floats()");
    CQL_CUDA(cudaDeviceSynchronize());
    CQL_CUDA(cudaMemcpy(ch->h.params, host_flat, n * sizeof(float), cudaMemcpyHostToDevice));
    with_precision(&ch->h, [&](auto p) { pack_all_weights<decltype(p)::value>(&ch->h, ch->h.own_stream); });
    CQL_CUDA(cudaStreamSynchronize(ch->h.own_stream));
  });
}

int cql_get_weights(cql_handle* ch, float* host_flat, int64_t n) {
  return guarded(ch, [&] {
    CQL_REQUIRE(host_flat && n == state_floats(ch->h.C), "cql_get_weights: n must equal cql_state_floats()");
    CQL_CUDA(cudaDeviceSynchronize());
    CQL_CUDA(cudaMemcpy(host_flat, ch->h.params, n * sizeof(float), cudaMemcpyDeviceToHost));
  });
}

int cql_set_optimizer(cql_handle* ch, const float* host_m, const float* host_v, int64_t n, int64_t step) {
  return guarded(ch, [&] {
    CQL_REQUIRE(host_m && host_v && n == state_floats(ch->h.C), "cql_set_optimizer: n must equal cql_state_floats()");
    CQL_REQUIRE(step >= 0, "cql_set_optimizer: step must be >= 0");
    CQL_CUDA(cudaDeviceSynchronize());
    CQL_CUDA(cudaMemcpy(ch->h.adam_m, host_m, n * sizeof(float), cudaMemcpyHostToDevice));
    CQL_CUDA(cudaMemcpy(ch->h.adam_v, host_v, n * sizeof(float), cudaMemcpyHostToDevice));
    const long long s = step;
    CQL_CUDA(cudaMemcpy(ch->h.step_dev, &s, sizeof(s), cudaMemcpyHostToDevice));
  });
}

int cql_get_optimizer(cql_handle* ch, float* host_m, float* host_v, int64_t n, int64_t* step) {
  return guarded(ch, [&] {
    CQL_REQUIRE(host_m && host_v && step && n == state_floats(ch->h.C), "cql_get_optimizer: bad arguments");
    CQL_CUDA(cudaDeviceSynchronize());
    CQL_CUDA(cudaMemcpy(host_m, ch->h.adam_m, n * sizeof(float), cudaMemcpyDeviceToHost));
    CQL_CUDA(cudaMemcpy(host_v, ch->h.adam_v, n * sizeof(float), cudaMemcpyDeviceToHost));
    long long s = 0;
    CQL_CUDA(cudaMemcpy(&s, ch->h.step_dev, sizeof(s), cudaMemcpyDeviceToHost));
    *step = s;
  });
}

int cql_load_transitions(cql_handle* ch, const float* obs, const float* act, const float* rew, const float* term,
                         int64_t n) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(obs && act && rew && term && n >= 1, "cql_load_transitions: bad arguments");
    CQL_CUDA(cudaDeviceSynchronize());
    ensure_table(h, n);
    float* rows = one_step_rows(h, n);
    // stage the 20 B/step columns on the device, expand to 32 B rows there
    float *d_obs, *d_act, *d_rew, *d_term;
    CQL_CUDA(cudaMalloc(&d_obs, (size_t)n * 2 * sizeof(float)));
    CQL_CUDA(cudaMalloc(&d_act, (size_t)n * 3 * sizeof(float)));
    d_rew = d_act + n; d_term = d_rew + n;
    cudaStream_t st = h.own_stream;
    CQL_CUDA(cudaMemcpyAsync(d_obs, obs, (size_t)n * 2 * sizeof(float), cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(d_act, act, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(d_rew, rew, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(d_term, term, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, st));
    k_build_transitions<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float2*>(d_obs), d_act, d_rew,
                                                                    d_term, n, reinterpret_cast<float4*>(rows));
    CQL_LAUNCH_CHECK(&h);
    h.launches += table_stats(h, rows, n, true, st);
    finish_n_steps(h, rows, n, st);
    CQL_CUDA(cudaStreamSynchronize(st));
    CQL_CUDA(cudaFree(d_obs));
    CQL_CUDA(cudaFree(d_act));
    h.n_trans = n;
    destroy_graph(ch);
  });
}

int cql_set_n_steps(cql_handle* ch, int32_t n_steps) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(n_steps >= 1 && n_steps <= CQL_MAX_N_STEPS, "cql_set_n_steps: n_steps must be 1..64 (CQL_MAX_N_STEPS)");
    CQL_CUDA(cudaDeviceSynchronize());
    if (n_steps != h.n_steps) h.n_trans = 0;         // the table was built for the other horizon
    h.n_steps = n_steps;
    destroy_graph(ch);
  });
}

int cql_set_table_rows(cql_handle* ch, const float* rows, int64_t n) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(rows && n >= 1, "cql_set_table_rows: bad arguments");
    CQL_CUDA(cudaDeviceSynchronize());
    ensure_table(h, n);
    CQL_CUDA(cudaMemcpyAsync(h.table, rows, (size_t)n * 8 * sizeof(float), cudaMemcpyHostToDevice, h.own_stream));
    h.launches += table_stats(h, h.table, n, h.n_steps == 1, h.own_stream);   // n-step rows: returns in the reward slot
    CQL_CUDA(cudaStreamSynchronize(h.own_stream));
    h.n_trans = n;
    destroy_graph(ch);
  });
}

int cql_get_table_stats(cql_handle* ch, cql_table_stats* out) {
  return guarded(ch, [&] {
    CQL_REQUIRE(out != nullptr, "cql_get_table_stats: NULL output");
    Handle& h = ch->h;
    if (h.stats_pending) {            // the producer's asynchronous copy: every producer synchronises before returning
      CQL_CUDA(cudaDeviceSynchronize());
      const double* m = h.stats_host;   // per column: n, mean, m2, min, max (struct Moments)
      for (int c = 0; c < 4; ++c)
        h.stats.col[c] = cql_column_stats{(int64_t)m[5 * c], m[5 * c + 3], m[5 * c + 4], m[5 * c + 1], m[5 * c + 2]};
      h.stats.rew_available = h.stats_rew_ok ? 1 : 0;
      if (!h.stats_rew_ok) h.stats.col[3] = cql_column_stats{};
      h.stats_pending = false;
    }
    *out = h.n_trans > 0 ? h.stats : cql_table_stats{};
  });
}

int cql_set_preprocessing(cql_handle* ch, const cql_preprocessing* p) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(p != nullptr, "cql_set_preprocessing: NULL parameters");
    const cql_preprocessing& c = *p;
    CQL_REQUIRE(c.obs_kind >= CQL_SCALER_NONE && c.obs_kind <= CQL_SCALER_STANDARD, "cql_set_preprocessing: bad obs_kind");
    CQL_REQUIRE(c.act_kind == CQL_SCALER_NONE || c.act_kind == CQL_SCALER_MIN_MAX,
                "cql_set_preprocessing: act_kind must be NONE or MIN_MAX");
    CQL_REQUIRE(c.rew_kind >= CQL_SCALER_NONE && c.rew_kind <= CQL_SCALER_STANDARD, "cql_set_preprocessing: bad rew_kind");
    // (a, b) of one column -> the kernels' (off, den): den = b - a (min_max) or b + 1e-3 (standard), rounded once
    auto affine = [](int kind, float a, float b, const char* what) {
      if (kind == CQL_SCALER_NONE) return Affine{0, 0.f, 1.f};
      CQL_REQUIRE(std::isfinite(a) && std::isfinite(b), std::string("cql_set_preprocessing: non-finite parameter of ") + what);
      if (kind == CQL_SCALER_MIN_MAX) {
        CQL_REQUIRE(b > a, std::string("cql_set_preprocessing: min_max needs maximum > minimum for ") + what);
        const volatile float den = b - a;
        return Affine{1, a, den};
      }
      CQL_REQUIRE(b >= 0.f, std::string("cql_set_preprocessing: standard needs std >= 0 for ") + what);
      const volatile float den = b + 1e-3f;
      return Affine{1, a, den};
    };
    Prep q{};
    q.obs[0] = affine(c.obs_kind, c.obs_a[0], c.obs_b[0], "obs.x");
    q.obs[1] = affine(c.obs_kind, c.obs_a[1], c.obs_b[1], "obs.y");
    q.act = affine(c.act_kind, c.act_a, c.act_b, "act");
    q.rew = affine(c.rew_kind, c.rew_a, c.rew_b, "rew");
    CQL_CUDA(cudaDeviceSynchronize());
    h.prep = q;
    h.prep_cfg = c;
    h.prep_cfg.pad = 0;
    destroy_graph(ch);              // the parameters are kernel arguments of the captured graphs
  });
}

int cql_get_preprocessing(cql_handle* ch, cql_preprocessing* out) {
  return guarded(ch, [&] {
    CQL_REQUIRE(out != nullptr, "cql_get_preprocessing: NULL output");
    *out = ch->h.prep_cfg;
  });
}

int cql_mdp_begin(cql_handle* ch, int64_t n_rows) {
  return guarded(ch, [&] {
    CQL_CUDA(cudaDeviceSynchronize());
    mdp_begin(ch->h, n_rows);
  });
}
int cql_mdp_append(cql_handle* ch, int32_t col, int32_t dtype, const void* host_chunk, int64_t count) {
  return guarded(ch, [&] { mdp_append(ch->h, col, dtype, host_chunk, count); });
}
int cql_mdp_finish(cql_handle* ch, int32_t top_k, float noise_scale, float* obs_out, float* act_out, float* rew_out,
                   float* term_out, int64_t* order_out) {
  return guarded(ch, [&] {
    ch->h.launches += mdp_finish(ch->h, top_k, noise_scale, obs_out, act_out, rew_out, term_out, order_out);
    destroy_graph(ch);
  });
}

int cql_set_table_sharded(cql_handle* ch, int32_t sharded) {
  return guarded(ch, [&] {
    ch->h.table_sharded = sharded != 0;
    destroy_graph(ch);
  });
}

int cql_synth_table(cql_handle* ch, int64_t n, int64_t n_users, int64_t n_items, uint64_t seed) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(n >= 1 && n_users >= 1 && n_items >= 1 && n_users <= n, "cql_synth_table: bad shape");
    CQL_REQUIRE(n_users < (1ll << 24) && n_items < (1ll << 24), "cql_synth_table: ids must stay below 2^24 (exact in float32)");
    CQL_CUDA(cudaDeviceSynchronize());
    ensure_table(h, n);
    float* rows = one_step_rows(h, n);
    k_synth_table<<<(unsigned)((n + 255) / 256), 256, 0, h.own_stream>>>(reinterpret_cast<float4*>(rows), n, n_users, n_items, seed);
    CQL_LAUNCH_CHECK(&h);
    h.launches += table_stats(h, rows, n, true, h.own_stream);
    finish_n_steps(h, rows, n, h.own_stream);
    CQL_CUDA(cudaStreamSynchronize(h.own_stream));
    h.n_trans = n;
    destroy_graph(ch);
  });
}

int cql_build_mdp(cql_handle* ch, const int32_t* user_idx, const int32_t* item_idx, const int64_t* timestamp,
                  const double* relevance, const double* action_noise, int64_t n, int32_t top_k, float noise_scale,
                  float* obs_out, float* act_out, float* rew_out, float* term_out, int64_t* order_out) {
  return guarded(ch, [&] {
    CQL_CUDA(cudaDeviceSynchronize());
    ch->h.launches += mdp_build_on_device(ch->h, user_idx, item_idx, timestamp, relevance, action_noise, n, top_k,
                                          noise_scale, obs_out, act_out, rew_out, term_out, order_out);
    destroy_graph(ch);
  });
}

int cql_seen_csr(cql_handle* ch, const int32_t* users_host, const int32_t* items_host, int64_t n, int64_t n_users_dim,
                 const uint8_t* wanted_host, int64_t* indptr_dev, int32_t* seen_dev, int64_t* n_seen_out, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_seen_csr");
    CQL_REQUIRE(n_seen_out != nullptr, "cql_seen_csr: n_seen_out is NULL");
    cudaStream_t st = pick_stream(&ch->h, stream);
    *n_seen_out = seen_csr_on_device(ch->h, users_host, items_host, n, n_users_dim, wanted_host, indptr_dev, seen_dev, st);
    ch->h.launches += 4;
  });
}

int cql_sample_rows(cql_handle* ch, const int64_t* idx_dev, int64_t pos, int64_t count, float* out_dev, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(h.n_trans > 0, "cql_sample_rows: no transitions loaded");
    CQL_REQUIRE(count >= 0 && out_dev, "cql_sample_rows: bad arguments");
    if (count == 0) return;
    cudaStream_t st = pick_stream(&h, stream);
    k_sample<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(reinterpret_cast<const float4*>(h.table), h.n_trans, idx_dev,
                                                             nullptr, pos, count, std::max<int64_t>(1, h.B), 0, 1,
                                                             h.cfg.seed, reinterpret_cast<float4*>(out_dev));
    CQL_LAUNCH_CHECK(&h);
    if (!stream) CQL_CUDA(cudaStreamSynchronize(st));   // NULL stream = the handle's own stream: return when done
  });
}

int cql_update(cql_handle* ch, int64_t n_steps, float* metrics6, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_update: graph replays");
    Handle& h = ch->h;
    CQL_REQUIRE(n_steps >= 0, "cql_update: n_steps < 0");
    CQL_REQUIRE(h.n_trans > 0, "cql_update: no transitions loaded (call cql_load_transitions first)");
    cudaStream_t st = pick_stream(&h, stream);
    ch->update_graph.run(h, st, n_steps, [&] { run_full_step(&h, st, BatchSource::Sampled, NoiseSource::Philox); });
    if (metrics6) {
      CQL_CUDA(cudaMemcpyAsync(h.metrics_host, h.metrics, 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
      CQL_CUDA(cudaStreamSynchronize(st));
      std::memcpy(metrics6, h.metrics_host, 6 * sizeof(float));
    }
  });
}

int cql_selftest_umma(cql_handle* ch, int precision, const float* A_host, const float* B_host, int n, int k,
                      float* D_host) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    const bool a_in_tmem = (precision & 0x100) != 0;     // +0x100: stage A in tensor memory (TS mode)
    precision &= 0xff;
    CQL_REQUIRE(precision == CQL_PREC_TF32X3 || precision == CQL_PREC_BF16, "cql_selftest_umma: precision must be tf32x3 or bf16");
    const bool tf32 = precision == CQL_PREC_TF32X3;
    CQL_REQUIRE(A_host && B_host && D_host, "cql_selftest_umma: NULL pointer");
    CQL_REQUIRE(n >= 16 && n <= 256 && n % 16 == 0, "cql_selftest_umma: n must be a multiple of 16 in 16..256");
    CQL_REQUIRE(k >= 32 && k % 32 == 0, "cql_selftest_umma: k must be a multiple of 32");
    const size_t smem = tc::selftest_smem(tf32, n, k);
    CQL_REQUIRE(smem <= 227 * 1024, "cql_selftest_umma: operands do not fit in shared memory");
    float *dA, *dB, *dD;
    CQL_CUDA(cudaMalloc(&dA, (size_t)128 * k * 4));
    CQL_CUDA(cudaMalloc(&dB, (size_t)n * k * 4));
    CQL_CUDA(cudaMalloc(&dD, (size_t)128 * n * 4));
    cudaStream_t st = h.own_stream;
    CQL_CUDA(cudaMemcpyAsync(dA, A_host, (size_t)128 * k * 4, cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(dB, B_host, (size_t)n * k * 4, cudaMemcpyHostToDevice, st));
    if (a_in_tmem) {
      CQL_REQUIRE((tf32 ? 2 * k : k / 2) + n <= 512, "cql_selftest_umma: A + D do not fit in tensor memory");
      if (tf32) {
        CQL_CUDA(cudaFuncSetAttribute(tc::umma_ts_selftest_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::umma_ts_selftest_kernel<true><<<1, 128, smem, st>>>(dA, dB, dD, n, k);
      } else {
        CQL_CUDA(cudaFuncSetAttribute(tc::umma_ts_selftest_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tc::umma_ts_selftest_kernel<false><<<1, 128, smem, st>>>(dA, dB, dD, n, k);
      }
    } else if (tf32) {
      CQL_CUDA(cudaFuncSetAttribute(tc::umma_selftest_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      tc::umma_selftest_kernel<true><<<1, 128, smem, st>>>(dA, dB, dD, n, k);
    } else {
      CQL_CUDA(cudaFuncSetAttribute(tc::umma_selftest_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      tc::umma_selftest_kernel<false><<<1, 128, smem, st>>>(dA, dB, dD, n, k);
    }
    CQL_LAUNCH_CHECK(&h);
    CQL_CUDA(cudaMemcpyAsync(D_host, dD, (size_t)128 * n * 4, cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaStreamSynchronize(st));
    CQL_CUDA(cudaFree(dA)); CQL_CUDA(cudaFree(dB)); CQL_CUDA(cudaFree(dD));
  });
}

int cql_mma_bench(cql_handle* ch, int mode, int iters, int64_t* out_clk2) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(out_clk2 && iters > 0 && mode >= 0 && mode < 16, "cql_mma_bench: bad arguments");
    long long* d = nullptr;
    CQL_CUDA(cudaMalloc(&d, 16));
    const size_t smem = 64 * 1024 + 64;
    CQL_CUDA(cudaFuncSetAttribute(tc::mma_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CQL_CUDA(cudaFuncSetAttribute(tc::mma_bench_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (mode & 4) tc::mma_bench_pair_kernel<<<2, 128, smem, h.own_stream>>>(mode, iters, d);
    else tc::mma_bench_kernel<<<1, 128, smem, h.own_stream>>>(mode, iters, d);
    CQL_LAUNCH_CHECK(&h);
    long long hst[2];
    CQL_CUDA(cudaStreamSynchronize(h.own_stream));
    CQL_CUDA(cudaMemcpy(hst, d, 16, cudaMemcpyDeviceToHost));
    CQL_CUDA(cudaFree(d));
    out_clk2[0] = hst[0]; out_clk2[1] = hst[1];
  });
}

int cql_timed_update(cql_handle* ch, float* out_ms8, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(out_ms8 != nullptr, "cql_timed_update: out is NULL");
    CQL_REQUIRE(h.n_trans > 0, "cql_timed_update: no transitions loaded");
    cudaStream_t st = pick_stream(&h, stream);
    for (int i = 0; i < 13; ++i)
      if (!h.ev[i]) CQL_CUDA(cudaEventCreate(&h.ev[i]));
    {
      // events between kernels only separate their durations without PDL overlap
      struct TimingScope {
        Handle& h;
        explicit TimingScope(Handle& h_) : h(h_) { h.timing = true; h.pdl_off = true; }
        ~TimingScope() { h.timing = false; h.pdl_off = false; }
      } timing(h);
      run_full_step(&h, st, BatchSource::Sampled, NoiseSource::Philox);
    }
    CQL_CUDA(cudaStreamSynchronize(st));
    auto ms = [&](int a, int b) { float t = 0.f; CQL_CUDA(cudaEventElapsedTime(&t, h.ev[a], h.ev[b])); return t; };
    const float fwd_all = ms(3, 4);           // TIMED_FWD_REPS launches of the critic forward, back to back
    out_ms8[0] = fwd_all / TIMED_FWD_REPS; out_ms8[1] = ms(5, 6); out_ms8[2] = ms(6, 7);
    out_ms8[3] = ms(0, 12) - (fwd_all - out_ms8[0]);
    out_ms8[4] = ms(8, 9); out_ms8[5] = ms(10, 11); out_ms8[6] = ms(1, 2);
    out_ms8[7] = out_ms8[3] - (out_ms8[0] + out_ms8[1] + out_ms8[2] + out_ms8[4] + out_ms8[5] + out_ms8[6]);
  });
}

int cql_update_batch(cql_handle* ch, const float* obs, const float* act, const float* rew, const float* next_obs,
                     const float* term, const float* noise, float* metrics6, float* grads_out, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(obs && act && rew && next_obs && term, "cql_update_batch: NULL batch pointer");
    cudaStream_t st = pick_stream(&h, stream);
    pack_rows(h, obs, act, rew, next_obs, term, h.batch_host);
    update_staged_batch(ch, noise, metrics6, grads_out, st);
  });
}

int cql_update_batch_rows(cql_handle* ch, const float* rows, const float* noise, float* metrics6, float* grads_out,
                          void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(rows != nullptr, "cql_update_batch_rows: NULL rows");
    cudaStream_t st = pick_stream(&h, stream);
    std::memcpy(h.batch_host, rows, (size_t)h.B * 8 * sizeof(float));
    update_staged_batch(ch, noise, metrics6, grads_out, st);
  });
}

int cql_update_batches(cql_handle* ch, int64_t n_batches, const float* obs, const float* act, const float* rew,
                       const float* next_obs, const float* term, float* metrics_out, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_update_batches");
    Handle& h = ch->h;
    CQL_REQUIRE(n_batches >= 0, "cql_update_batches: n_batches < 0");
    if (n_batches == 0) return;
    CQL_REQUIRE(obs && act && rew && next_obs && term, "cql_update_batches: NULL batch pointer");
    cudaStream_t st = pick_stream(&h, stream);
    const int B = h.B;
    constexpr int RING = 8;
    const size_t row_floats = (size_t)B * 8;
    if (!ch->ring) {
      CQL_CUDA(cudaMallocHost(&ch->ring, RING * row_floats * sizeof(float)));
      CQL_CUDA(cudaMalloc(&ch->dev_ring, RING * row_floats * sizeof(float)));
      CQL_CUDA(cudaMalloc(&ch->dev_metrics, RING * 8 * sizeof(float)));
      CQL_CUDA(cudaStreamCreateWithFlags(&ch->copy_stream, cudaStreamNonBlocking));
      CQL_CUDA(cudaStreamCreateWithFlags(&ch->copy_stream_out, cudaStreamNonBlocking));
      for (auto& e : ch->ring_ev) CQL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      for (auto& e : ch->ev_used) CQL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      for (auto& e : ch->ev_met) CQL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      for (auto& e : ch->ev_met_out) CQL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    cudaStream_t cs = ch->copy_stream, cso = ch->copy_stream_out;
    if (ch->metrics_rows_cap < n_batches) {
      if (ch->metrics_rows) CQL_CUDA(cudaFreeHost(ch->metrics_rows));
      ch->metrics_rows = nullptr; ch->metrics_rows_cap = 0;
      CQL_CUDA(cudaMallocHost(&ch->metrics_rows, (size_t)n_batches * 8 * sizeof(float)));
      ch->metrics_rows_cap = n_batches;
    }
    auto step = [&] { run_full_step(&h, st, BatchSource::Provided, NoiseSource::Philox); };   // minibatch already in h.batch
    ch->step_graph.run(h, st, 0, step);                                   // captured here, replayed in the loop
    // Copies ride on their own stream: minibatch i goes pinned ring -> device ring there (every step, 32 B x B), the
    // compute stream only waits for its event, moves it into h.batch (device to device), replays the step and drops the
    // step's metrics into a device slot, which the copy stream takes to the host (every step).  On one stream each
    // step paid both PCIe copies' start-up latency in series (e2e 0.885 of the HBM-resident rate).
    CQL_CUDA(cudaEventRecord(ch->ev_used[0], st));                        // orders the copy stream behind earlier work on st
    CQL_CUDA(cudaStreamWaitEvent(cs, ch->ev_used[0], 0));
    for (int64_t i = 0; i < n_batches; ++i) {
      const int slot = (int)(i % RING);
      if (i >= RING) CQL_CUDA(cudaEventSynchronize(ch->ring_ev[slot]));     // that slot's host->device copy has run
      float* stage = ch->ring + (size_t)slot * row_floats;
      pack_rows(h, obs + (size_t)i * B * 2, act + (size_t)i * B, rew + (size_t)i * B, next_obs + (size_t)i * B * 2,
                term + (size_t)i * B, stage);
      float* dslot = ch->dev_ring + (size_t)slot * row_floats;
      if (i >= RING) CQL_CUDA(cudaStreamWaitEvent(cs, ch->ev_used[slot], 0));   // the device slot has been consumed
      CQL_CUDA(cudaMemcpyAsync(dslot, stage, row_floats * sizeof(float), cudaMemcpyHostToDevice, cs));
      CQL_CUDA(cudaEventRecord(ch->ring_ev[slot], cs));
      CQL_CUDA(cudaStreamWaitEvent(st, ch->ring_ev[slot], 0));
      CQL_CUDA(cudaMemcpyAsync(h.staged_batch(), dslot, row_floats * sizeof(float), cudaMemcpyDeviceToDevice, st));
      CQL_CUDA(cudaEventRecord(ch->ev_used[slot], st));
      ch->step_graph.run(h, st, 1, step);
      if (i >= RING) CQL_CUDA(cudaStreamWaitEvent(st, ch->ev_met_out[slot], 0));   // the metrics slot has left the device
      CQL_CUDA(cudaMemcpyAsync(ch->dev_metrics + (size_t)slot * 8, h.metrics, 8 * sizeof(float), cudaMemcpyDeviceToDevice, st));
      CQL_CUDA(cudaEventRecord(ch->ev_met[slot], st));
      CQL_CUDA(cudaStreamWaitEvent(cso, ch->ev_met[slot], 0));
      CQL_CUDA(cudaMemcpyAsync(ch->metrics_rows + (size_t)i * 8, ch->dev_metrics + (size_t)slot * 8, 8 * sizeof(float),
                               cudaMemcpyDeviceToHost, cso));
      CQL_CUDA(cudaEventRecord(ch->ev_met_out[slot], cso));
    }
    CQL_CUDA(cudaStreamSynchronize(st));
    CQL_CUDA(cudaStreamSynchronize(cso));
    if (metrics_out)
      for (int64_t i = 0; i < n_batches; ++i) std::memcpy(metrics_out + i * 6, ch->metrics_rows + i * 8, 6 * sizeof(float));
  });
}

int cql_upload_batch(cql_handle* ch, const float* obs, const float* act, const float* rew, const float* next_obs,
                     const float* term, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(obs && act && rew && next_obs && term, "cql_upload_batch: NULL batch pointer");
    cudaStream_t st = pick_stream(&h, stream);
    const int B = h.B;
    CQL_CUDA(cudaStreamSynchronize(st));      // the staging buffer may still be in flight from the previous step
    pack_rows(h, obs, act, rew, next_obs, term, h.batch_host);
    CQL_CUDA(cudaMemcpyAsync(h.staged_batch(), h.batch_host, (size_t)B * 8 * sizeof(float), cudaMemcpyHostToDevice, st));
  });
}

int cql_step_phase(cql_handle* ch, int phase, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    cudaStream_t st = pick_stream(&h, stream);
    with_precision(&h, [&](auto p) {
      constexpr Prec P = decltype(p)::value;
      switch (phase) {
        case 0: phase0<P>(&h, st, BatchSource::Sampled, NoiseSource::Philox); break;
        case 1: phase1<P>(&h, st); break;
        case 2: phase2<P>(&h, st); break;
        case 3: phase3<P>(&h, st); break;
        case 4: phase0<P>(&h, st, BatchSource::Provided, NoiseSource::Philox); break;   // after cql_upload_batch
        default: throw Error{"cql_step_phase: phase must be 0..4"};
      }
    });
  });
}

int cql_dp_attach(cql_handle* ch, int32_t world, int32_t rank, const void* const* stage_ptrs,
                  const void* const* signal_ptrs, int64_t stage_floats, int64_t buffer_floats) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(world >= 1 && world <= DP_MAX_WORLD && rank >= 0 && rank < world, "cql_dp_attach: bad world / rank");
    CQL_REQUIRE(stage_ptrs && signal_ptrs, "cql_dp_attach: NULL pointer table");
    const int64_t need = (int64_t)grad_floats(h.C);
    CQL_REQUIRE(stage_floats >= need && stage_floats % 4 == 0, "cql_dp_attach: staging buffer too small (need the CQL_BUF_ALL_GRADS size, multiple of 4)");
    CQL_REQUIRE(buffer_floats >= 2 * stage_floats, "cql_dp_attach: buffer_floats must cover the two staging halves (2 x stage_floats)");
    // fused exchange: behind the two halves, [2][world][stage_floats] {value, tag} pairs pushed by the peers
    // (packets are tiled by 32 value groups = 128 floats: a slot must be a whole number of tiles)
    const bool ll_room = stage_floats % 128 == 0 && buffer_floats >= 2 * stage_floats + 4 * (int64_t)world * stage_floats;
    DpPeer& p = ch->h.dp;
    p.world = world; p.rank = rank; p.stage_floats = stage_floats;
    for (int r = 0; r < world; ++r) {
      CQL_REQUIRE(stage_ptrs[r] && signal_ptrs[r], "cql_dp_attach: NULL peer pointer");
      p.stage[r] = (float*)stage_ptrs[r];
      p.sig[r] = (unsigned long long*)signal_ptrs[r];
    }
    if (!ch->dp_local) CQL_CUDA(cudaMalloc(&ch->dp_local, 256));
    CQL_CUDA(cudaMemset(ch->dp_local, 0, 256));
    p.epoch = (unsigned long long*)ch->dp_local;
    p.ticket = (unsigned int*)((char*)ch->dp_local + 64);
    p.error = (int*)((char*)ch->dp_local + 128);
    p.debug = switches().dp_debug;
    h.dp_fused = world > 1 && ll_room && h.cfg.precision == CQL_PREC_F16X3 && !switches().no_fused_dp;
    destroy_graph(ch);
  });
}

int cql_dp_allreduce(cql_handle* ch, int which, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    DpPeer& p = h.dp;
    CQL_REQUIRE(p.world >= 1, "cql_dp_allreduce: call cql_dp_attach first");
    if (h.dp_fused) return;                // the update kernels exchange the gradients themselves (dp_peer.cuh)
    float* buf = nullptr;
    int64_t n = 0, off = 0;
    int group = 0;
    switch (which) {                      // staging offsets follow the CQL_BUF_ALL_GRADS layout [actor | critics | scalars]
      case CQL_BUF_SCALAR_GRADS: buf = h.g_scalars(); n = SCALAR_SLOT; off = (int64_t)(1 + h.C) * NET_STRIDE; group = 0; break;
      case CQL_BUF_CRITIC_GRADS: buf = h.g_critics(); n = (int64_t)h.C * NET_STRIDE; off = NET_STRIDE; group = 1; break;
      case CQL_BUF_ACTOR_GRADS: buf = h.g_actor(); n = NET_STRIDE; off = 0; group = 2; break;
      default: throw Error{"cql_dp_allreduce: which must be a CQL_BUF_*_GRADS group"};
    }
    if (p.world == 1) return;
    cudaStream_t st = pick_stream(&h, stream);
    const int grid = (int)std::min<int64_t>(h.num_sms, (n / 4 + 255) / 256);
    k_dp_exchange<<<grid, 256, 0, st>>>(p, buf, off, n, group);      // grid <= SMs: every block resident while waiting
    CQL_LAUNCH_CHECK(&h);
  });
}

int cql_dp_error(cql_handle* ch, int32_t* flag_out) {
  return guarded(ch, [&] {
    CQL_REQUIRE(flag_out, "cql_dp_error: NULL output");
    *flag_out = 0;
    if (ch->dp_local) CQL_CUDA(cudaMemcpy(flag_out, (char*)ch->dp_local + 128, sizeof(int32_t), cudaMemcpyDeviceToHost));
  });
}

int cql_dp_mode(cql_handle* ch, int32_t* fused_out) {
  return guarded(ch, [&] {
    CQL_REQUIRE(fused_out, "cql_dp_mode: NULL output");
    *fused_out = ch->h.dp_fused ? 1 : 0;
  });
}

int cql_device_buffer(cql_handle* ch, int which, void** dev_ptr, int64_t* n_floats) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(dev_ptr && n_floats, "cql_device_buffer: NULL out pointer");
    switch (which) {
      case CQL_BUF_SCALAR_GRADS: *dev_ptr = h.g_scalars(); *n_floats = SCALAR_SLOT; break;
      case CQL_BUF_CRITIC_GRADS: *dev_ptr = h.g_critics(); *n_floats = (int64_t)h.C * NET_STRIDE; break;
      case CQL_BUF_ACTOR_GRADS: *dev_ptr = h.g_actor(); *n_floats = NET_STRIDE; break;
      case CQL_BUF_METRICS: *dev_ptr = h.metrics; *n_floats = 8; break;
      case CQL_BUF_PARAMS: *dev_ptr = h.params; *n_floats = state_floats(h.C); break;
      case CQL_BUF_ALL_GRADS: *dev_ptr = h.grads; *n_floats = grad_floats(h.C); break;
      default: throw Error{"cql_device_buffer: unknown buffer id"};
    }
  });
}

int cql_score_topk_dev(cql_handle* ch, const int32_t* users, int64_t n_users, const int32_t* items, int64_t n_items,
                       const int64_t* seen_indptr, const int32_t* seen_items, int32_t k, int32_t mode,
                       int32_t* out_items, float* out_scores, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_score_topk_dev");
    CQL_REQUIRE((n_users == 0 || users) && (n_items == 0 || items) && out_items && out_scores,
                "cql_score_topk_dev: NULL pointer");
    score_topk_dev_impl(ch, users, n_users, items, n_items, seen_indptr, seen_items, k, mode, out_items, out_scores,
                        pick_stream(&ch->h, stream));
    if (!stream) CQL_CUDA(cudaStreamSynchronize(pick_stream(&ch->h, stream)));
  });
}

int cql_score_topk(cql_handle* ch, const int32_t* users, int64_t n_users, const int32_t* items, int64_t n_items,
                   const int64_t* seen_indptr, const int32_t* seen_items, int32_t k, int32_t mode, int32_t* out_items,
                   float* out_scores, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_score_topk");
    CQL_REQUIRE((n_users == 0 || users) && (n_items == 0 || items) && (n_users == 0 || (out_items && out_scores)),
                "cql_score_topk: NULL pointer");
    CQL_REQUIRE(k >= 1 && k <= CQL_MAX_TOPK, "cql_score_topk: k must be 1..1024");
    if (n_users == 0) return;
    cudaStream_t st = pick_stream(&ch->h, stream);
    int32_t* d_users = (int32_t*)scratch(ch, 0, (size_t)n_users * 4);
    int32_t* d_items = (int32_t*)scratch(ch, 1, (size_t)std::max<int64_t>(1, n_items) * 4);
    int32_t* d_oi = (int32_t*)scratch(ch, 2, (size_t)n_users * k * 4);
    float* d_os = (float*)scratch(ch, 3, (size_t)n_users * k * 4);
    CQL_CUDA(cudaMemcpyAsync(d_users, users, (size_t)n_users * 4, cudaMemcpyHostToDevice, st));
    if (n_items) CQL_CUDA(cudaMemcpyAsync(d_items, items, (size_t)n_items * 4, cudaMemcpyHostToDevice, st));
    int64_t* d_ptr = nullptr;
    int32_t* d_seen = nullptr;
    if (seen_indptr) {
      int32_t mx = 0;
      for (int64_t i = 0; i < n_users; ++i) {
        CQL_REQUIRE(users[i] >= 0, "cql_score_topk: negative user id");
        mx = std::max(mx, users[i]);
      }
      const int64_t np = (int64_t)mx + 2;
      const int64_t ns = seen_indptr[np - 1];
      d_ptr = (int64_t*)scratch(ch, 4, (size_t)np * 8);
      d_seen = (int32_t*)scratch(ch, 5, (size_t)std::max<int64_t>(1, ns) * 4);
      CQL_CUDA(cudaMemcpyAsync(d_ptr, seen_indptr, (size_t)np * 8, cudaMemcpyHostToDevice, st));
      if (ns) {
        CQL_REQUIRE(seen_items, "cql_score_topk: seen_items is NULL");
        CQL_CUDA(cudaMemcpyAsync(d_seen, seen_items, (size_t)ns * 4, cudaMemcpyHostToDevice, st));
      }
    }
    score_topk_dev_impl(ch, d_users, n_users, d_items, n_items, d_ptr, d_seen, k, mode, d_oi, d_os, st);
    CQL_CUDA(cudaMemcpyAsync(out_items, d_oi, (size_t)n_users * k * 4, cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaMemcpyAsync(out_scores, d_os, (size_t)n_users * k * 4, cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaStreamSynchronize(st));
  });
}

int cql_score_pairs(cql_handle* ch, const int32_t* users, const int32_t* items, int64_t n, int32_t mode,
                    float* out_scores, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(n >= 0 && (n == 0 || (users && items && out_scores)), "cql_score_pairs: bad arguments");
    CQL_REQUIRE(mode == CQL_SCORE_Q || mode == CQL_SCORE_POLICY, "cql_score_pairs: bad mode");
    if (n == 0) return;
    cudaStream_t st = pick_stream(&h, stream);
    int32_t* d_u = (int32_t*)scratch(ch, 0, (size_t)n * 4);
    int32_t* d_i = (int32_t*)scratch(ch, 1, (size_t)n * 4);
    float* d_o = (float*)scratch(ch, 3, (size_t)n * 4);
    CQL_CUDA(cudaMemcpyAsync(d_u, users, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(d_i, items, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    k_score_pairs<<<(unsigned)((n + BM - 1) / BM), NT, FWD_SMEM, st>>>(h.params, d_u, d_i, n, h.C, mode, d_o, h.prep);
    CQL_LAUNCH_CHECK(&h);
    CQL_CUDA(cudaMemcpyAsync(out_scores, d_o, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaStreamSynchronize(st));
  });
}

int cql_rank_metrics(cql_handle* ch, const int32_t* rec_items, int64_t n_users, int32_t k_rec, const int32_t* users,
                     const int64_t* gt_indptr, const int32_t* gt_items, const int32_t* ks, int32_t n_ks,
                     double* out_means, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_rank_metrics");
    Handle& h = ch->h;
    CQL_REQUIRE(n_users >= 0 && k_rec >= 1 && n_ks >= 1 && n_ks <= MET_MAX_KS && ks && out_means, "cql_rank_metrics: bad arguments");
    for (int q = 0; q < n_ks; ++q) CQL_REQUIRE(ks[q] >= 1, "cql_rank_metrics: k must be >= 1");
    if (n_users == 0) {
      for (int i = 0; i < MET_COUNT * n_ks; ++i) out_means[i] = 0.0;
      return;
    }
    CQL_REQUIRE(rec_items && users && gt_indptr, "cql_rank_metrics: NULL input");
    cudaStream_t st = pick_stream(&h, stream);
    int32_t mx = 0;
    for (int64_t i = 0; i < n_users; ++i) {
      CQL_REQUIRE(users[i] >= 0, "cql_rank_metrics: negative user id");
      mx = std::max(mx, users[i]);
    }
    const int64_t np = (int64_t)mx + 2, ng = gt_indptr[np - 1];
    CQL_REQUIRE(ng == 0 || gt_items, "cql_rank_metrics: gt_items is NULL");
    int32_t* d_rec = (int32_t*)scratch(ch, 0, (size_t)n_users * k_rec * 4);
    int32_t* d_users = (int32_t*)scratch(ch, 1, (size_t)n_users * 4);
    int64_t* d_ptr = (int64_t*)scratch(ch, 4, (size_t)np * 8);
    int32_t* d_gt = (int32_t*)scratch(ch, 5, (size_t)std::max<int64_t>(1, ng) * 4);
    double* d_pu = (double*)scratch(ch, 2, (size_t)MET_COUNT * n_ks * n_users * 8);
    double* d_out = (double*)scratch(ch, 3, (size_t)MET_COUNT * n_ks * 8);
    CQL_CUDA(cudaMemcpyAsync(d_rec, rec_items, (size_t)n_users * k_rec * 4, cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(d_users, users, (size_t)n_users * 4, cudaMemcpyHostToDevice, st));
    CQL_CUDA(cudaMemcpyAsync(d_ptr, gt_indptr, (size_t)np * 8, cudaMemcpyHostToDevice, st));
    if (ng) CQL_CUDA(cudaMemcpyAsync(d_gt, gt_items, (size_t)ng * 4, cudaMemcpyHostToDevice, st));
    MetricArgs ma{};
    ma.rec_items = d_rec; ma.users = d_users; ma.gt_indptr = d_ptr; ma.gt_items = d_gt;
    ma.n_users = n_users; ma.k_rec = k_rec; ma.n_ks = n_ks; ma.per_user = d_pu;
    for (int q = 0; q < n_ks; ++q) ma.ks[q] = ks[q];
    k_rank_metrics<<<(unsigned)((n_users + 127) / 128), 128, 0, st>>>(ma);
    CQL_LAUNCH_CHECK(&h);
    k_metric_mean<<<MET_COUNT * n_ks, 256, 0, st>>>(d_pu, n_users, d_out);
    CQL_LAUNCH_CHECK(&h);
    CQL_CUDA(cudaMemcpyAsync(out_means, d_out, (size_t)MET_COUNT * n_ks * 8, cudaMemcpyDeviceToHost, st));
    CQL_CUDA(cudaStreamSynchronize(st));
  });
}

int cql_topk_filter_dev(cql_handle* ch, const float* scores_dev, int64_t n_users, int64_t n_items,
                        const int32_t* users_dev, const int32_t* items_dev, const int64_t* seen_indptr,
                        const int32_t* seen_items, int32_t k, int32_t* out_items, float* out_scores, void* stream) {
  return guarded(ch, [&] {
    Handle& h = ch->h;
    CQL_REQUIRE(scores_dev && out_items && out_scores && n_users >= 0 && n_items >= 1, "cql_topk_filter_dev: bad arguments");
    CQL_REQUIRE(k >= 1 && k <= 128, "cql_topk_filter_dev: k must be 1..128");
    if (n_users == 0) return;
    cudaStream_t st = pick_stream(&h, stream);
    if (k <= 32) {     // streamed through a shared-memory ring (bulk copies), two-pass selection: topk_staged.cuh
      TksArgs ta{};
      ta.scores = scores_dev; ta.n_rows = n_users; ta.n_items = n_items; ta.users = users_dev; ta.items = items_dev;
      ta.seen_indptr = seen_indptr; ta.seen_items = seen_items; ta.k = k; ta.out_s = out_scores; ta.out_i = out_items;
      ta.chunk_len = TKS_CH;                                   // chunk starts stay multiples of TKS_WORKERS float4s
      ta.nchunks = (int)((n_items + TKS_CH - 1) / TKS_CH);
      ta.aligned = ((reinterpret_cast<uintptr_t>(scores_dev) & 15) == 0 && (n_items & 3) == 0) ? 1 : 0;
      const unsigned grid = (unsigned)std::min<int64_t>(n_users, TKS_CTAS_PER_SM * (int64_t)h.num_sms);
      k_topk_filter_staged<<<grid, TKS_THREADS, TKS_SMEM, st>>>(ta);
      CQL_LAUNCH_CHECK(&h);
      if (!stream) CQL_CUDA(cudaStreamSynchronize(st));
      return;
    }
    const int threads = 256;
    k_topk_filter<<<(unsigned)n_users, threads, (threads / 32) * 2 * k * sizeof(float) + SEEN_CACHE * sizeof(int32_t), st>>>(
        scores_dev, n_items, users_dev, items_dev, seen_indptr, seen_items, k, out_scores, out_items);
    CQL_LAUNCH_CHECK(&h);
    if (!stream) CQL_CUDA(cudaStreamSynchronize(st));
  });
}

int cql_offline_eval(cql_handle* ch, float return_threshold, cql_offline_sums* out, void* stream) {
  return guarded(ch, [&] {
    NvtxRange nvtx("cql_offline_eval");
    Handle& h = ch->h;
    CQL_REQUIRE(out != nullptr, "cql_offline_eval: NULL output");
    CQL_REQUIRE(h.n_trans > 0, "cql_offline_eval: no replay table loaded (build or load one, or evaluate a log)");
    CQL_REQUIRE(h.n_steps == 1, "cql_offline_eval: the table holds n-step rows (n_steps > 1); evaluate one-step rows");
    double s[OE_SUMS];
    with_precision(&h, [&](auto p) { offline_eval<decltype(p)::value>(&h, return_threshold, s, pick_stream(&h, stream)); });
    *out = cql_offline_sums{s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], h.n_trans, (int64_t)s[8], (int64_t)s[9]};
  });
}

}  // extern "C"
