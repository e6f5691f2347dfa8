// infer.cuh -- d3rlpy's per-observation inference (cql_predict_value, cql_sample_action; DESIGN.md section 1,
// "Inference").
//
// Pairs x = (user, item) run in chunks of INF_CHUNK rows through the update's launch_fwd, as cql_offline_eval drives it:
// k_inf_rows scales the ids into actor rows (or, with explicit actions, straight into critic rows), the actor forward
// gives mu and logstd, k_inf_greedy forms the critic rows (x, tanh(mu(x))), the critic forward gives every Q_c and
// k_inf_reduce leaves mean_c Q_c (and sigma) per pair through ens_mean_std, the offline scorers' arithmetic.
// k_inf_sample is the policy head of cql_sample_action.  Nothing of the handle's state is written.
#pragma once
#include "offline_eval.cuh"

namespace cql {

constexpr int64_t INF_CHUNK = 1 << 18;                      // pairs per forward chunk
constexpr uint64_t INF_SEED_XOR = 0xE7037ED1A0B428DBull;    // Philox key of cql_sample_action: seed ^ INF_SEED_XOR

// pair rows [c0, c0 + m): observations (user, item) observation-scaled as the update scales them; with explicit actions
// (raw rating units, action-scaled here) the critic rows XC, else the actor rows XA
__global__ void k_inf_rows(const int32_t* __restrict__ users, const int32_t* __restrict__ items,
                           const float* __restrict__ actions, int64_t c0, int m, const Prep prep, float4* __restrict__ XA,
                           float4* __restrict__ XC) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= m) return;
  const int64_t i = c0 + l;
  const float x0 = prep_fwd(prep.obs[0], (float)users[i]), x1 = prep_fwd(prep.obs[1], (float)items[i]);
  if (actions) XC[l] = make_float4(x0, x1, act_fwd(prep.act, actions[i]), 0.f);
  else XA[l] = make_float4(x0, x1, 0.f, 0.f);
}

// critic rows (x, pi(x)) with the greedy action in network space; tanh correctly rounded through double, as the
// offline scorers' and the update's TD-target rows
__global__ void k_inf_greedy(const float4* __restrict__ XA, const QSrc srcA, int m, float4* __restrict__ XC) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  const float4 x = XA[r];
  XC[r] = make_float4(x.x, x.y, (float)tanh((double)q_at(srcA, 0, r, 0)), 0.f);
}

// per pair: mean_c Q_c and, when sd is not null, the population std over the critics
__global__ void k_inf_reduce(const QSrc srcQ, int C, int64_t c0, int m, float* __restrict__ mean, float* __restrict__ sd) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  float s;
  mean[c0 + r] = ens_mean_std(srcQ, C, r, sd ? &s : nullptr);
  if (sd) sd[c0 + r] = s;
}

// the policy head: greedy reverse(tanh(mu)), or reverse(tanh(mu + exp(clamp(logstd)) * eps)) with eps the Box-Muller
// draw of Philox words 0 and 1 at (seed ^ INF_SEED_XOR, stream, pair index), as k_noise forms its Gaussian draws
__global__ void k_inf_sample(const QSrc srcA, int64_t c0, int m, int greedy, uint64_t key, uint64_t stream, int squash,
                             const Affine act, float* __restrict__ out) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  const float mu = q_at(srcA, 0, r, 0);
  float a;
  if (greedy) {
    a = (float)tanh((double)mu);
  } else {
    uint32_t w[4];
    Philox::gen(key, stream, (uint64_t)(c0 + r), w);
    const float eps = sqrtf(-2.f * logf(u01(w[0]))) * cospif(2.f * u01(w[1]));
    a = policy_sample(mu, clamp_ls(q_at(srcA, 0, r, 1)), eps, squash).a;
  }
  out[c0 + r] = act_rev(act, a);
}

// Host arrays in, host arrays out, on `st` (synchronised before returning).  predict: mean_host [n] and, when std_host
// is not null, std_host [n]; actions_host null = the greedy action.  sample: out_host [n] (greedy or Philox stream
// `stream`).  n > 0; the caller has validated the inputs.
template <Prec P>
void infer_pairs(Handle* h, const int32_t* users_host, const int32_t* items_host, const float* actions_host, int64_t n,
                 bool sample, int greedy, uint64_t stream, float* mean_host, float* std_host, cudaStream_t st) {
  const int C = h->C;
  DevTmp tmp(st);
  int32_t* users = tmp.get<int32_t>(n);
  int32_t* items = tmp.get<int32_t>(n);
  const float* actions = nullptr;
  CQL_CUDA(cudaMemcpyAsync(users, users_host, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  CQL_CUDA(cudaMemcpyAsync(items, items_host, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  if (actions_host) {
    float* a = tmp.get<float>(n);
    CQL_CUDA(cudaMemcpyAsync(a, actions_host, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    actions = a;
  }
  float* mean = tmp.get<float>(n);
  float* sd = std_host ? tmp.get<float>(n) : nullptr;
  const int cm = (int)std::min<int64_t>(INF_CHUNK, n);
  const bool need_actor = sample || !actions;
  float4* XA = need_actor ? tmp.get<float4>(cm) : nullptr;
  float* outA = need_actor ? tmp.get<float>(2 * (size_t)cm) : nullptr;
  float4* XC = sample ? nullptr : tmp.get<float4>(cm);
  float* QC = sample ? nullptr : tmp.get<float>((size_t)C * cm);
  const size_t part_floats = (size_t)Q_MAX_PARTS * std::max<size_t>(2 * (size_t)cm, sample ? 0 : (size_t)C * cm);
  float* part = tmp.get<float>(part_floats);
  for (int64_t c0 = 0; c0 < n; c0 += INF_CHUNK) {
    const int m = (int)std::min<int64_t>(INF_CHUNK, n - c0);
    const dim3 grid((m + 255) / 256);
    launch(h, st, PDL, k_inf_rows, grid, dim3(256), 0, (const int32_t*)users, (const int32_t*)items, actions, c0, m,
           h->prep, XA, XC);
    QSrc srcA;
    if (need_actor) {
      FwdJobs ja{};
      ja.n = 1;
      ja.j[0] = FwdJob{XA, h->net_params(slot_actor()), outA, nullptr, m, 1, 0};
      launch_fwd<P, 2, 2>(h, ja, st, &srcA, part, part_floats);
    }
    if (sample) {
      launch(h, st, PDL, k_inf_sample, grid, dim3(256), 0, srcA, c0, m, greedy, h->cfg.seed ^ INF_SEED_XOR, stream,
             h->cfg.squash, h->prep.act, mean);
      continue;
    }
    if (!actions) launch(h, st, PDL, k_inf_greedy, grid, dim3(256), 0, (const float4*)XA, srcA, m, XC);
    FwdJobs jc{};
    jc.n = 1;
    jc.j[0] = FwdJob{XC, h->net_params(slot_critic(0)), QC, nullptr, m, C, 0};
    QSrc srcQ;
    launch_fwd<P, 3, 1>(h, jc, st, &srcQ, part, part_floats);
    launch(h, st, PDL, k_inf_reduce, grid, dim3(256), 0, srcQ, C, c0, m, mean, sd);
  }
  CQL_CUDA(cudaMemcpyAsync(mean_host, mean, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  if (sd) CQL_CUDA(cudaMemcpyAsync(std_host, sd, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CQL_CUDA(cudaStreamSynchronize(st));
}

}  // namespace cql
