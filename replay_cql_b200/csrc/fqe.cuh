// fqe.cuh -- fitted Q evaluation (d3rlpy's FQE, DESIGN.md section 1): a critic-only update of fresh Q-networks toward
// y = r + gamma_k min_c Q_targ_c(s', pi(s')) (1 - term) under the frozen policy pi(x) = tanh(mu(x)).
//
// An FQE handle is an ordinary handle (cql_create) whose actor slot holds the policy and whose critic slots hold the FQE
// critics; only the update schedule differs.  One update: k_fqe_head (Adam bias terms, minibatch, actor rows of s'), the
// actor forward on s', k_fqe_prep (data rows (s, a), target rows (s', pi(s'))), one critic forward over both (critics and
// target critics), k_fqe_td (TD error, dQ, loss), the critic backward and the critics' Adam step, which also counts the
// update.  The target is a hard copy made by the host after the right updates (cql_fqe_update): the Adam step of every
// update writes its target copy into FqeState's sink, never into the target slots.
#pragma once
#include "update.cuh"

namespace cql {

// Adam bias corrections and the minibatch: rows_in (the caller's rows, staged raw) or the rows of the epoch permutation
// at position (completed updates) * B with rank 0 / world 1, so every rank of a data-parallel job draws the same rows.
// The rows are scaled here (the table stays raw); XA receives the actor rows of s'.  FQE has no noise.
__global__ void k_fqe_head(const float4* __restrict__ table, int64_t n_trans, const float4* __restrict__ rows_in,
                           const long long* __restrict__ step_dev, StepInfo* __restrict__ info, float beta1, float beta2,
                           int B, uint64_t seed, float4* __restrict__ batch, float4* __restrict__ XA, const Prep prep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const long long done = *step_dev;
  if (i == 0) {
    const long long t = done + 1;
    info->step = t;
    info->bc1 = 1.0 - pow((double)beta1, (double)t);
    info->bc2_sqrt = sqrt(1.0 - pow((double)beta2, (double)t));
  }
  if (i >= B) return;
  float4 a, b;
  if (rows_in) {
    a = rows_in[2 * i];
    b = rows_in[2 * i + 1];
  } else {
    const int64_t t = stream_index((int64_t)done * B + i, n_trans, B, seed);
    a = __ldg(table + 2 * t);
    b = __ldg(table + 2 * t + 1);
  }
  if (prep.any()) { a = prep_row0(prep, a); b = prep_row1(prep, b); }
  batch[2 * i] = a;
  batch[2 * i + 1] = b;
  XA[i] = make_float4(b.x, b.y, 0.f, 0.f);
}

// critic data rows (s, a) and target rows (s', pi(s')); tanh correctly rounded through double, as k_prep's TD-target row
__global__ void k_fqe_prep(const float4* __restrict__ batch, const QSrc srcA, int B, float4* __restrict__ XC,
                           float4* __restrict__ XT) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float mu = q_at(srcA, 0, b, 0);
  const float4 r0 = batch[2 * b], r1 = batch[2 * b + 1];
  XC[b] = make_float4(r0.x, r0.y, r0.z, 0.f);
  XT[b] = make_float4(r1.x, r1.y, (float)tanh((double)mu), 0.f);
}

constexpr int FQE_TD_THREADS = 256;

// One thread per (critic, row): err = Q_c(s, a) - y and dQ = 2 err / B (k_scalar_adam_dq's data-row term without the
// conservative coefficient).  The block that finishes last sums the loss sum_c mean_b err^2 in a fixed order (critic by
// critic, block_sum over rows), so a given batch always gives the same bits.
__global__ void __launch_bounds__(FQE_TD_THREADS) k_fqe_td(const float4* __restrict__ batch, const QSrc srcC, const QSrc srcT,
                                                           int B, int C, float gamma, int nstep, float* __restrict__ dQ,
                                                           float* __restrict__ sq, float* __restrict__ loss,
                                                           unsigned int* __restrict__ ticket) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < C * B) {
    const int c = p / B, b = p % B;
    float qt = q_at(srcT, 0, b);
    for (int c2 = 1; c2 < C; ++c2) qt = fminf(qt, q_at(srcT, c2, b));
    const float4 r0 = batch[2 * b], r1 = batch[2 * b + 1];
    const float disc = nstep ? r1.w : gamma;
    const float y = r0.w + disc * qt * (1.f - r1.z);
    const float err = q_at(srcC, c, b) - y;
    dQ[p] = 2.f * err / (float)B;
    sq[p] = err * err;
  }
  __shared__ bool last;
  __shared__ float red[FQE_TD_THREADS / 32];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    last = t == gridDim.x - 1;
    if (last) *ticket = 0;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  float total = 0.f;
  for (int c = 0; c < C; ++c) {
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += FQE_TD_THREADS) s += sq[(int64_t)c * B + b];
    total += block_sum<FQE_TD_THREADS>(s, red) / (float)B;
  }
  if (threadIdx.x == 0) *loss = total;
}

// FQE mode of a handle (cql_fqe_enable): the target schedule and the scratch the ordinary updates' Adam step writes its
// target copy to
struct FqeState {
  bool on = false;
  int interval = 100;        // target_update_interval: the target is synchronised after updates 1, 1 + I, 1 + 2 I, ...
  TargetSink sink{};
};

// the device slots FQE keeps its scalars in (the CQL-only loss buffers are unused on an FQE handle)
inline float* fqe_loss(Handle* h) { return h->loss_sums + 4; }
inline unsigned int* fqe_ticket(Handle* h) { return reinterpret_cast<unsigned int*>(h->loss_sums + 15); }

inline BwdJob fqe_bwd_job(Handle* h) {
  const int splits = std::max(1, std::min(tiles_of(h->B), (2 * h->num_sms) / (4 * h->C)));
  return BwdJob{h->XC, h->dQ, h->h2C, h->net_params(slot_critic(0)), h->smallC, nullptr, h->pw2C, h->B, h->C, splits};
}

// one FQE update (launches counted in Handle::launches, DESIGN.md section 5); rows_in: the caller's staged rows, or
// nullptr to sample the replay table
template <Prec P>
inline void fqe_step(Handle* h, const FqeState& fq, cudaStream_t st, const float4* rows_in) {
  NvtxRange nvtx("cql.fqe.update");
  const int B = h->B, C = h->C;
  const cql_config& c = h->cfg;
  CQL_REQUIRE(rows_in || h->n_trans > 0, "cql_fqe_update: no transitions loaded");
  const float4* batch4 = reinterpret_cast<const float4*>(h->batch);
  launch(h, st, PLAIN, k_fqe_head, dim3((B + 255) / 256), dim3(256), 0, reinterpret_cast<const float4*>(h->table), h->n_trans,
         rows_in, h->step_dev, h->stepinfo, c.beta1, c.beta2, B, c.seed, reinterpret_cast<float4*>(h->batch), h->XA, h->prep);
  FwdJobs ja{};
  ja.n = 1;
  ja.j[0] = FwdJob{h->XA, h->net_params(slot_actor()), h->outA, nullptr, B, 1, 0};
  QSrc srcA;
  launch_fwd<P, 2, 2>(h, ja, st, &srcA);
  launch(h, st, PDL, k_fqe_prep, dim3((B + 255) / 256), dim3(256), 0, batch4, srcA, B, h->XC, h->XT);
  FwdJobs jq{};
  jq.n = 2;
  jq.j[0] = FwdJob{h->XC, h->net_params(slot_critic(0)), h->QC, h->h2C, B, C, 0};
  jq.j[1] = FwdJob{h->XT, h->net_params(slot_targ_critic(C, 0)), h->QT, nullptr, B, C, 0};
  QSrc srcQ[2];
  launch_fwd<P, 3, 1>(h, jq, st, srcQ);
  launch(h, st, PDL, k_fqe_td, dim3((C * B + FQE_TD_THREADS - 1) / FQE_TD_THREADS), dim3(FQE_TD_THREADS), 0, batch4, srcQ[0],
         srcQ[1], B, C, c.gamma, h->n_steps > 1 ? 1 : 0, h->dQ, h->pairv, fqe_loss(h), fqe_ticket(h));
  const BwdJob jb = fqe_bwd_job(h);
  const BwdPlan plan = launch_bwd<P, 3, 1, true, false>(h, jb, h->g_critics(), st);
  optimizer_step<P>(h, critic_group(h), plan, st, true, &fq.sink);
}

// after a synchronising update: the target critics (parameters and packed operand copies) := the critics, bit for bit
inline void fqe_sync_target(Handle* h, cudaStream_t st) {
  const int C = h->C;
  CQL_CUDA(cudaMemcpyAsync(h->net_params(slot_targ_critic(C, 0)), h->net_params(slot_critic(0)),
                           (size_t)C * NET_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (h->packed_fwd)
    CQL_CUDA(cudaMemcpyAsync(h->packed_fwd + (size_t)slot_targ_critic(C, 0) * h->packed_net_bytes,
                             h->packed_fwd + (size_t)slot_critic(0) * h->packed_net_bytes, (size_t)C * h->packed_net_bytes,
                             cudaMemcpyDeviceToDevice, st));
  if (h->packed_fwd2)
    CQL_CUDA(cudaMemcpyAsync(h->packed_fwd2 + (size_t)slot_targ_critic(C, 0) * h->packed_net_bytes2,
                             h->packed_fwd2 + (size_t)slot_critic(0) * h->packed_net_bytes2, (size_t)C * h->packed_net_bytes2,
                             cudaMemcpyDeviceToDevice, st));
}

}  // namespace cql
