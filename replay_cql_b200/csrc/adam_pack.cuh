// adam_pack.cuh -- Adam + Polyak + operand packing of one group of networks in ONE launch (f16x3 path).
//
// After an Adam step every tensor-core operand copy of W2 must be refreshed: forward orientation (one-CTA and CTA-pair
// layouts) of the network and of its target copy, and the transposed orientation (both layouts) for the backward.
// Round 1 ran k_adam_polyak, then a pack kernel (now two, with the pair layouts): three dependent launches twice per
// update.  Here a CTA owns 8 consecutive W2 rows: it applies Adam + Polyak to them, packs them (row maximum by a warp
// reduction -> exact power-of-two row scale) for the forward layouts of network and target, and -- through a
// shared-memory tile -- writes the one 16-byte K chunk those 8 rows contribute to EVERY operand row of the transposed
// layouts.  A transposed operand row spans all 256 W2 rows (owned by 32 different CTAs), so its scale cannot be a row
// maximum here; it is ONE power of two per network from a bound on max|W2|: the maximum seen in the previous step
// (tracked with atomicMax in three rotating slots: read / accumulate / clear) plus 4 lr (an Adam step moves an entry by
// at most ~3.2 lr), with one spare binade.  The scale only has to keep fp16 in range: entries 2^-15 of the maximum are
// still represented to 2^-24 of the maximum (fp16 subnormals), far inside the 1e-4 gates (DESIGN.md section 3).
// The last CTA of each network handles the small tensors (W1, b1, b2, W3, b3) and the layer maxima (HMeta::wmax).
//
// At world size 1 the launch also sums the backward's gradient partials itself (k_reduce_grads_tc's fixed order, so the
// gradients are bit-identical): a W2 CTA sums the dW2 split partials of its own 8 rows, and the small tensors are spread
// over AP_SMALL_BLOCKS CTAs of 128 entries x 8 partial chunks each, whose layer maxima meet in global memory (the last of
// them writes HMeta::wmax).  One launch boundary and one dependent L2 round trip less per gradient group.
#pragma once
#include "mlp_tc_h2.cuh"

namespace cql {
namespace tc {

struct AdamPackNet {
  float* p;            // network slot (fp32 parameters)
  float* m;
  float* v;
  float* g;            // gradient (read; written when the launch sums the partials itself)
  float* targ;         // target slot
  uint8_t* fwd;        // packed forward, one-CTA layout (HCfg)            -- never null
  uint8_t* fwd2;       // packed forward, pair layout (H2Cfg)              -- null for the actor
  uint8_t* bwd;        // packed transposed, one-CTA layout                -- never null
  uint8_t* bwd2;       // packed transposed, pair layout                   -- null for the actor
  uint8_t* tfwd;       // target: packed forward, one-CTA layout
  uint8_t* tfwd2;      // target: packed forward, pair layout              -- null for the actor
  int* w2max;          // [3] rotating slots: float bits of max|W2|
};
struct AdamPackJobs {
  AdamPackNet n[CQL_MAX_CRITICS];
  int in_dim, out_dim;
  float lr, beta1, beta2, eps, tau;
  long long* step_inc;      // the update's LAST launch: completed-steps counter to increment (else null)
  DpPeer dp;                // data-parallel peers (world > 1: gradients = mean over the ranks' staging buffers)
  int dp_group;             // gradient group of this launch (1 critics, 2 actor)
  long long dp_off;         // offset of network 0 of this launch inside a staging buffer
  // world size 1: the gradient partials of the backward (small1 == nullptr: the gradient is read from n[i].g)
  const float* small1;      // [n_nets][slots1][SMALL_STRIDE]  W1 | b1  (bwd1)
  const float* small2;      // [n_nets][splits][SMALL_STRIDE]  b2 | W3 | b3  (bwd2)
  const float* pw2;         // [n_nets][splits][H * H]         W2  (bwd2)
  int slots1, splits;
  int* wmax_acc;            // [CQL_MAX_CRITICS][16] layer maxima across the small-tensor CTAs, then [CQL_MAX_CRITICS] tickets
};

__device__ __forceinline__ float adam_one(float& p, float& m, float& v, float g, float step_size, float bc2s, float beta1,
                                          float beta2, float eps) {
  const float mi = m + (g - m) * (1.f - beta1);
  const float vi = v * beta2 + (1.f - beta2) * g * g;
  m = mi;
  v = vi;
  p = p - step_size * (mi / (sqrtf(vi) / bc2s + eps));
  return p;
}

// one 16-byte chunk (8 consecutive K values of operand row n) -> hi|lo in the one-CTA and (optionally) the pair layout
__device__ __forceinline__ void store_chunk(const float (&x)[8], float s, uint8_t* one, uint8_t* pair, int n, int kc) {
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) split_h2(x[2 * i] * s, x[2 * i + 1] * s, hi[i], lo[i]);
  const uint4 h4 = make_uint4(hi[0], hi[1], hi[2], hi[3]), l4 = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  uint8_t* b = one + (size_t)(n / HCfg::NS) * HCfg::B_BYTES + chunk_off(HCfg::NS, n % HCfg::NS, kc);
  *reinterpret_cast<uint4*>(b) = h4;
  *reinterpret_cast<uint4*>(b + HCfg::B_TERM_BYTES) = l4;
  if (pair != nullptr) {
    *reinterpret_cast<uint4*>(pair + pair_chunk_off(n, kc, 0)) = h4;
    *reinterpret_cast<uint4*>(pair + pair_chunk_off(n, kc, 1)) = l4;
  }
}

constexpr int AP_ROWS = 8;                    // W2 rows per CTA
constexpr int AP_W2_BLOCKS = H / AP_ROWS;     // 32
constexpr int AP_SMALL_E = 128;               // small-tensor entries per CTA (x 8 partial chunks = 1024 threads)
// small-tensor CTAs per network when the launch sums the partials: W1 | b1 | b2 | W3 | b3 (1537 / 1538 entries)
constexpr int ap_small_blocks(int in_dim, int out_dim) { return (net_floats(in_dim, out_dim) - H * H + AP_SMALL_E - 1) / AP_SMALL_E; }

// The small tensors when the launch sums the partials (world size 1): CTA AP_W2_BLOCKS + s takes the compact entries
// [128 s, 128 s + 128) of W1 | b1 | b2 | W3 | b3; thread (chunk, entry) sums one of the 8 partial chunks, the first 128
// threads combine them in chunk order and apply Adam + Polyak to their entry (loads issued before the partials').
__device__ __forceinline__ void adam_small_fold(const AdamPackJobs& jobs, const AdamPackNet& nt, float step_size, float bc2s,
                                             int slot_clr, int* wm) {
  __shared__ float part[8][AP_SMALL_E];
  __shared__ int last;
  const int tid = threadIdx.x, in_dim = jobs.in_dim, out_dim = jobs.out_dim;
  const int w2_lo = off_W2(in_dim), n_e = net_floats(in_dim, out_dim) - H * H;
  const int s_blk = blockIdx.x - AP_W2_BLOCKS, n_blk = gridDim.x - AP_W2_BLOCKS;
  const int el = tid % AP_SMALL_E, chunk = tid / AP_SMALL_E;
  const int e = s_blk * AP_SMALL_E + el;                     // compact index: W1 | b1 then b2 | W3 | b3
  const int idx = e < w2_lo ? e : e + H * H;                 // index inside the network slot
  const bool own = tid < AP_SMALL_E && e < n_e;
  float p = 0.f, m = 0.f, v = 0.f, t = 0.f;
  if (own) { p = nt.p[idx]; m = nt.m[idx]; v = nt.v[idx]; t = nt.targ[idx]; }
  float s = 0.f;
  if (e < n_e) {                                             // small1 / small2 are indexed by the compact index
    if (e < w2_lo) s = chunk_sum8<float, 16>(jobs.small1 + (size_t)blockIdx.y * jobs.slots1 * SMALL_STRIDE + e, jobs.slots1, SMALL_STRIDE, chunk);
    else s = chunk_sum8<float, 16>(jobs.small2 + (size_t)blockIdx.y * jobs.splits * SMALL_STRIDE + e, jobs.splits, SMALL_STRIDE, chunk);
  }
  part[chunk][el] = s;
  if (tid < 16) wm[tid] = 0;
  if (s_blk == 0 && tid == 0) {
    nt.w2max[slot_clr] = 0;
    // the step counter (position in the epoch permutation, Philox stream); nothing in this launch reads it
    if (jobs.step_inc != nullptr && blockIdx.y == 0) *jobs.step_inc += 1;
  }
  __syncthreads();
  if (own) {
    float g = part[0][el];
#pragma unroll
    for (int c = 1; c < 8; ++c) g += part[c][el];
    nt.g[idx] = g;
    // adam_one + Polyak with every rounding written out, as the per-unit path below is compiled: there the second moment
    // is contracted as fma(g, g (1 - beta2), beta2 v) and the step as fma(-m / denom, step_size, p); left to the compiler
    // this context got fma(v, beta2, (1 - beta2) g g) -- one rounding apart, which Adam carries into every later step
    m = __fmaf_rn(__fsub_rn(g, m), __fsub_rn(1.f, jobs.beta1), m);
    v = __fmaf_rn(g, __fmul_rn(g, __fsub_rn(1.f, jobs.beta2)), __fmul_rn(jobs.beta2, v));
    p = __fmaf_rn(-__fdiv_rn(m, __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2s), jobs.eps)), step_size, p);
    t = __fmaf_rn(t, __fsub_rn(1.f, jobs.tau), __fmul_rn(jobs.tau, p));
    nt.p[idx] = p; nt.m[idx] = m; nt.v[idx] = v; nt.targ[idx] = t;
    // layer maxima for the operand generators: W1 columns -> wm[c], b1 -> wm[3], W3 rows -> wm[4 + o] (targets at + 8)
    int slot = -1;
    if (idx < off_b1(in_dim)) slot = idx % in_dim;
    else if (idx < w2_lo) slot = 3;
    else if (idx >= off_W3(in_dim) && idx < off_b3(in_dim, out_dim)) slot = 4 + (idx - off_W3(in_dim)) / H;
    if (slot >= 0) {
      atomicMax(&wm[slot], __float_as_int(fabsf(p)));
      atomicMax(&wm[8 + slot], __float_as_int(fabsf(t)));
    }
  }
  __syncthreads();
  int* acc = jobs.wmax_acc + blockIdx.y * 16;
  unsigned int* ticket = reinterpret_cast<unsigned int*>(jobs.wmax_acc + CQL_MAX_CRITICS * 16) + blockIdx.y;
  if (tid < 16 && wm[tid] != 0) atomicMax(&acc[tid], wm[tid]);
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const unsigned int k = atomicAdd(ticket, 1u);
    last = k == (unsigned int)n_blk - 1;
    if (last) *ticket = 0;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (tid < 8) {                                             // read and clear for the next launch
    const float w = __int_as_float(atomicExch(&acc[tid], 0)), wt = __int_as_float(atomicExch(&acc[8 + tid], 0));
    reinterpret_cast<HMeta*>(nt.fwd + HCfg::META_OFF)->wmax[tid] = w;
    reinterpret_cast<HMeta*>(nt.bwd + HCfg::META_OFF)->wmax[tid] = w;
    reinterpret_cast<HMeta*>(nt.tfwd + HCfg::META_OFF)->wmax[tid] = wt;
    if (nt.fwd2) reinterpret_cast<HMeta*>(nt.fwd2 + H2Cfg::META_OFF)->wmax[tid] = w;
    if (nt.bwd2) reinterpret_cast<HMeta*>(nt.bwd2 + H2Cfg::META_OFF)->wmax[tid] = w;
    if (nt.tfwd2) reinterpret_cast<HMeta*>(nt.tfwd2 + H2Cfg::META_OFF)->wmax[tid] = wt;
  }
}

__global__ void __launch_bounds__(1024, 1) k_adam_pack(const AdamPackJobs jobs, const StepInfo* __restrict__ si) {
  grid_dep_wait();
  __shared__ __align__(16) float tile[AP_ROWS][H + 4];   // (vector accesses: 16-byte alignment stated, not left to the layout)
  __shared__ int wm[16];
  const AdamPackNet nt = jobs.n[blockIdx.y];
  const int in_dim = jobs.in_dim, out_dim = jobs.out_dim;
  const float step_size = (float)((double)jobs.lr / si->bc1), bc2s = (float)si->bc2_sqrt;
  const int slot_rd = (int)(si->step % 3), slot_acc = (int)((si->step + 1) % 3), slot_clr = (int)((si->step + 2) % 3);
  const int tid = threadIdx.x, lane = tid & 31;
  const bool dp = jobs.dp.world > 1;
  const long long dpb = jobs.dp_off + (long long)blockIdx.y * NET_STRIDE;      // this network's element 0 in the gradient layout
  DpSlices sl{};
  if (dp) {
    // phase B of the exchange: this rank owns one slice of the group -- sum the ranks' contributions (rank order),
    // push the mean to everybody; then every block goes on to consume (phase C) whatever owner holds its values
    sl = dp_slices(jobs.dp, jobs.dp_off, (long long)gridDim.y * NET_STRIDE);
    dp_ll_owner_reduce(jobs.dp, jobs.dp_group, sl, jobs.n[0].g, ((long long)blockIdx.y * gridDim.x + blockIdx.x) * blockDim.x + tid,
                       (long long)gridDim.x * gridDim.y * blockDim.x);
  }
  if (blockIdx.x < AP_W2_BLOCKS) {
    // ---------------- 8 rows of W2: Adam + Polyak, forward packs, then the transposed K chunk ----------------
    // 1024 threads, TWO consecutive entries each (128 threads per row).  With 256 threads x 8 entries the kernel was bound
    // by the latency of each thread's 24 IEEE sqrt / divide sequences at 8 warps per SM (ncu r02: 11.4 us warm, issue
    // slots 20 %, 1390 warp instructions per warp).
    __shared__ __align__(16) float gw2[AP_ROWS][H];                 // data-parallel: the rows' mean gradients
    __shared__ float rmax[AP_ROWS][4], rmaxt[AP_ROWS][4];
    const int r8 = tid >> 7, c2 = tid & 127;
    const int n = blockIdx.x * AP_ROWS + r8;
    const size_t off = (size_t)off_W2(in_dim) + (size_t)n * H + c2 * 2;
    const float w2max_prev = __int_as_float(nt.w2max[slot_rd]);      // (read with the first loads, not after the barrier)
    float2 g;
    if (jobs.small1 == nullptr) g = *reinterpret_cast<const float2*>(nt.g + off);
    float2 m = *reinterpret_cast<const float2*>(nt.m + off), v = *reinterpret_cast<const float2*>(nt.v + off);
    float2 p = *reinterpret_cast<const float2*>(nt.p + off), t = *reinterpret_cast<const float2*>(nt.targ + off);
    if (jobs.small1 != nullptr) {                      // this thread's two entries summed over the dW2 split partials
      g = reduce8<float2, 4>(jobs.pw2 + (size_t)blockIdx.y * jobs.splits * H * H + (off - off_W2(in_dim)), jobs.splits,
                             (size_t)H * H);
      *reinterpret_cast<float2*>(nt.g + off) = g;
    }
    if (dp) {                                          // every fourth thread fetches the chunk's 8 means (from the slice's owner)
      if ((c2 & 3) == 0) {
        float4 g0 = *reinterpret_cast<const float4*>(nt.g + off), g1 = *reinterpret_cast<const float4*>(nt.g + off + 4);
        dp_ll_mean8(jobs.dp, jobs.dp_group, sl, dpb + (long long)off, g0, g1);
        *reinterpret_cast<float4*>(&gw2[r8][c2 * 2]) = g0;
        *reinterpret_cast<float4*>(&gw2[r8][c2 * 2 + 4]) = g1;
      }
      __syncthreads();
      g = *reinterpret_cast<const float2*>(&gw2[r8][c2 * 2]);
    }
    adam_one(p.x, m.x, v.x, g.x, step_size, bc2s, jobs.beta1, jobs.beta2, jobs.eps);
    adam_one(p.y, m.y, v.y, g.y, step_size, bc2s, jobs.beta1, jobs.beta2, jobs.eps);
    t.x = t.x * (1.f - jobs.tau) + jobs.tau * p.x;
    t.y = t.y * (1.f - jobs.tau) + jobs.tau * p.y;
    *reinterpret_cast<float2*>(nt.m + off) = m;
    *reinterpret_cast<float2*>(nt.v + off) = v;
    *reinterpret_cast<float2*>(nt.p + off) = p;
    *reinterpret_cast<float2*>(nt.targ + off) = t;
    *reinterpret_cast<float2*>(&tile[r8][c2 * 2]) = p;
    // forward orientation: operand row n = W2 row n, scale from the row maximum (4 warps per row)
    float mx = fmaxf(fabsf(p.x), fabsf(p.y)), mt = fmaxf(fabsf(t.x), fabsf(t.y));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, o));
    }
    if (lane == 0) { rmax[r8][(tid >> 5) & 3] = mx; rmaxt[r8][(tid >> 5) & 3] = mt; }
    __syncthreads();
    mx = fmaxf(fmaxf(rmax[r8][0], rmax[r8][1]), fmaxf(rmax[r8][2], rmax[r8][3]));
    mt = fmaxf(fmaxf(rmaxt[r8][0], rmaxt[r8][1]), fmaxf(rmaxt[r8][2], rmaxt[r8][3]));
    float s, inv_s, st, inv_st;
    pow2_scale(mx, s, inv_s);
    pow2_scale(mt, st, inv_st);
    {
      // this thread's quarter (4 bytes of hi, 4 bytes of lo) of the 16-byte chunk kc of operand row n
      const int kc = c2 >> 2, piece = (c2 & 3) * 4;
      uint32_t hi, lo, thi, tlo;
      split_h2(p.x * s, p.y * s, hi, lo);
      split_h2(t.x * st, t.y * st, thi, tlo);
      const size_t one_off = (size_t)(n / HCfg::NS) * HCfg::B_BYTES + chunk_off(HCfg::NS, n % HCfg::NS, kc) + piece;
      *reinterpret_cast<uint32_t*>(nt.fwd + one_off) = hi;
      *reinterpret_cast<uint32_t*>(nt.fwd + one_off + HCfg::B_TERM_BYTES) = lo;
      *reinterpret_cast<uint32_t*>(nt.tfwd + one_off) = thi;
      *reinterpret_cast<uint32_t*>(nt.tfwd + one_off + HCfg::B_TERM_BYTES) = tlo;
      if (nt.fwd2 != nullptr) {
        *reinterpret_cast<uint32_t*>(nt.fwd2 + pair_chunk_off(n, kc, 0) + piece) = hi;
        *reinterpret_cast<uint32_t*>(nt.fwd2 + pair_chunk_off(n, kc, 1) + piece) = lo;
      }
      if (nt.tfwd2 != nullptr) {
        *reinterpret_cast<uint32_t*>(nt.tfwd2 + pair_chunk_off(n, kc, 0) + piece) = thi;
        *reinterpret_cast<uint32_t*>(nt.tfwd2 + pair_chunk_off(n, kc, 1) + piece) = tlo;
      }
    }
    if (c2 == 0) {
      reinterpret_cast<HMeta*>(nt.fwd + HCfg::META_OFF)->inv_s[n] = inv_s;
      reinterpret_cast<HMeta*>(nt.tfwd + HCfg::META_OFF)->inv_s[n] = inv_st;
      if (nt.fwd2) reinterpret_cast<HMeta*>(nt.fwd2 + H2Cfg::META_OFF)->inv_s[n] = inv_s;
      if (nt.tfwd2) reinterpret_cast<HMeta*>(nt.tfwd2 + H2Cfg::META_OFF)->inv_s[n] = inv_st;
      atomicMax(&nt.w2max[slot_acc], __float_as_int(mx));
    }
    // (the barrier above already ordered the tile[] writes before the reads below)
    // transposed orientation: operand row n' = W2 column n', K index = W2 row: these 8 rows are K chunk blockIdx.x of
    // EVERY operand row.  One power-of-two scale per network (see the header of this file).
    if (tid < H) {
      const float bound = 2.f * (w2max_prev + 4.f * jobs.lr);
      float sT, inv_sT;
      pow2_scale(bound, sT, inv_sT);
      const int np = tid;
      float x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = tile[i][np];
      store_chunk(x, sT, nt.bwd, nt.bwd2, np, (int)blockIdx.x);
      if (blockIdx.x == 0) {
        reinterpret_cast<HMeta*>(nt.bwd + HCfg::META_OFF)->inv_s[np] = inv_sT;
        if (nt.bwd2) reinterpret_cast<HMeta*>(nt.bwd2 + H2Cfg::META_OFF)->inv_s[np] = inv_sT;
      }
    }
    if (dp) dp_consume_done(jobs.dp, jobs.dp_group, gridDim.x * gridDim.y);
    return;
  }
  if (jobs.small1 != nullptr) {
    adam_small_fold(jobs, nt, step_size, bc2s, slot_clr, wm);
    return;
  }
  if (tid >= 256) return;     // the small tensors are 256 threads' work (exited threads do not count at the barriers below)
  // ---------------- the small tensors: W1 | b1, b2, W3 | b3 (+ layer maxima for the operand generators) ----------------
  if (tid < 16) wm[tid] = 0;
  if (tid == 0) nt.w2max[slot_clr] = 0;
  __syncthreads();
  // data-parallel: the mean gradients of the small entries are fetched into shared memory FIRST, two 16-byte groups per
  // thread with all ranks' loads in flight together (one after the other, each entry would cost an NVLink round trip)
  __shared__ __align__(16) float gsm[2048];
  const int w2_lo = off_W2(in_dim), w2_hi = w2_lo + H * H;
  if (dp) {
    {                                                        // 2048 compact entries = 256 threads x two 16-byte groups
      const int c = tid * 8;
      const int idx = c < w2_lo ? c : c + H * H;             // compact index -> index inside the network slot (w2_lo % 8 == 0)
      if (idx + 7 < NET_STRIDE) {
        float4 a = *reinterpret_cast<const float4*>(nt.g + idx), b = *reinterpret_cast<const float4*>(nt.g + idx + 4);
        dp_ll_mean8(jobs.dp, jobs.dp_group, sl, dpb + idx, a, b);
        *reinterpret_cast<float4*>(gsm + c) = a;
        *reinterpret_cast<float4*>(gsm + c + 4) = b;
      }
    }
    __syncthreads();
  }
  auto grad_of = [&](int idx) { return dp ? gsm[idx < w2_lo ? idx : idx - H * H] : nt.g[idx]; };
  const int k = tid;                                        // 256 threads = 256 hidden units
  int idxs[8];
  int n_idx = 0;
  for (int c = 0; c < in_dim; ++c) idxs[n_idx++] = off_W1(in_dim) + k * in_dim + c;
  idxs[n_idx++] = off_b1(in_dim) + k;
  idxs[n_idx++] = off_b2(in_dim) + k;
  for (int o = 0; o < out_dim; ++o) idxs[n_idx++] = off_W3(in_dim) + o * H + k;
  // Every load of this thread (gradient, parameter, both moments, target: 5 x n_idx, plus b3 in the first out_dim
  // threads) is issued BEFORE the first store: with load / compute / store per entry the compiler cannot move a load
  // above the previous entry's stores (the pointers may alias), and this one CTA then walked through 7 dependent L2 round
  // trips -- with the launch skipped the update was 12 us shorter per k_adam_pack, most of it this chain (r02 skip test).
  const bool has_b3 = tid < out_dim;
  const int ib3 = off_b3(in_dim, out_dim) + tid;
  float gv[9], pv[9], mv[9], vv[9], tv[9];
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < n_idx) { gv[i] = grad_of(idxs[i]); pv[i] = nt.p[idxs[i]]; mv[i] = nt.m[idxs[i]]; vv[i] = nt.v[idxs[i]]; tv[i] = nt.targ[idxs[i]]; }
  if (has_b3) { gv[8] = grad_of(ib3); pv[8] = nt.p[ib3]; mv[8] = nt.m[ib3]; vv[8] = nt.v[ib3]; tv[8] = nt.targ[ib3]; }
#pragma unroll
  for (int i = 0; i < 9; ++i)
    if (i < n_idx || (i == 8 && has_b3)) {
      adam_one(pv[i], mv[i], vv[i], gv[i], step_size, bc2s, jobs.beta1, jobs.beta2, jobs.eps);
      tv[i] = tv[i] * (1.f - jobs.tau) + jobs.tau * pv[i];
    }
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < n_idx) { nt.p[idxs[i]] = pv[i]; nt.m[idxs[i]] = mv[i]; nt.v[idxs[i]] = vv[i]; nt.targ[idxs[i]] = tv[i]; }
  if (has_b3) { nt.p[ib3] = pv[8]; nt.m[ib3] = mv[8]; nt.v[ib3] = vv[8]; nt.targ[ib3] = tv[8]; }
  {
    // layer maxima for the operand generators: W1 columns -> wm[c], b1 -> wm[3], W3 rows -> wm[4 + o] (targets at + 8)
    int i = 0;
    for (int c = 0; c < in_dim; ++c, ++i) {
      atomicMax(&wm[c], __float_as_int(fabsf(pv[i])));
      atomicMax(&wm[8 + c], __float_as_int(fabsf(tv[i])));
    }
    atomicMax(&wm[3], __float_as_int(fabsf(pv[i])));
    atomicMax(&wm[8 + 3], __float_as_int(fabsf(tv[i])));
    i += 2;                                                   // (b2 has no maximum)
    for (int o = 0; o < out_dim; ++o, ++i) {
      atomicMax(&wm[4 + o], __float_as_int(fabsf(pv[i])));
      atomicMax(&wm[8 + 4 + o], __float_as_int(fabsf(tv[i])));
    }
  }
  __syncthreads();
  if (tid < 8) {
    const float w = __int_as_float(wm[tid]), wt = __int_as_float(wm[8 + tid]);
    reinterpret_cast<HMeta*>(nt.fwd + HCfg::META_OFF)->wmax[tid] = w;
    reinterpret_cast<HMeta*>(nt.bwd + HCfg::META_OFF)->wmax[tid] = w;
    reinterpret_cast<HMeta*>(nt.tfwd + HCfg::META_OFF)->wmax[tid] = wt;
    if (nt.fwd2) reinterpret_cast<HMeta*>(nt.fwd2 + H2Cfg::META_OFF)->wmax[tid] = w;
    if (nt.bwd2) reinterpret_cast<HMeta*>(nt.bwd2 + H2Cfg::META_OFF)->wmax[tid] = w;
    if (nt.tfwd2) reinterpret_cast<HMeta*>(nt.tfwd2 + H2Cfg::META_OFF)->wmax[tid] = wt;
  }
  // the step counter (position in the epoch permutation, Philox stream); nothing in this launch reads it
  if (jobs.step_inc != nullptr && blockIdx.y == 0 && tid == 0) *jobs.step_inc += 1;
  if (dp) dp_consume_done(jobs.dp, jobs.dp_group, gridDim.x * gridDim.y);
}

// after the weights were set from the host: every rotating slot of every network = its true max|W2|
__global__ void __launch_bounds__(256) k_w2max_init(const float* __restrict__ params, int n_slots, int* __restrict__ w2max) {
  const int slot = blockIdx.x;
  if (slot >= n_slots) return;
  const bool is_actor = slot == 0 || slot == n_slots / 2;      // [actor | critics | targ_actor | targ_critics]
  const float* W2 = params + (size_t)slot * NET_STRIDE + off_W2(is_actor ? 2 : 3);
  float mx = 0.f;
  for (int i = threadIdx.x; i < H * H; i += blockDim.x) mx = fmaxf(mx, fabsf(W2[i]));
  __shared__ int sm;
  if (threadIdx.x == 0) sm = 0;
  __syncthreads();
  atomicMax(&sm, __float_as_int(mx));
  __syncthreads();
  if (threadIdx.x < 3) w2max[slot * 4 + threadIdx.x] = sm;
}

}  // namespace tc
}  // namespace cql
