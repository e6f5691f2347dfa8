// mlp_tc_h.cuh -- FP32-grade hidden-layer contraction on the fp16 tensor-core path ("f16x3").
//
// Same idea as the tf32 3-term split (mlp_tc_ts.cuh): x = x_hi + x_lo with 11-bit significands each, and
// a_lo*w_hi + a_hi*w_lo + a_hi*w_hi accumulated in FP32 tensor memory.  fp16 has the SAME significand width as
// tf32 (10 explicit bits), so the split is equally exact -- but kind::f16 runs at twice the kind::tf32 rate and its
// operands are half as wide, so a 128-column W2 slice (hi + lo) fits in the 128 KB resident operand buffer: a row
// tile is visited by 2 (net, slice) work items instead of 4, halving the producers' layer-1 work as well.
//
// What fp16 lacks is exponent range (5 bits).  Every operand row therefore carries an exact power-of-two scale:
//   * A (activations, one row per thread): s_m = 2^e from a bound on the row, |H1[m][k]| <= sum_c |x_c| max_k|W1[k][c]|
//     + max_k|b1[k]|, chosen so that the row stays below 2^15;
//   * B (W2 rows, packed once per Adam step): s_n = 2^e from the row maximum, stored with the packed operand;
// the epilogue multiplies the accumulator by 1/(s_m s_n) -- exact.  Small entries of a scaled row fall into fp16
// subnormals, whose spacing 2^-24 is still 2^-39 of the row maximum: the representation error is
// max(2^-22 |x|, 2^-39 max|row|), far inside the 1e-4 gates.
//
// TMEM columns: [0,256) two 128-column accumulators; [256,512) four A stages of 64 K: hi[32 cols] | lo[32 cols]
// (two fp16 per 32-bit column).  warps 0-7 epilogue (group g = warp / 4 drains accumulator g, i.e. every other
// work item -- the epilogue was the bottleneck with one group), 8-23 producers, 24 MMA issuer.
#pragma once
#include <cuda_fp16.h>
#include "mlp_tc.cuh"
#include "mlp_tc_bwd1.cuh"
#include "mlp_tc_bwd2.cuh"

namespace cql {
namespace tc {

template <int NEW_, int NS_ = 128>
struct HCfgT {
  static constexpr int ES = 2, EPC = 8, UK = 16;
  static constexpr int NS = NS_;                      // output columns per work item (128; 32 for the small launches)
  static constexpr int SLICES = H / NS;               // 2
  static constexpr int NPW = 16;
  static constexpr int KC = 64;                       // K per stage
  static constexpr int STAGES = 4;
  static constexpr int NCHUNK = H / KC;               // 4
  static constexpr int KPW = KC / (NPW / 4);          // K elements per producer warp per stage: 16 = 8 columns
  static constexpr int NEW = NEW_;                    // epilogue warps: 8 = two groups of 4, one per TMEM accumulator
  static constexpr int MMA_WARP = NEW + NPW;
  static constexpr int THREADS = (NEW + 1 + NPW) * 32;   // 800
  static constexpr int PROD_THREADS = NPW * 32;
  static constexpr uint32_t B_TERM_BYTES = NS * H * ES;            // 64 KB
  static constexpr uint32_t B_BYTES = 2 * B_TERM_BYTES;            // 128 KB (hi | lo)
  static constexpr size_t META_OFF = (size_t)SLICES * B_BYTES;     // float inv_s[256] | float wmax[8]
  static constexpr size_t PACKED_NET_BYTES = META_OFF + 2048;
  static constexpr uint32_t A_COL0 = 256;             // after the two accumulators (2 x NS <= 256 columns)
  static constexpr uint32_t A_STAGE_COLS = KC;        // 32 hi + 32 lo columns
  static constexpr uint32_t A_LO_COLS = KC / 2;
  static constexpr uint32_t TMEM_ALLOC = 512;
  static constexpr uint32_t OFF_B = 0;
  static constexpr uint32_t OFF_W1 = B_BYTES;                  // float4[256] pair-packed W1|b1
  static constexpr uint32_t OFF_EB = OFF_W1 + H * 16;          // float4[2][NS] (one copy per epilogue group)
  static constexpr uint32_t OFF_BAR = OFF_EB + 2 * NS * 16;
  static constexpr uint32_t N_BARS = 2 * STAGES + 4 + 2;
  static constexpr uint32_t OFF_SLOT = OFF_BAR + N_BARS * 8;
  static constexpr uint32_t OFF_FLUSH = OFF_SLOT + 16;         // bwd1: float[2 groups][4 warps][16][32] dW1/db1 partials
  static constexpr uint32_t OFF_RED = OFF_FLUSH + 2 * 4 * 16 * 32 * 4;   // bwd1: per epilogue warp float[32][33] + float4[32]
  static constexpr uint32_t RED_WARP_BYTES = 32 * 33 * 4 + 32 * 16;
  static constexpr uint32_t SMEM_BYTES = OFF_RED + NEW_ * RED_WARP_BYTES;
};
using HCfg = HCfgT<8>;     // update kernels; ALSO the layout of a packed net in global memory (128-row slices)
using HCfgS = HCfgT<8, 32>;   // small launches (B rows): 32-column work items, four times as many CTAs
using HCfg4 = HCfgT<4>;    // scorer (one epilogue group keeps the per-row state)

// The resident operand of a work item: NS rows x 256 K, hi | lo, compact K-major layout in shared memory.  The packed net
// in global memory is laid out in 128-row slices (HCfg); a 32-row sub-slice of it is 2 x 32 pieces of 512 bytes.
template <class C>
__device__ __forceinline__ void load_operand_slice(uint8_t* Bs, const uint8_t* packed_net, int slice, uint64_t* bar) {
  if constexpr (C::NS == HCfg::NS) {
    const uint8_t* src = packed_net + (size_t)slice * HCfg::B_BYTES;
    mbar_arrive_expect_tx(bar, C::B_BYTES);
    for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bar);
  } else {
    constexpr int PER = HCfg::NS / C::NS;                                  // sub-slices per 128-row slice
    const uint8_t* src = packed_net + (size_t)(slice / PER) * HCfg::B_BYTES + (size_t)(slice % PER) * (C::NS * 16);
    mbar_arrive_expect_tx(bar, C::B_BYTES);
    for (int term = 0; term < 2; ++term)
      for (int kc = 0; kc < H / 8; ++kc)
        bulk_g2s(Bs + term * C::B_TERM_BYTES + kc * (C::NS * 16), src + (size_t)term * HCfg::B_TERM_BYTES + (size_t)kc * (HCfg::NS * 16),
                 C::NS * 16, bar);
  }
}

// meta block of a packed net
struct HMeta {
  float inv_s[H];     // 1 / scale of operand row n
  float wmax[8];      // max|W1[:,0]|, max|W1[:,1]|, max|W1[:,2]|, max|b1|, max|W3[0,:]|, max|W3[1,:]|, -, -
};

// power-of-two scale that brings `bound` below 2^15, and its inverse (bit arithmetic on the exponent; exact)
__device__ __forceinline__ void pow2_scale(float bound, float& s, float& inv_s) {
  int e = (int)((__float_as_uint(bound) >> 23) & 0xffu);      // bound in [2^(e-127), 2^(e-126))
  e = max(e, 20);                                             // zero / denormal rows: any finite scale works
  s = __uint_as_float((uint32_t)(268 - e) << 23);             // 2^(141-e):  bound * s < 2^15
  inv_s = __uint_as_float((uint32_t)(e - 14) << 23);          // 2^(e-141)
}

// x (already scaled) -> fp16 hi and fp16 lo = rn(x - hi), two values per 32-bit word (low half = first value)
__device__ __forceinline__ void split_h2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// Producer-side split, cheaper on the FMA pipe (which bounds the operand generators: 0.5 warp-instr/clk/SMSP):
// hi = x truncated to an 11-bit significand by masking (ALU pipe, exactly representable in fp16 above 2^-14),
// lo = rn_fp16(x - hi) with ONE packed subtraction.  x - hi has <= 13 significant bits, so |x - hi - lo| <= 2^-22 |x|.
__device__ __forceinline__ void split_h2_trunc(float2 x, uint32_t& hi, uint32_t& lo) {
  const float h0 = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
  const float h1 = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
  float2 l;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "sub.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(l.x), "=f"(l.y)
      : "f"(x.x), "f"(x.y), "f"(h0), "f"(h1));
  const __half2 hh = __floats2half2_rn(h0, h1);
  const __half2 ll = __floats2half2_rn(l.x, l.y);
  hi = *reinterpret_cast<const uint32_t*>(&hh);
  lo = *reinterpret_cast<const uint32_t*>(&ll);
}

// packed fp32x2 multiply
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "mul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

// Packed weights, per net: per slice [term hi|lo][kchunk16 (8 fp16)][n_local/8][8][16 B] (chunk_off with rows = NS),
// then HMeta.  One WARP per operand row n (32 lanes = the 32 K-chunks), so the row maximum is a warp reduction.
// transpose=0: B[n][k] = W2[n][k] (forward);  1: B[n][k] = W2[k][n] (backward dH1 = dZ2 W2).
__global__ void __launch_bounds__(256) k_pack_multi_h(const PackJobs jobs, int out_dim_actor) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
 
  using C = HCfg;
  const PackJobs::J jb = jobs.j[blockIdx.y];
  const int c = blockIdx.x * blockDim.x + threadIdx.x;        // 16-byte chunk id: n * 32 + kc
  const int n = c >> 5, kc = c & 31;
  const float* W2 = jb.net + off_W2(jb.in_dim);
  float v[8];
  float mx = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = kc * 8 + i;
    v[i] = jb.transpose ? W2[(size_t)k * H + n] : W2[(size_t)n * H + k];
    mx = fmaxf(mx, fabsf(v[i]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s, inv_s;
  pow2_scale(mx, s, inv_s);
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) split_h2(v[2 * i] * s, v[2 * i + 1] * s, hi[i], lo[i]);
  const int slice = n / C::NS, nl = n % C::NS;
  uint8_t* base = jb.dst + (size_t)slice * C::B_BYTES + chunk_off(C::NS, nl, kc);
  *reinterpret_cast<uint4*>(base) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(base + C::B_TERM_BYTES) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  HMeta* meta = reinterpret_cast<HMeta*>(jb.dst + C::META_OFF);
  if (kc == 0) meta->inv_s[n] = inv_s;
  if (blockIdx.x == 0) {                                      // maxima of the small layers (scales of the A rows)
    __shared__ int wm[8];
    if (threadIdx.x < 8) wm[threadIdx.x] = 0;
    __syncthreads();
    const int out_dim = jb.in_dim == 2 ? out_dim_actor : 1;
    const int k = threadIdx.x;                                // 256 threads = 256 hidden units
    const float* W1 = jb.net + off_W1(jb.in_dim);
    for (int cc = 0; cc < jb.in_dim; ++cc) atomicMax(&wm[cc], __float_as_int(fabsf(W1[k * jb.in_dim + cc])));
    atomicMax(&wm[3], __float_as_int(fabsf(jb.net[off_b1(jb.in_dim) + k])));
    for (int o = 0; o < out_dim; ++o) atomicMax(&wm[4 + o], __float_as_int(fabsf(jb.net[off_W3(jb.in_dim) + o * H + k])));
    __syncthreads();
    if (threadIdx.x < 8) meta->wmax[threadIdx.x] = __int_as_float(wm[threadIdx.x]);
  }
}

constexpr int FWD_H2_COST = 13;     // relative cost of a forward item that stores H2 (plain item = 10)

struct HItem { int job, net, slice, tile, pair_id; };
template <int SLICES = HCfg::SLICES>
__device__ __forceinline__ HItem decode_item_h(const TcFwdJobs& jobs, int item) {
  HItem it;
  it.job = 0;
  while (it.job + 1 < jobs.n && item >= jobs.item_begin[it.job + 1]) ++it.job;
  const int local = item - jobs.item_begin[it.job];
  const int tiles = (jobs.j[it.job].rows + TM - 1) / TM;
  const int pair = local / tiles;
  it.tile = local % tiles;
  it.net = pair / SLICES;
  it.slice = pair % SLICES;
  it.pair_id = it.job * 64 + pair;
  return it;
}

// bound on |H1[row][:]| from the row's input and the per-net maxima of |W1| columns and |b1|
__device__ __forceinline__ float h1_row_bound(const float4& x, const float4& wm) {
  return fmaf(fabsf(x.x), wm.x, fmaf(fabsf(x.y), wm.y, fmaf(fabsf(x.z), wm.z, wm.w)));
}

template <int IN, int OUT, class C = HCfg>
__global__ void __launch_bounds__(HCfg::THREADS, 1) tc_fwd_h_kernel(const TcFwdJobs jobs) {
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + C::OFF_B;
  float4* w1p = reinterpret_cast<float4*>(sm + C::OFF_W1);   // [k/2][2]: {wx_k,wx_k1,wy_k,wy_k1}, {wz_k,wz_k1,b_k,b_k1}
  float4* ebs = reinterpret_cast<float4*>(sm + C::OFF_EB);   // [2][NS]: b2, w3_0, w3_1, 1 / s_n
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bload = tempty + 2;
  uint64_t* drain = bload + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // contiguous item range per CTA, balanced by COST: an item whose epilogue also stores H2 is ~30 % more expensive,
  // and those items are contiguous (one job), so an equal-count split leaves their CTAs as the tail of the launch
  int item_lo, item_hi;
  {
    long long cb[4];
    int wj[3];
    cb[0] = 0;
    for (int j = 0; j < jobs.n; ++j) {
      wj[j] = jobs.j[j].h2 != nullptr ? (jobs.h2_cost > 0 ? jobs.h2_cost : FWD_H2_COST) : 10;
      cb[j + 1] = cb[j] + (long long)(jobs.item_begin[j + 1] - jobs.item_begin[j]) * wj[j];
    }
    auto item_at = [&](long long cost) {
      int j = 0;
      while (j + 1 < jobs.n && cost >= cb[j + 1]) ++j;
      const int it = jobs.item_begin[j] + (int)((cost - cb[j]) / wj[j]);
      return it < jobs.item_begin[j + 1] ? it : jobs.item_begin[j + 1];
    };
    const long long total_cost = cb[jobs.n];
    item_lo = blockIdx.x == 0 ? 0 : item_at(total_cost * blockIdx.x / gridDim.x);
    item_hi = blockIdx.x == gridDim.x - 1 ? jobs.item_begin[jobs.n] : item_at(total_cost * (blockIdx.x + 1) / gridDim.x);
  }

  if (warp == C::MMA_WARP) {
    tmem_alloc(slot, C::TMEM_ALLOC);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], C::NPW); mbar_init(&empty[s], 1); }
      for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4); }
      mbar_init(bload, 1);
      mbar_init(drain, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;
  grid_dep_wait();            // everything above overlapped the predecessor's tail (programmatic dependent launch)

  if (warp == C::MMA_WARP) {
    // =============================== MMA issuer ===============================
    const uint32_t idesc = instr_desc(FMT_F16, TM, C::NS);
    const uint32_t b_lbo = C::NS * 16;
    const uint32_t b_base = smem_u32(Bs);
    int cur_pair = -1;
    uint32_t it = 0, nb = 0, nd = 0, tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const HItem ii = decode_item_h<C::SLICES>(jobs, item);
      if (ii.pair_id != cur_pair) {
        if (cur_pair >= 0) {
          if (elect_one()) umma_commit(drain);
          __syncwarp();
          mbar_wait(drain, nd & 1);
          ++nd;
        }
        const TcFwdJob& jb = jobs.j[ii.job];
        if (elect_one()) load_operand_slice<C>(Bs, jb.packed + (size_t)ii.net * HCfg::PACKED_NET_BYTES, ii.slice, bload);
        __syncwarp();
        mbar_wait(bload, nb & 1);
        ++nb;
        cur_pair = ii.pair_id;
      }
      const uint32_t acc = tcount & 1;
      mbar_wait(&tempty[acc], ((tcount >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem + acc * C::NS;
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        const uint32_t s = it % C::STAGES;
        mbar_wait(&full[s], (it / C::STAGES) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_stage = tmem + C::A_COL0 + s * C::A_STAGE_COLS;
#pragma unroll
          for (int j = 0; j < C::KC / C::UK; ++j) {
            const uint32_t g = c * (C::KC / C::UK) + j;
            const uint64_t b_hi = smem_desc(b_base + 2 * g * b_lbo, b_lbo, 128);
            const uint64_t b_lo = smem_desc(b_base + C::B_TERM_BYTES + 2 * g * b_lbo, b_lbo, 128);
            const uint32_t a_hi = a_stage + j * 8, a_lo = a_hi + C::A_LO_COLS;     // 8 columns = 16 fp16 per MMA
            umma_ts<false>(d_tmem, a_lo, b_hi, idesc, (c == 0 && j == 0) ? 0u : 1u);
            umma_ts<false>(d_tmem, a_hi, b_lo, idesc, 1u);
            umma_ts<false>(d_tmem, a_hi, b_hi, idesc, 1u);
          }
          umma_commit(&empty[s]);
          if (c == C::NCHUNK - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
      }
      ++tcount;
    }
  } else if (warp >= C::NEW) {
    // =============================== producers: layer 1 -> scaled fp16 hi|lo -> TMEM ===============================
    const int pw = warp - C::NEW, ptid = tid - C::NEW * 32;
    const int kq = pw >> 2;                                        // which K quarter of every stage
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + kq * (C::KPW / 2);
    int cur_netkey = -1;
    float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t it = 0;
    auto load_x = [&](const HItem& ni) {
      const TcFwdJob& nj = jobs.j[ni.job];
      const int r = ni.tile * TM + (warp & 3) * 32 + lane;
      return r < nj.rows ? __ldg(nj.X + r) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    float4 x_next = make_float4(0.f, 0.f, 0.f, 0.f);
    HItem ii_next = item_lo < item_hi ? decode_item_h<C::SLICES>(jobs, item_lo) : HItem{};   // one decode (integer division) per item
    for (int item = item_lo; item < item_hi; ++item) {
      const HItem ii = ii_next;
      if (item + 1 < item_hi) ii_next = decode_item_h<C::SLICES>(jobs, item + 1);
      const TcFwdJob& jb = jobs.j[ii.job];
      const int netkey = ii.job * 64 + ii.net;
      if (netkey != cur_netkey) {
        cur_netkey = netkey;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        const float* net = jb.params + (size_t)ii.net * NET_STRIDE;
        for (int pr = ptid; pr < H / 2; pr += C::PROD_THREADS) {
          const int k = 2 * pr;
          const float* wa = net + off_W1(IN) + k * IN;
          const float* wb = wa + IN;
          w1p[2 * pr] = make_float4(wa[0], wb[0], wa[1], wb[1]);
          w1p[2 * pr + 1] = make_float4(IN == 3 ? wa[2] : 0.f, IN == 3 ? wb[2] : 0.f, net[off_b1(IN) + k], net[off_b1(IN) + k + 1]);
        }
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packed + (size_t)ii.net * HCfg::PACKED_NET_BYTES + HCfg::META_OFF);
        wm = make_float4(__ldg(&meta->wmax[0]), __ldg(&meta->wmax[1]), IN == 3 ? __ldg(&meta->wmax[2]) : 0.f, __ldg(&meta->wmax[3]));
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      }
      // this item's input row was prefetched while the previous item was generated; fetch the next one now
      const float4 x = (item == item_lo) ? load_x(ii) : x_next;
      if (item + 1 < item_hi) x_next = load_x(ii_next);
      float sa, inv_sa;
      pow2_scale(h1_row_bound(x, wm), sa, inv_sa);
      const float2 xx = make_float2(x.x, x.x), xy = make_float2(x.y, x.y), xz = make_float2(x.z, x.z), ss = make_float2(sa, sa);
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        const uint32_t s = it % C::STAGES;
        uint32_t hi[C::KPW / 2], lo[C::KPW / 2];
#pragma unroll
        for (int pp = 0; pp < C::KPW / 2; ++pp) {
          const int pr = (c * C::KC + kq * C::KPW) / 2 + pp;
          const float4 wA = w1p[2 * pr], wB = w1p[2 * pr + 1];
          float2 v = ffma2(xx, make_float2(wA.x, wA.y), make_float2(wB.z, wB.w));   // chain starts from the bias
          v = ffma2(xy, make_float2(wA.z, wA.w), v);
          if (IN == 3) v = ffma2(xz, make_float2(wB.x, wB.y), v);
          v = fmul2(make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f)), ss);             // exact: power-of-two scale
          split_h2_trunc(v, hi[pp], lo[pp]);
        }
        mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);          // values are ready before the slot is: wait late
        tc_fence_after();
        tmem_st8(lane_base + s * C::A_STAGE_COLS, hi);
        tmem_st8(lane_base + s * C::A_STAGE_COLS + C::A_LO_COLS, lo);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
  } else {
    // =============================== epilogue: TMEM -> unscale -> layer 3 (+ H2) ===============================
    const int grp = warp >> 2, qw = warp & 3, gtid = tid & 127;          // group = accumulator, qw = TMEM lane quarter
    float4* ebg = ebs + grp * C::NS;
    float2* efg = reinterpret_cast<float2*>(sm + C::OFF_FLUSH) + grp * C::NS;   // folded constants (region used by bwd1 only)
    int cur_pair = -1;
    const int row_in_tile = qw * 32 + lane;
    float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int item = item_lo + grp; item < item_hi; item += 2) {
      const uint32_t tcount = (uint32_t)(item - item_lo);
      const HItem ii = decode_item_h<C::SLICES>(jobs, item);
      const TcFwdJob& jb = jobs.j[ii.job];
      if (ii.pair_id != cur_pair) {
        cur_pair = ii.pair_id;
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp));
        const float* net = jb.params + (size_t)ii.net * NET_STRIDE;
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packed + (size_t)ii.net * HCfg::PACKED_NET_BYTES + HCfg::META_OFF);
        for (int cidx = gtid; cidx < C::NS; cidx += 128) {
          const int col = ii.slice * C::NS + cidx;
          const float inv_n = __ldg(&meta->inv_s[col]);
          ebg[cidx] = make_float4(net[off_b2(IN) + col], net[off_W3(IN) + col],
                                  OUT == 2 ? net[off_W3(IN) + H + col] : 0.f, inv_n);
          // folded form for items that do not store H2 (exact, powers of two):
          // relu(v/(s_m s_n) + b2) w3 = relu(v/s_m + b2 s_n) (w3/s_n); two columns per 16-byte word
          if (OUT == 1) efg[cidx] = make_float2(net[off_b2(IN) + col] / inv_n, net[off_W3(IN) + col] * inv_n);
        }
        wm = make_float4(__ldg(&meta->wmax[0]), __ldg(&meta->wmax[1]), IN == 3 ? __ldg(&meta->wmax[2]) : 0.f, __ldg(&meta->wmax[3]));
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp));
      }
      const uint32_t acc = grp;
      const int row = ii.tile * TM + row_in_tile;
      const float4 x = row < jb.rows ? __ldg(jb.X + row) : make_float4(0.f, 0.f, 0.f, 0.f);
      float sa, inv_sa;
      pow2_scale(h1_row_bound(x, wm), sa, inv_sa);                 // the producers' scale of this row, recomputed
      mbar_wait(&tfull[acc], (tcount >> 1) & 1);
      tc_fence_after();
      const bool store_h2 = jb.h2 != nullptr;
      const int tiles64 = (jb.rows + 63) / 64;
      float* h2row = store_h2 ? jb.h2 + (((size_t)ii.net * tiles64 + (row >> 6)) * H + ii.slice * C::NS) * 64 + (row & 63)
                              : nullptr;
      float q0 = 0.f, q1 = 0.f;
      if (OUT == 1 && !store_h2) {
#pragma unroll 1
        for (int c0 = 0; c0 < C::NS; c0 += 32) {
          float v[32];
          tmem_ld32(tmem + ((uint32_t)(qw * 32) << 16) + acc * C::NS + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float4 e = reinterpret_cast<const float4*>(efg)[(c0 + i) >> 1];
            q0 = fmaf(fmaxf(fmaf(v[i], inv_sa, e.x), 0.f), e.y, q0);
            q0 = fmaf(fmaxf(fmaf(v[i + 1], inv_sa, e.z), 0.f), e.w, q0);
          }
        }
      } else
#pragma unroll 1
      for (int c0 = 0; c0 < C::NS; c0 += 32) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(qw * 32) << 16) + acc * C::NS + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float4 e = ebg[c0 + i];
          const float hv = fmaxf(fmaf(v[i] * inv_sa, e.w, e.x), 0.f);
          v[i] = hv;
          q0 = fmaf(hv, e.y, q0);
          if (OUT == 2) q1 = fmaf(hv, e.z, q1);
        }
        if (store_h2 && (row >> 6) < tiles64) {
#pragma unroll
          for (int i = 0; i < 32; ++i) h2row[(size_t)(c0 + i) * 64] = v[i];
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (row < jb.rows) {
        float* o = jb.out_part + (((size_t)ii.net * C::SLICES + ii.slice) * jb.rows + row) * OUT;
        o[0] = q0;
        if (OUT == 2) o[1] = q1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::MMA_WARP) tmem_dealloc(tmem, C::TMEM_ALLOC);
}


// ---------------------------------------------------------------------------------------------------------------
// Input gradient of the hidden layer on the same fp16 hi/lo path:  dH1 = dZ2 W2, then dZ1 = dH1 * relu'(Z1), dW1, db1
// and (optionally) dx.  Structure of tc_bwd1_ts_kernel (mlp_tc_bwd1.cuh); differences: W2^T packed as scaled fp16
// hi|lo in 128-column slices, the dZ2 row scaled by 2^e from the bound |dOut_0| max|W3_0| + |dOut_1| max|W3_1|,
// two epilogue groups (one per accumulator), accumulator unscaled by 1/(s_m s_n) before the ReLU mask.
template <int IN, int OUT, bool WGRADS, bool DX, class C = HCfg>
__global__ void __launch_bounds__(HCfg::THREADS, 1) tc_bwd1_h_kernel(const Bwd1Job jb) {
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + C::OFF_B;
  float2* w3s = reinterpret_cast<float2*>(sm + C::OFF_W1);    // [256] (W3[0][j], W3[1][j])
  float4* ebs = reinterpret_cast<float4*>(sm + C::OFF_EB);    // [2][NS]  (W1[k][0..2], b1[k]) of the slice's columns
  float* invs = reinterpret_cast<float*>(sm + C::OFF_W1 + H * 8);   // [2][NS] 1/s_n of the slice's columns (after w3s)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bload = tempty + 2;
  uint64_t* drain = bload + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles = (jb.rows + TM - 1) / TM;
  const int tiles64 = (jb.rows + 63) / 64;
  const int total = jb.n_nets * C::SLICES * tiles;
  const int item_lo = (int)((long long)total * blockIdx.x / gridDim.x);
  const int item_hi = (int)((long long)total * (blockIdx.x + 1) / gridDim.x);

  if (warp == C::MMA_WARP) {
    tmem_alloc(slot, C::TMEM_ALLOC);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], C::NPW); mbar_init(&empty[s], 1); }
      for (int q = 0; q < 2; ++q) { mbar_init(&tfull[q], 1); mbar_init(&tempty[q], 4); }
      mbar_init(bload, 1);
      mbar_init(drain, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;
  grid_dep_wait();            // everything above overlapped the predecessor's tail (programmatic dependent launch)
  if (WGRADS) zero_small1_slots<IN>(jb, 2);          // slots (CTA, epilogue group)

  if (warp == C::MMA_WARP) {
    const uint32_t idesc = instr_desc(FMT_F16, TM, C::NS);
    const uint32_t b_lbo = C::NS * 16;
    const uint32_t b_base = smem_u32(Bs);
    int cur_pair = -1;
    uint32_t it = 0, nb = 0, nd = 0, tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles;
      if (pair != cur_pair) {
        if (cur_pair >= 0) { if (elect_one()) umma_commit(drain); __syncwarp(); mbar_wait(drain, nd & 1); ++nd; }
        if (elect_one()) load_operand_slice<C>(Bs, jb.packedT + (size_t)(pair / C::SLICES) * HCfg::PACKED_NET_BYTES, pair % C::SLICES, bload);
        __syncwarp();
        mbar_wait(bload, nb & 1);
        ++nb;
        cur_pair = pair;
      }
      const uint32_t acc = tcount & 1;
      mbar_wait(&tempty[acc], ((tcount >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem + acc * C::NS;
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        const uint32_t s = it % C::STAGES;
        mbar_wait(&full[s], (it / C::STAGES) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_stage = tmem + C::A_COL0 + s * C::A_STAGE_COLS;
#pragma unroll
          for (int j = 0; j < C::KC / C::UK; ++j) {
            const uint32_t g = c * (C::KC / C::UK) + j;
            const uint64_t b_hi = smem_desc(b_base + 2 * g * b_lbo, b_lbo, 128);
            const uint64_t b_lo = smem_desc(b_base + C::B_TERM_BYTES + 2 * g * b_lbo, b_lbo, 128);
            const uint32_t a_hi = a_stage + j * 8, a_lo = a_hi + C::A_LO_COLS;
            umma_ts<false>(d_tmem, a_lo, b_hi, idesc, (c == 0 && j == 0) ? 0u : 1u);
            umma_ts<false>(d_tmem, a_hi, b_lo, idesc, 1u);
            umma_ts<false>(d_tmem, a_hi, b_hi, idesc, 1u);
          }
          umma_commit(&empty[s]);
          if (c == C::NCHUNK - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
      }
      ++tcount;
    }
  } else if (warp >= C::NEW) {
    // ---------------- producers: dZ2 row -> scaled fp16 hi|lo -> TMEM ----------------
    const int pw = warp - C::NEW, ptid = tid - C::NEW * 32;
    const int kq = pw >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + kq * (C::KPW / 2);
    int cur_net = -1;
    float w3m0 = 0.f, w3m1 = 0.f;
    uint32_t it = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles, tile = item % tiles, net_i = pair / C::SLICES;
      if (net_i != cur_net) {
        cur_net = net_i;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        for (int j = ptid; j < H; j += C::PROD_THREADS)
          w3s[j] = make_float2(net[off_W3(IN) + j], OUT == 2 ? net[off_W3(IN) + H + j] : 0.f);
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packedT + (size_t)net_i * HCfg::PACKED_NET_BYTES + HCfg::META_OFF);
        w3m0 = __ldg(&meta->wmax[4]);
        w3m1 = OUT == 2 ? __ldg(&meta->wmax[5]) : 0.f;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      }
      const int r = tile * TM + (warp & 3) * 32 + lane;
      const bool ok = r < jb.rows;
      float d0 = 0.f;
      if (OUT == 1 && DX && !WGRADS && jb.q_parts > 0) { if (ok) d0 = actor_dq_of<IN, OUT>(jb, net_i, r); }
      else if (ok) d0 = __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT);
      const float d1 = (ok && OUT == 2) ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + 1) : 0.f;
      float sa, inv_sa;
      pow2_scale(fmaf(fabsf(d0), w3m0, fabsf(d1) * w3m1), sa, inv_sa);
      const float d0s = d0 * sa, d1s = d1 * sa;                       // exact
      const int rc = ok ? r : 0;
      const float* h2r = jb.h2 + ((size_t)net_i * tiles64 + (rc >> 6)) * H * 64 + (rc & 63);
      float hn[C::KPW];                                    // next stage's H2 values, loaded one stage ahead
#pragma unroll
      for (int e = 0; e < C::KPW; ++e) hn[e] = __ldg(h2r + (size_t)(kq * C::KPW + e) * 64);
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        const uint32_t s = it % C::STAGES;
        const int j0 = c * C::KC + kq * C::KPW;
        float hv[C::KPW];
#pragma unroll
        for (int e = 0; e < C::KPW; ++e) hv[e] = hn[e];
        if (c + 1 < C::NCHUNK) {
#pragma unroll
          for (int e = 0; e < C::KPW; ++e) hn[e] = __ldg(h2r + (size_t)(j0 + C::KC + e) * 64);
        }
        uint32_t hi[C::KPW / 2], lo[C::KPW / 2];
#pragma unroll
        for (int e = 0; e < C::KPW; e += 2) {
          const float2 wa = w3s[j0 + e], wb = w3s[j0 + e + 1];
          float ga = d0s * wa.x, gb = d0s * wb.x;
          if (OUT == 2) { ga = fmaf(d1s, wa.y, ga); gb = fmaf(d1s, wb.y, gb); }
          split_h2_trunc(make_float2(hv[e] > 0.f ? ga : 0.f, hv[e + 1] > 0.f ? gb : 0.f), hi[e / 2], lo[e / 2]);
        }
        mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
        tc_fence_after();
        tmem_st8(lane_base + s * C::A_STAGE_COLS, hi);
        tmem_st8(lane_base + s * C::A_STAGE_COLS + C::A_LO_COLS, lo);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
  } else {
    // ---------------- epilogue (two groups): dZ1, dx, dW1/db1 ----------------
    constexpr int NCH = C::NS / 32;
    const int grp = warp >> 2, qw = warp & 3, gtid = tid & 127;
    float4* ebg = ebs + grp * C::NS;
    float* ivg = invs + grp * C::NS;
    float a_b[NCH], a_w0[NCH], a_w1[NCH], a_w2[NCH];      // lane l <-> column chunk*32 + l of the current slice
#pragma unroll
    for (int q = 0; q < NCH; ++q) { a_b[q] = 0.f; a_w0[q] = 0.f; a_w1[q] = 0.f; a_w2[q] = 0.f; }
    // The four warps of a group hold partial column sums over different rows: they are added through shared memory
    // (fixed warp order) and ONE slot per (CTA, group) goes to global memory -- 4x fewer partials for the reduction.
    float* flbuf = reinterpret_cast<float*>(sm + C::OFF_FLUSH) + grp * (4 * 16 * 32);
    float* red_t = reinterpret_cast<float*>(sm + C::OFF_RED + warp * C::RED_WARP_BYTES);       // [32][33]
    float4* red_x = reinterpret_cast<float4*>(red_t + 32 * 33);                                 // [32] this item's input rows
    auto flush = [&](int pair) {                    // called uniformly by the 4 warps of the group
      if (!WGRADS || pair < 0) return;
      const int net_i = pair / C::SLICES, slice = pair % C::SLICES;
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        float* f = flbuf + (qw * 16 + q * 4) * 32 + lane;
        f[0] = a_w0[q]; f[32] = a_w1[q]; f[64] = a_w2[q]; f[96] = a_b[q];
        a_b[q] = 0.f; a_w0[q] = 0.f; a_w1[q] = 0.f; a_w2[q] = 0.f;
      }
      asm volatile("bar.sync %0, 128;" ::"r"(2 + grp));
      float* o = jb.small1 + ((size_t)net_i * jb.slots + blockIdx.x * 2 + grp) * SMALL_STRIDE;
      // warp w of the group sums chunk q = w over the four warps (order 0..3) and writes that chunk's columns
      if (qw < NCH) {
        const int q = qw;
        float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float* f = flbuf + (w * 16 + q * 4) * 32 + lane;
          t0 += f[0]; t1 += f[32]; t2 += f[64]; t3 += f[96];
        }
        const int k = slice * C::NS + q * 32 + lane;
        o[k * IN + 0] = t0;
        o[k * IN + 1] = t1;
        if (IN == 3) o[k * IN + 2] = t2;
        o[H * IN + k] = t3;
      }
      asm volatile("bar.sync %0, 128;" ::"r"(2 + grp));
    };
    int cur_pair = -1;
    float w3m0 = 0.f, w3m1 = 0.f;
    for (int item = item_lo + grp; item < item_hi; item += 2) {
      const uint32_t tcount = (uint32_t)(item - item_lo);
      const int pair = item / tiles, tile = item % tiles, net_i = pair / C::SLICES, slice = pair % C::SLICES;
      if (pair != cur_pair) {
        flush(cur_pair);
        cur_pair = pair;
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp));
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packedT + (size_t)net_i * HCfg::PACKED_NET_BYTES + HCfg::META_OFF);
        for (int cidx = gtid; cidx < C::NS; cidx += 128) {
          const int k = slice * C::NS + cidx;
          ebg[cidx] = make_float4(net[off_W1(IN) + k * IN], net[off_W1(IN) + k * IN + 1],
                                  IN == 3 ? net[off_W1(IN) + k * IN + 2] : 0.f, net[off_b1(IN) + k]);
          ivg[cidx] = __ldg(&meta->inv_s[k]);
        }
        w3m0 = __ldg(&meta->wmax[4]);
        w3m1 = OUT == 2 ? __ldg(&meta->wmax[5]) : 0.f;
        asm volatile("bar.sync %0, 128;" ::"r"(2 + grp));
      }
      const uint32_t acc = grp;
      const int row = tile * TM + qw * 32 + lane;
      const bool ok = row < jb.rows;
      const float4 x = ok ? __ldg(jb.X + row) : make_float4(0.f, 0.f, 0.f, 0.f);
      float d0 = 0.f;
      if (OUT == 1 && DX && !WGRADS && jb.q_parts > 0) { if (ok) d0 = actor_dq_of<IN, OUT>(jb, net_i, row); }
      else if (ok) d0 = __ldg(jb.dOut + ((size_t)net_i * jb.rows + row) * OUT);
      const float d1 = (ok && OUT == 2) ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + row) * OUT + 1) : 0.f;
      float sa, inv_sa;
      pow2_scale(fmaf(fabsf(d0), w3m0, fabsf(d1) * w3m1), sa, inv_sa);     // the producers' scale of this row
      if (WGRADS) {
        __syncwarp();
        red_x[lane] = x;                                                      // rows beyond jb.rows are zero
      }
      mbar_wait(&tfull[acc], (tcount >> 1) & 1);
      tc_fence_after();
      float dx0 = 0.f, dx1 = 0.f, dx2 = 0.f;
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(qw * 32) << 16) + acc * C::NS + q * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float4 w = ebg[q * 32 + i];
          // layer-1 pre-activation in the FORWARD's order (chain starts from the bias): the ReLU mask agrees with
          // the forward bit for bit
          float z = fmaf(x.y, w.y, fmaf(x.x, w.x, w.w));
          if (IN == 3) z = fmaf(x.z, w.z, z);
          // without dx the column scale 1/s_n is applied once per column sum instead of once per element
          const float d = z > 0.f ? (DX ? v[i] * inv_sa * ivg[q * 32 + i] : v[i] * inv_sa) : 0.f;
          v[i] = d;
          if (DX) {
            dx0 = fmaf(d, w.x, dx0);
            dx1 = fmaf(d, w.y, dx1);
            if (IN == 3) dx2 = fmaf(d, w.z, dx2);
          }
        }
        if (WGRADS) {
          // column sums over the warp's 32 rows through a transposed shared-memory tile: thread = row writes its 32
          // values, then lane = column walks the rows (2 LDS + 4 FMA per row) -- 224 instructions per chunk instead
          // of ~590 for four 31-step shuffle butterflies; the row order is fixed, so the result is deterministic
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 32; ++i) red_t[lane * 33 + i] = v[i];
          __syncwarp();
          float s0 = 0.f, s1 = 0.f, s2 = 0.f, sb = 0.f;
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float dv = red_t[r * 33 + lane];
            const float4 xr = red_x[r];
            s0 = fmaf(dv, xr.x, s0);
            s1 = fmaf(dv, xr.y, s1);
            if (IN == 3) s2 = fmaf(dv, xr.z, s2);
            sb += dv;
          }
          const float cs = DX ? 1.f : ivg[q * 32 + lane];
          a_w0[q] = fmaf(s0, cs, a_w0[q]); a_w1[q] = fmaf(s1, cs, a_w1[q]); a_w2[q] = fmaf(s2, cs, a_w2[q]);
          a_b[q] = fmaf(sb, cs, a_b[q]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (DX && ok)
        jb.dX_part[((size_t)net_i * C::SLICES + slice) * jb.rows + row] = make_float4(dx0, dx1, dx2, 0.f);
    }
    flush(cur_pair);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::MMA_WARP) tmem_dealloc(tmem, C::TMEM_ALLOC);
}


// ---------------------------------------------------------------------------------------------------------------
// Weight gradient of the hidden layer, dW2 = dZ2^T H1, on the fp16 hi/lo path.  Structure of tc_bwd2_kernel
// (mlp_tc_bwd2.cuh): thread t owns hidden unit t and generates row t of BOTH operands on chip; the 256x256 FP32
// accumulator fills the tensor memory.  The contraction runs over batch rows, so the scales are per operand ROW
// (= per hidden unit = per thread), constant over the CTA's whole row range:
//   s_A[t] from |W3[:,t]| . max_r |dOut[r,:]|,   s_B[t] from |W1[t,:]| . max_r |x[r,:]| + |b1[t]|
// with the maxima taken in a pre-pass over the CTA's rows; the partial is unscaled by 1/(s_A[j] s_B[k]) on the way out.
// A stage holds 32 rows (K = 32 = two MMAs), the same operand bytes as the tf32 kernel's 16 rows.
struct B2HCfg {
  static constexpr int ES = 2, EPC = 8, UK = 16;
  static constexpr int RS = 32;                             // rows (K extent) per stage
  static constexpr int STAGES = 3;
  static constexpr int PROD_WARPS = 16;                     // two threads per hidden unit, 16 rows of a stage each
  static constexpr int PROD_THREADS = PROD_WARPS * 32;
  static constexpr int THREADS = PROD_THREADS + 32;         // + MMA warp
  static constexpr int RPT = RS / 2;                        // rows per thread per stage
  static constexpr uint32_t OP_TERM_BYTES = H * RS * ES;    // 16 KB
  static constexpr uint32_t OP_BYTES = 2 * OP_TERM_BYTES;   // 32 KB (hi | lo)
  static constexpr uint32_t STAGE_BYTES = 2 * OP_BYTES;     // A then B: 64 KB
  static constexpr uint32_t OFF_X = STAGES * STAGE_BYTES;       // float4[STAGES][RS]
  static constexpr uint32_t OFF_DO = OFF_X + STAGES * RS * 16;  // float[STAGES][RS][2]
  static constexpr uint32_t OFF_INV = OFF_DO + STAGES * RS * 8; // float invA[256] | invB[256]
  static constexpr uint32_t OFF_SMALL = OFF_INV + 2 * H * 4;    // float[256][4]: second half's db2 | dW3[0..1] | -
  static constexpr uint32_t OFF_MAX = OFF_SMALL + H * 16;       // int[8] row maxima (float bits)
  static constexpr uint32_t OFF_BAR = OFF_MAX + 32;
  static constexpr uint32_t OFF_SLOT = OFF_BAR + (2 * STAGES + 1) * 8;
  static constexpr uint32_t BYTES = OFF_SLOT + 16;
};

template <int IN, int OUT>
__global__ void __launch_bounds__(B2HCfg::THREADS, 1) tc_bwd2_h_kernel(const Bwd2Job jb) {
  using C = B2HCfg;
  extern __shared__ __align__(1024) uint8_t sm[];
  float4* xs = reinterpret_cast<float4*>(sm + C::OFF_X);
  float* dos = reinterpret_cast<float*>(sm + C::OFF_DO);
  float* invA = reinterpret_cast<float*>(sm + C::OFF_INV);
  float* invB = invA + H;
  float4* small_h1 = reinterpret_cast<float4*>(sm + C::OFF_SMALL);
  int* rmax = reinterpret_cast<int*>(sm + C::OFF_MAX);
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* empty = full + C::STAGES;
  uint64_t* done = empty + C::STAGES;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = blockIdx.x, net_i = blockIdx.y;
  const float* net = jb.params + (size_t)net_i * NET_STRIDE;
  const int tiles64 = (jb.rows + 63) / 64;
  const int n_stage_total = (jb.rows + C::RS - 1) / C::RS;
  const int st_lo = (int)((long long)n_stage_total * split / jb.splits);
  const int st_hi = (int)((long long)n_stage_total * (split + 1) / jb.splits);

  if (warp == C::PROD_WARPS) {
    tmem_alloc(slot, 512);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], C::PROD_WARPS); mbar_init(&empty[s], 1); }
      mbar_init(done, 1);
      fence_mbar_init();
    }
  }
  if (tid < 8) rmax[tid] = 0;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;
  grid_dep_wait();            // everything above overlapped the predecessor's tail (programmatic dependent launch)

  if (warp == C::PROD_WARPS) {
    const uint32_t idesc = instr_desc(FMT_F16, 128, 256);
    const uint32_t lbo = H * 16;
    uint32_t it = 0;
    for (int sg = st_lo; sg < st_hi; ++sg, ++it) {
      const uint32_t s = it % C::STAGES;
      mbar_wait(&full[s], (it / C::STAGES) & 1);
      tc_fence_after();
      const uint32_t a_base = smem_u32(sm + s * C::STAGE_BYTES);
      const uint32_t b_base = a_base + C::OP_BYTES;
      if (elect_one()) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
          for (int j = 0; j < C::RS / C::UK; ++j) {
            const uint32_t acc = (it == 0 && j == 0) ? 0u : 1u;
            const uint64_t a_hi = smem_desc(a_base + half * 2048 + 2 * j * lbo, lbo, 128);
            const uint64_t b_hi = smem_desc(b_base + 2 * j * lbo, lbo, 128);
            const uint64_t a_lo = smem_desc(a_base + C::OP_TERM_BYTES + half * 2048 + 2 * j * lbo, lbo, 128);
            const uint64_t b_lo = smem_desc(b_base + C::OP_TERM_BYTES + 2 * j * lbo, lbo, 128);
            const uint32_t d = tmem + half * 256;
            umma<false>(d, a_lo, b_hi, idesc, acc);
            umma<false>(d, a_hi, b_lo, idesc, 1u);
            umma<false>(d, a_hi, b_hi, idesc, 1u);
          }
        }
        umma_commit(&empty[s]);
        if (sg == st_hi - 1) umma_commit(done);
      }
      __syncwarp();
    }
  } else {
    // ---------------- producers: thread (t, rh): hidden unit t (A row j = t, B row k = t), rows rh*16 .. +16 of a stage
    const int t = tid & (H - 1), rh = tid >> 8;
    float w3[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) w3[o] = net[off_W3(IN) + o * H + t];
    const float w1x = net[off_W1(IN) + t * IN], w1y = net[off_W1(IN) + t * IN + 1];
    const float w1z = IN == 3 ? net[off_W1(IN) + t * IN + 2] : 0.f;
    const float b1v = net[off_b1(IN) + t];
    // pre-pass: maxima of |x| components and |dOut| components over this CTA's rows -> per-unit scales
    {
      float mx0 = 0.f, mx1 = 0.f, mx2 = 0.f, md0 = 0.f, md1 = 0.f;
      const int r_lo = st_lo * C::RS, r_hi = min(jb.rows, st_hi * C::RS);
      for (int r = r_lo + tid; r < r_hi; r += C::PROD_THREADS) {
        const float4 x = __ldg(jb.X + r);
        mx0 = fmaxf(mx0, fabsf(x.x)); mx1 = fmaxf(mx1, fabsf(x.y)); mx2 = fmaxf(mx2, fabsf(x.z));
        md0 = fmaxf(md0, fabsf(__ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT)));
        if (OUT == 2) md1 = fmaxf(md1, fabsf(__ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + 1)));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, o)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, o));
        mx2 = fmaxf(mx2, __shfl_xor_sync(0xffffffffu, mx2, o)); md0 = fmaxf(md0, __shfl_xor_sync(0xffffffffu, md0, o));
        md1 = fmaxf(md1, __shfl_xor_sync(0xffffffffu, md1, o));
      }
      if (lane == 0) {
        atomicMax(&rmax[0], __float_as_int(mx0)); atomicMax(&rmax[1], __float_as_int(mx1)); atomicMax(&rmax[2], __float_as_int(mx2));
        atomicMax(&rmax[3], __float_as_int(md0)); atomicMax(&rmax[4], __float_as_int(md1));
      }
      asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
    }
    float sA, sB;
    {
      float ia, ib;
      float bA = fabsf(w3[0]) * __int_as_float(rmax[3]);
      if (OUT == 2) bA = fmaf(fabsf(w3[OUT - 1]), __int_as_float(rmax[4]), bA);
      pow2_scale(bA, sA, ia);
      const float bB = fmaf(fabsf(w1x), __int_as_float(rmax[0]), fmaf(fabsf(w1y), __int_as_float(rmax[1]),
                       fmaf(fabsf(w1z), __int_as_float(rmax[2]), fabsf(b1v))));
      pow2_scale(bB, sB, ib);
      if (rh == 0) { invA[t] = ia; invB[t] = ib; }
    }
    float s_db2 = 0.f, s_dw3[OUT], s_db3[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) { s_dw3[o] = 0.f; s_db3[o] = 0.f; }
    uint32_t it = 0;
    auto h2_ptr = [&](int sg) {
      const int row0 = sg * C::RS + rh * C::RPT;
      return jb.h2 + (((size_t)net_i * tiles64 + (row0 >> 6)) * H + t) * 64 + (row0 & 63);
    };
    // software pipeline: the next stage's H2 values (all threads) and x / dOut rows (threads < RS) are loaded into
    // registers while the current stage is computed -- a stage's global-load latency is off the critical path
    float4 hq[C::RPT / 4], hn[C::RPT / 4];
    float4 xn = make_float4(0.f, 0.f, 0.f, 0.f);
    float dn[OUT];
    auto prefetch = [&](int sg) {
      const float* h2p = h2_ptr(sg);
#pragma unroll
      for (int q = 0; q < C::RPT / 4; ++q) hn[q] = __ldg(reinterpret_cast<const float4*>(h2p) + q);
      if (tid < C::RS) {
        const int r = sg * C::RS + tid;
        xn = r < jb.rows ? __ldg(jb.X + r) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int o = 0; o < OUT; ++o) dn[o] = r < jb.rows ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + o) : 0.f;
      }
    };
    if (st_lo < st_hi) prefetch(st_lo);
    for (int sg = st_lo; sg < st_hi; ++sg, ++it) {
      const uint32_t s = it % C::STAGES;
#pragma unroll
      for (int q = 0; q < C::RPT / 4; ++q) hq[q] = hn[q];
      const float4 xc = xn;
      float dc[OUT];
#pragma unroll
      for (int o = 0; o < OUT; ++o) dc[o] = dn[o];
      if (sg + 1 < st_hi) prefetch(sg + 1);
      mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
      float4* xst = xs + s * C::RS;
      float* dost = dos + s * C::RS * 2;
      if (tid < C::RS) {
        xst[tid] = xc;
#pragma unroll
        for (int o = 0; o < OUT; ++o) dost[tid * 2 + o] = dc[o];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      uint8_t* Ast = sm + s * C::STAGE_BYTES;
      uint8_t* Bst = Ast + C::OP_BYTES;
#pragma unroll
      for (int kk = 0; kk < C::RPT / C::EPC; ++kk) {
        const int kc = rh * (C::RPT / C::EPC) + kk;        // 16-byte K chunk (8 rows) of the stage
        float hv[8], dz[8], h1[8];
        hv[0] = hq[2 * kk].x; hv[1] = hq[2 * kk].y; hv[2] = hq[2 * kk].z; hv[3] = hq[2 * kk].w;
        hv[4] = hq[2 * kk + 1].x; hv[5] = hq[2 * kk + 1].y; hv[6] = hq[2 * kk + 1].z; hv[7] = hq[2 * kk + 1].w;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int rl = kc * 8 + e;
          float g = 0.f;
#pragma unroll
          for (int o = 0; o < OUT; ++o) {
            const float d = dost[rl * 2 + o];
            g = fmaf(d, w3[o], g);
            s_dw3[o] = fmaf(d, hv[e], s_dw3[o]);
            if (t == 0) s_db3[o] += d;
          }
          dz[e] = hv[e] > 0.f ? g : 0.f;
          s_db2 += dz[e];
          const float4 x = xst[rl];
          float z = fmaf(x.y, w1y, fmaf(x.x, w1x, b1v));        // the forward's order: chain starts from the bias
          if (IN == 3) z = fmaf(x.z, w1z, z);
          h1[e] = fmaxf(z, 0.f);
        }
        const uint32_t off = chunk_off(H, t, kc);
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) split_h2_trunc(make_float2(dz[2 * e] * sA, dz[2 * e + 1] * sA), hi[e], lo[e]);
        *reinterpret_cast<uint4*>(Ast + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(Ast + C::OP_TERM_BYTES + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
#pragma unroll
        for (int e = 0; e < 4; ++e) split_h2_trunc(make_float2(h1[2 * e] * sB, h1[2 * e + 1] * sB), hi[e], lo[e]);
        *reinterpret_cast<uint4*>(Bst + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(Bst + C::OP_TERM_BYTES + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
    }
    // small gradients of unit t: the two row-halves are added in a fixed order (first half + second half)
    if (rh == 1) small_h1[t] = make_float4(s_db2, s_dw3[0], OUT == 2 ? s_dw3[OUT - 1] : 0.f, t == 0 ? s_db3[0] : 0.f);
    float db3_1 = 0.f;
    if (OUT == 2 && t == 0 && rh == 1) rmax[6] = __float_as_int(s_db3[OUT - 1]);   // (plain bit copy; slot unused otherwise)
    asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
    if (rh == 0) {
      const float4 o2 = small_h1[t];
      if (OUT == 2 && t == 0) db3_1 = __int_as_float(rmax[6]);
      float* sm2 = jb.small2 + ((size_t)net_i * jb.splits + split) * SMALL_STRIDE;
      sm2[H * IN + H + t] = s_db2 + o2.x;
      sm2[H * IN + 2 * H + t] = s_dw3[0] + o2.y;
      if (OUT == 2) sm2[H * IN + 2 * H + H + t] = s_dw3[OUT - 1] + o2.z;
      if (t == 0) {
        sm2[H * IN + 2 * H + OUT * H] = s_db3[0] + o2.w;
        if (OUT == 2) sm2[H * IN + 2 * H + OUT * H + 1] = s_db3[OUT - 1] + db3_1;
      }
    }
  }
  // ---------------- epilogue: unscale and dump the 256x256 accumulator as this split's partial ----------------
  // all 16 producer warps take part: warp w reads TMEM lane quarter w % 4 and every fourth 32-column chunk
  float* out = jb.pw2 + ((size_t)net_i * jb.splits + split) * H * H;
  if (warp < C::PROD_WARPS) {
    const int qw = warp & 3, part = warp >> 2;
    if (st_hi > st_lo) {
      mbar_wait(done, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const int j = half * 128 + qw * 32 + lane;
      const float ia = invA[j];
      float* orow = out + (size_t)j * H;
#pragma unroll 1
      for (int c0 = part * 32; c0 < H; c0 += 32 * (C::PROD_WARPS / 4)) {
        float v[32];
        if (st_hi > st_lo) {
          tmem_ld32(tmem + ((uint32_t)(qw * 32) << 16) + half * 256 + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = v[i] * ia * invB[c0 + i];
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          *reinterpret_cast<float4*>(orow + c0 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::PROD_WARPS) tmem_dealloc(tmem, 512);
}

}  // namespace tc
}  // namespace cql
