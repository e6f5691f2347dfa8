// score_tc.cuh -- K5 on tensor cores: FP32-grade user x item scoring with the seen filter and top-k fused in, never
// materialising a score.  One kernel, two numeric formats (the Split traits below):
//   * SplitTf32 -- tf32 3-term split (mlp_tc_ts.cuh), 64-column W2 slices: 4 passes per network (tf32x3, bf16);
//   * SplitF16  -- fp16 hi/lo 3-term split (mlp_tc_h.cuh), twice the tensor rate and 128-column W2 slices: 2 passes
//     per network (f16x3).  Rows carry the exact power-of-two scales described in mlp_tc_h.cuh.
//
// A CTA owns BLOCKS of up to CH row tiles (128 items each) of ONE user and runs the networks over a block
// pass by pass -- pass = (network, W2 slice): actor slices, then critic_0 slices, ... --
// reloading the 128 KB resident W2 slice once per pass (amortised over CH tiles) and keeping the per-row
// state (mu partial sums -> greedy action a = tanh(mu), Q partial sums) in shared memory.  After the last
// pass the epilogue warps fold the block's scores into the user's running top-k (lazy seen filter: only
// candidates that beat the current k-th score are looked up in the user's sorted seen list).
// The per-item pipeline (producers -> TMEM -> tcgen05.mma TS -> epilogue) is the one of mlp_tc_ts.cuh / mlp_tc_h.cuh.
#pragma once
#include "mlp_tc_ts.cuh"
#include "mlp_tc_h.cuh"
#include "score.cuh"

namespace cql {
namespace tc {

constexpr int SC_CH = 16;                       // tiles per block (2048 rows of per-row state)

struct ScoreTcArgs {
  const float* params;        // flat fp32 state
  const uint8_t* packed;      // W2 of slots 0..C (actor, critics) in the split's operand layout, forward orientation
  const int32_t* users;       // [U]
  const int32_t* items;       // [I]
  const int64_t* seen_indptr; // CSR over user id or nullptr
  const int32_t* seen_items;
  int64_t n_users, n_items;
  int C, k, mode, chunks;     // chunks = blocks per user
  float* part_s;              // [U][chunks][k]
  int* part_i;
  const float* item_x;        // [I] scaled item coordinates (obs scaler on), or nullptr: (float)item
  Prep prep;                  // user coordinate (once per block) and the policy score's reverse action transform
};
// observation coordinates of a scored pair; the producers and the f16x3 epilogue's row-scale recomputation both come here
__device__ __forceinline__ float score_user(const ScoreTcArgs& a, int64_t urow) {
  return prep_fwd(a.prep.obs[0], (float)a.users[urow]);
}
__device__ __forceinline__ float score_item(const ScoreTcArgs& a, int64_t idx) {
  return idx < a.n_items ? (a.item_x ? __ldg(a.item_x + idx) : (float)__ldg(a.items + idx)) : 0.f;
}

// The numeric format of a scorer: how the MMA reads the A operand from TMEM, how a producer turns a row's layer-1
// pre-activations into hi | lo operand words (Prod), and how the epilogue turns accumulator columns into Q (Epi).
//   Prod: b1 = w1p's bias entry of a hidden unit; net / row = state taken per (block, network) / per row;
//         pair = the hi | lo words of hidden pair pp.  w1p holds {wx_k, wx_k1, wy_k, wy_k1}, {wz_k, wz_k1, b1_k, b1_k1}.
//   Epi:  block / row = state taken per block / per row; slice = a pass's layer-2/3 constants into ebs;
//         dot32 = q0 + sum over 32 accumulator columns of relu(layer 2) * w3.

// tf32 3-term split: one fp32 word per element
struct SplitTf32 {
  using Cfg = TsCfg;
  static constexpr uint32_t FMT = FMT_TF32;
  static constexpr bool TF32 = true;                  // umma_ts kind
  static constexpr uint32_t A_STEP = Cfg::UK;         // A columns per MMA
  static constexpr uint32_t A_LO = Cfg::KC;           // lo term's column offset within an A stage
  static constexpr int A_WORDS = Cfg::KPW;            // columns per term a producer warp writes per stage

  struct Prod {
    __device__ __forceinline__ static float b1(float, float, float b) { return b; }
    __device__ __forceinline__ void net(const ScoreTcArgs&, int) {}
    __device__ __forceinline__ void row(float, float, float) {}
    __device__ __forceinline__ void pair(int pp, const float4& wA, const float4& wB, float2 xx, float2 xy, float2 xz,
                                         int, uint32_t (&hi)[A_WORDS], uint32_t (&lo)[A_WORDS]) const {
      float2 v = ffma2(xx, make_float2(wA.x, wA.y), make_float2(wB.z, wB.w));
      v = ffma2(xy, make_float2(wA.z, wA.w), v);
      v = ffma2(xz, make_float2(wB.x, wB.y), v);      // actor: wz = 0
      float h0, l0, h1, l1;
      split_tf32_fast(fmaxf(v.x, 0.f), h0, l0);
      split_tf32_fast(fmaxf(v.y, 0.f), h1, l1);
      hi[2 * pp] = __float_as_uint(h0); lo[2 * pp] = __float_as_uint(l0);
      hi[2 * pp + 1] = __float_as_uint(h1); lo[2 * pp + 1] = __float_as_uint(l1);
    }
  };

  struct Epi {
    __device__ __forceinline__ void block(const ScoreTcArgs&, int64_t, int) {}
    __device__ __forceinline__ void slice(const ScoreTcArgs& a, float4* ebs, int net_i, int slice, int tid) {
      const float* net = a.params + (size_t)net_i * NET_STRIDE;
      const int IN = net_i == 0 ? 2 : 3;
      if (tid < Cfg::NS) {
        const int col = slice * Cfg::NS + tid;
        ebs[tid] = make_float4(net[off_b2(IN) + col], net[off_W3(IN) + col], 0.f, 0.f);   // actor: W3 row 0 = mu
      }
    }
    __device__ __forceinline__ void row(const ScoreTcArgs&, const float*, int, int) {}
    __device__ __forceinline__ float dot32(const float (&v)[32], const float4* ebs, int c0, float q0) const {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float4 e = ebs[c0 + i];
        q0 = fmaf(fmaxf(v[i] + e.x, 0.f), e.y, q0);
      }
      return q0;
    }
  };
};

// fp16 hi/lo 3-term split: two fp16 per word, every row scaled by an exact power of two
struct SplitF16 {
  using Cfg = HCfg4;
  static constexpr uint32_t FMT = FMT_F16;
  static constexpr bool TF32 = false;
  static constexpr uint32_t A_STEP = 8;               // 8 columns = 16 fp16 per MMA
  static constexpr uint32_t A_LO = Cfg::A_LO_COLS;
  static constexpr int A_WORDS = Cfg::KPW / 2;

  // the packed network's scales: operand row n's 1 / s_n, the maxima of |W1| columns and |b1| (the rows' bounds)
  __device__ __forceinline__ static const HMeta* meta(const ScoreTcArgs& a, int net_i) {
    return reinterpret_cast<const HMeta*>(a.packed + (size_t)net_i * Cfg::PACKED_NET_BYTES + Cfg::META_OFF);
  }
  __device__ __forceinline__ static float4 wmax(const HMeta* m) {
    return make_float4(__ldg(&m->wmax[0]), __ldg(&m->wmax[1]), __ldg(&m->wmax[2]), __ldg(&m->wmax[3]));
  }

  struct Prod {
    float2 ss;                                        // the row's scale
    float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);      // the network's wmax
    // the whole block belongs to one user: the first link of the layer-1 chain, b + u * w_user, is taken here once
    // per (block, network) instead of once per pair (same operation, so bit-identical)
    __device__ __forceinline__ static float b1(float uf, float w_user, float b) { return fmaf(uf, w_user, b); }
    __device__ __forceinline__ void net(const ScoreTcArgs& a, int net_i) { wm = wmax(meta(a, net_i)); }
    __device__ __forceinline__ void row(float uf, float itf, float av) {
      float sa, inv_sa;
      pow2_scale(h1_row_bound(make_float4(uf, itf, av, 0.f), wm), sa, inv_sa);
      ss = make_float2(sa, sa);
    }
    __device__ __forceinline__ void pair(int pp, const float4& wA, const float4& wB, float2, float2 xy, float2 xz,
                                         int net_i, uint32_t (&hi)[A_WORDS], uint32_t (&lo)[A_WORDS]) const {
      float2 v = ffma2(xy, make_float2(wA.z, wA.w), make_float2(wB.z, wB.w));   // chain starts from b + u * w_user
      if (net_i != 0) v = ffma2(xz, make_float2(wB.x, wB.y), v);                // the actor has no action input
      v = fmul2(make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f)), ss);
      split_h2_trunc(v, hi[pp], lo[pp]);
    }
  };

  struct Epi {
    float uf;                                         // the block's user coordinate
    int64_t i0;                                       // the block's first item
    float4 wm;                                        // the network's wmax
    float inv_sa;                                     // the row's inverse scale
    __device__ __forceinline__ void block(const ScoreTcArgs& a, int64_t urow, int chunk) {
      uf = score_user(a, urow);
      i0 = (int64_t)chunk * SC_CH * TM;
      wm = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __device__ __forceinline__ void slice(const ScoreTcArgs& a, float4* ebs, int net_i, int slice, int tid) {
      const float* net = a.params + (size_t)net_i * NET_STRIDE;
      const int IN = net_i == 0 ? 2 : 3;
      const HMeta* m = meta(a, net_i);
      if (tid < Cfg::NS) {
        const int col = slice * Cfg::NS + tid;
        // column scale folded into the constants (exact: powers of two): relu(v/(s_m s_n) + b2) w3 =
        // relu(v/s_m + b2 s_n) (w3/s_n); two columns per 16-byte word.  actor: W3 row 0 = mu
        const float inv_n = __ldg(&m->inv_s[col]);
        reinterpret_cast<float2*>(ebs)[tid] = make_float2(net[off_b2(IN) + col] / inv_n, net[off_W3(IN) + col] * inv_n);
      }
      wm = wmax(m);
    }
    // the producers' scale of this row, recomputed from the same inputs (greedy action for the critics)
    __device__ __forceinline__ void row(const ScoreTcArgs& a, const float* st_a, int net_i, int ridx) {
      const float itf = score_item(a, i0 + ridx);
      float sa;
      pow2_scale(h1_row_bound(make_float4(uf, itf, net_i == 0 ? 0.f : st_a[ridx], 0.f), wm), sa, inv_sa);
    }
    __device__ __forceinline__ float dot32(const float (&v)[32], const float4* ebs, int c0, float q0) const {
#pragma unroll
      for (int i = 0; i < 32; i += 2) {
        const float4 e = ebs[(c0 + i) >> 1];           // (b2 s_n, w3 / s_n) of columns c0+i, c0+i+1
        q0 = fmaf(fmaxf(fmaf(v[i], inv_sa, e.x), 0.f), e.y, q0);
        q0 = fmaf(fmaxf(fmaf(v[i + 1], inv_sa, e.z), 0.f), e.w, q0);
      }
      return q0;
    }
  };
};

template <class Cfg>
struct ScoreSmem : Cfg {
  static constexpr uint32_t OFF_STA = Cfg::OFF_SLOT + 16;                  // float[CH*128] greedy action
  static constexpr uint32_t OFF_STQ = OFF_STA + SC_CH * TM * 4;            // float[CH*128] running sum
  static constexpr uint32_t OFF_SCORE = OFF_STQ + SC_CH * TM * 4;          // float[CH*128] final score
  static constexpr uint32_t OFF_AREADY = OFF_SCORE + SC_CH * TM * 4;       // mbarrier
  static constexpr uint32_t OFF_SEEN = OFF_AREADY + 16;                    // int[SEEN_CACHE] current user's seen list
  static constexpr uint32_t OFF_TOP = OFF_SEEN + SEEN_CACHE * 4;           // float[k] | int[k]
  __host__ __device__ static inline uint32_t off_fold(int k) { return OFF_TOP + (uint32_t)k * 8; }     // fold_block_select scratch
  static inline uint32_t bytes(int k) { return off_fold(k) + FB_SCRATCH_WORDS * 4; }
};

template <class S>
__global__ void __launch_bounds__(S::Cfg::THREADS, 1) tc_score_kernel(const ScoreTcArgs a) {
  using C = ScoreSmem<typename S::Cfg>;
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + C::OFF_B;
  float4* w1p = reinterpret_cast<float4*>(sm + C::OFF_W1);
  float4* ebs = reinterpret_cast<float4*>(sm + C::OFF_EB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bload = tempty + 2;
  uint64_t* drain = bload + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);
  float* st_a = reinterpret_cast<float*>(sm + C::OFF_STA);
  float* st_q = reinterpret_cast<float*>(sm + C::OFF_STQ);
  float* score = reinterpret_cast<float*>(sm + C::OFF_SCORE);
  uint64_t* a_ready = reinterpret_cast<uint64_t*>(sm + C::OFF_AREADY);
  int32_t* seen_cache = reinterpret_cast<int32_t*>(sm + C::OFF_SEEN);
  float* topS = reinterpret_cast<float*>(sm + C::OFF_TOP);
  int* topI = reinterpret_cast<int*>(topS + a.k);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t tiles_total = (a.n_items + TM - 1) / TM;
  const int64_t n_blocks = a.n_users * a.chunks;
  const int64_t blk_lo = n_blocks * blockIdx.x / gridDim.x, blk_hi = n_blocks * (blockIdx.x + 1) / gridDim.x;
  const int n_nets = a.mode == CQL_SCORE_POLICY ? 1 : 1 + a.C;
  const int n_pass = n_nets * C::SLICES;
  auto tiles_of_block = [&](int64_t blk) {
    const int64_t chunk = blk % a.chunks;
    const int64_t t0 = chunk * SC_CH;
    return (int)max((int64_t)0, min((int64_t)SC_CH, tiles_total - t0));
  };

  if (warp == C::MMA_WARP) {
    tmem_alloc(slot, C::TMEM_ALLOC);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], C::NPW); mbar_init(&empty[s], 1); }
      for (int q = 0; q < 2; ++q) { mbar_init(&tfull[q], 1); mbar_init(&tempty[q], 4); }
      mbar_init(bload, 1);
      mbar_init(drain, 1);
      mbar_init(a_ready, 4);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;

  if (warp == C::MMA_WARP) {
    // =============================== MMA issuer ===============================
    const uint32_t idesc = instr_desc(S::FMT, TM, C::NS);
    const uint32_t b_lbo = C::NS * 16;
    const uint32_t b_base = smem_u32(Bs);
    uint32_t it = 0, nb = 0, nd = 0, tcount = 0;
    bool first = true;
    for (int64_t blk = blk_lo; blk < blk_hi; ++blk) {
      const int tb = tiles_of_block(blk);
      if (tb == 0) continue;
      for (int p = 0; p < n_pass; ++p) {
        if (!first) {
          if (elect_one()) umma_commit(drain);
          __syncwarp();
          mbar_wait(drain, nd & 1);
          ++nd;
        }
        first = false;
        const uint8_t* src = a.packed + (size_t)(p / C::SLICES) * C::PACKED_NET_BYTES + (size_t)(p % C::SLICES) * C::B_BYTES;
        if (elect_one()) {
          mbar_arrive_expect_tx(bload, C::B_BYTES);
          for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bload);
        }
        __syncwarp();
        mbar_wait(bload, nb & 1);
        ++nb;
        for (int t = 0; t < tb; ++t) {
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
                const uint32_t a_hi = a_stage + j * S::A_STEP, a_lo = a_hi + S::A_LO;
                umma_ts<S::TF32>(d_tmem, a_lo, b_hi, idesc, (c == 0 && j == 0) ? 0u : 1u);
                umma_ts<S::TF32>(d_tmem, a_hi, b_lo, idesc, 1u);
                umma_ts<S::TF32>(d_tmem, a_hi, b_hi, idesc, 1u);
              }
              umma_commit(&empty[s]);
              if (c == C::NCHUNK - 1) umma_commit(&tfull[acc]);
            }
            __syncwarp();
          }
          ++tcount;
        }
      }
    }
  } else if (warp >= 4) {
    // =============================== producers ===============================
    const int pw = warp - 4, ptid = tid - 128;
    const int kq = pw >> 2;
    const int row_in_tile = (warp & 3) * 32 + lane;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + kq * S::A_WORDS;
    uint32_t it = 0, nblk = 0;
    typename S::Prod prod;
    for (int64_t blk = blk_lo; blk < blk_hi; ++blk) {
      const int tb = tiles_of_block(blk);
      if (tb == 0) continue;
      const float uf = score_user(a, blk / a.chunks);
      const int64_t i0 = (blk % a.chunks) * SC_CH * TM;
      for (int p = 0; p < n_pass; ++p) {
        const int net_i = p / C::SLICES;
        if (p % C::SLICES == 0) {                 // new network: W1|b1 (actor in_dim 2, critics in_dim 3)
          asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
          const float* net = a.params + (size_t)net_i * NET_STRIDE;
          const int IN = net_i == 0 ? 2 : 3;
          for (int pr = ptid; pr < H / 2; pr += C::PROD_THREADS) {
            const int k = 2 * pr;
            const float* wa = net + off_W1(IN) + k * IN;
            const float* wb = wa + IN;
            w1p[2 * pr] = make_float4(wa[0], wb[0], wa[1], wb[1]);
            w1p[2 * pr + 1] = make_float4(IN == 3 ? wa[2] : 0.f, IN == 3 ? wb[2] : 0.f, S::Prod::b1(uf, wa[0], net[off_b1(IN) + k]),
                                          S::Prod::b1(uf, wb[0], net[off_b1(IN) + k + 1]));
          }
          prod.net(a, net_i);
          asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
          if (net_i == 1) mbar_wait(a_ready, nblk & 1);   // greedy actions of this block are in st_a
        }
        for (int t = 0; t < tb; ++t) {
          const int64_t idx = i0 + (int64_t)t * TM + row_in_tile;
          const float itf = score_item(a, idx);
          const float av = net_i == 0 ? 0.f : st_a[t * TM + row_in_tile];
          const float2 xx = make_float2(uf, uf), xy = make_float2(itf, itf), xz = make_float2(av, av);
          prod.row(uf, itf, av);
          for (int c = 0; c < C::NCHUNK; ++c, ++it) {
            const uint32_t s = it % C::STAGES;
            uint32_t hi[S::A_WORDS], lo[S::A_WORDS];
#pragma unroll
            for (int pp = 0; pp < C::KPW / 2; ++pp) {
              const int pr = (c * C::KC + kq * C::KPW) / 2 + pp;
              const float4 wA = w1p[2 * pr], wB = w1p[2 * pr + 1];
              prod.pair(pp, wA, wB, xx, xy, xz, net_i, hi, lo);
            }
            mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
            tc_fence_after();
#pragma unroll
            for (int q = 0; q < S::A_WORDS; q += 8) {
              tmem_st8(lane_base + s * C::A_STAGE_COLS + q, *reinterpret_cast<const uint32_t(*)[8]>(&hi[q]));
              tmem_st8(lane_base + s * C::A_STAGE_COLS + S::A_LO + q, *reinterpret_cast<const uint32_t(*)[8]>(&lo[q]));
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
          }
        }
      }
      ++nblk;
    }
  } else {
    // =============================== epilogue + top-k ===============================
    const int row_in_tile = warp * 32 + lane;
    uint32_t tcount = 0;
    int64_t cur_user_row = -1;
    SeenView sv{a.seen_items, nullptr, 0, 0};
    for (int64_t blk = blk_lo; blk < blk_hi; ++blk) {
      const int tb = tiles_of_block(blk);
      const int64_t urow = blk / a.chunks;
      const int chunk = (int)(blk % a.chunks);
      // top-k list is per (user, chunk): reset
      asm volatile("bar.sync 2, 128;");
      for (int e = tid; e < a.k; e += 128) { topS[e] = -INFINITY; topI[e] = -1; }
      if (urow != cur_user_row) {
        cur_user_row = urow;
        sv = stage_seen(a.seen_indptr, a.seen_items, a.users[urow], seen_cache, tid, 128);
      }
      asm volatile("bar.sync 2, 128;");
      typename S::Epi epi;
      epi.block(a, urow, chunk);
      if (tb > 0) {
        float b3sum = 0.f;
        for (int c = 0; c < a.C; ++c) b3sum += a.params[(size_t)slot_critic(c) * NET_STRIDE + off_b3(3, 1)];
        const float b3mu = a.params[(size_t)slot_actor() * NET_STRIDE + off_b3(2, 2)];
        for (int p = 0; p < n_pass; ++p) {
          const int net_i = p / C::SLICES, slice = p % C::SLICES;
          asm volatile("bar.sync 2, 128;");
          epi.slice(a, ebs, net_i, slice, tid);
          asm volatile("bar.sync 2, 128;");
          for (int t = 0; t < tb; ++t) {
            const uint32_t acc = tcount & 1;
            const int ridx = t * TM + row_in_tile;
            epi.row(a, st_a, net_i, ridx);
            mbar_wait(&tfull[acc], (tcount >> 1) & 1);
            tc_fence_after();
            float q0 = 0.f;
#pragma unroll 1
            for (int c0 = 0; c0 < C::NS; c0 += 32) {
              float v[32];
              tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + acc * C::NS + c0, v);
              tmem_ld_wait();
              q0 = epi.dot32(v, ebs, c0, q0);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            const bool first_slice = slice == 0 && (net_i <= 1);      // actor slice 0 / first critic slice 0: reset
            const float sum = first_slice ? q0 : st_q[ridx] + q0;
            st_q[ridx] = sum;
            if (net_i == 0 && slice == C::SLICES - 1) {
              const float act = tanhf(sum + b3mu);
              st_a[ridx] = act;
              if (a.mode == CQL_SCORE_POLICY) score[ridx] = act_rev(a.prep.act, act);
            } else if (net_i == a.C && slice == C::SLICES - 1) {
              score[ridx] = (sum + b3sum) / (float)a.C;
            }
            ++tcount;
          }
          if (net_i == 0 && slice == C::SLICES - 1 && n_nets > 1) {     // greedy actions of the block are complete
            __syncwarp();
            if (lane == 0) mbar_arrive(a_ready);
          }
        }
        // fold the block into the (user, chunk) top-k list
        asm volatile("bar.sync 2, 128;");
        {
          const int64_t i0 = (int64_t)chunk * SC_CH * TM;
          const int rows = (int)min((int64_t)tb * TM, a.n_items - i0);
          if (a.k <= 32) {       // order-independent two-pass selection by all four epilogue warps (score.cuh)
            fold_block_select(score, rows, a.items, i0, sv, a.seen_indptr != nullptr, a.k, topS, topI,
                              reinterpret_cast<float*>(sm + C::off_fold(a.k)), tid, 2);
          } else if (warp == 0) {
            for (int base = 0; base < rows; base += 32) {
              const int r = base + lane;
              const float s = r < rows ? score[r] : -INFINITY;
              const int item = r < rows ? a.items[i0 + r] : -1;
              bool cand = item >= 0 && better(s, item, topS[a.k - 1], topI[a.k - 1]);
              if (cand && a.seen_indptr && is_seen(sv, item)) cand = false;
              unsigned m = __ballot_sync(0xffffffffu, cand);
              while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const float s2 = __shfl_sync(0xffffffffu, s, src);
                const int i2 = __shfl_sync(0xffffffffu, item, src);
                if (better(s2, i2, topS[a.k - 1], topI[a.k - 1])) warp_topk_insert(topS, topI, a.k, s2, i2);
              }
            }
          }
        }
        asm volatile("bar.sync 2, 128;");
      }
      float* ps = a.part_s + (size_t)blk * a.k;
      int* pi = a.part_i + (size_t)blk * a.k;
      for (int e = tid; e < a.k; e += 128) { ps[e] = topS[e]; pi[e] = topI[e]; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::MMA_WARP) tmem_dealloc(tmem, C::TMEM_ALLOC);
}

}  // namespace tc
}  // namespace cql
