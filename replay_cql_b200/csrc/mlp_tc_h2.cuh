// mlp_tc_h2.cuh -- the f16x3 hidden-layer kernels on CTA PAIRS (tcgen05 cta_group::2).
//
// Why: in the one-CTA kernels (mlp_tc_h.cuh) a 128-row H1 tile is generated TWICE -- once per 128-column W2 slice,
// because a whole W2 (256 columns, fp16 hi|lo = 256 KB) does not fit one SM's shared memory -- and that CUDA-core
// operand generation, not the tensor pipe, bounds them (ncu r01: 62 % of all executed instructions are the producers',
// tensor pipe 45 %).  A CTA pair holds W2 JOINTLY: each CTA keeps 64 of the 128 operand rows of either pass
// (2 passes x hi|lo x 64 rows x 256 K = 128 KB per CTA), and one `tcgen05.mma.cta_group::2` of shape
// M = 256 (128 rows per CTA), N = 128 reads both halves.  Each CTA's producers therefore generate its 128-row
// H1 tile ONCE (into its own tensor memory, 4 stages of 64 K = the whole K = 256) and the tile feeds both passes:
//   pass 0: D[:, 0:128]   += A(chunks 0..3) x W2[0:128, :]^T     (stages stay full)
//   pass 1: D[:, 128:256] += A(chunks 0..3) x W2[128:256, :]^T   (each stage is released after its pass-1 MMAs)
// The two 128-column accumulators are drained by two epilogue groups, each while the OTHER pass computes, so the
// tensor pipe does not wait for an epilogue; producers refill stage c of the next tile while pass 1 still runs.
//
// Roles per CTA (800 threads): warps 0-7 epilogue (group g = pass g), 8-23 producers, 24 = MMA issuer in the leader
// CTA (cluster rank 0) / W2 loader in the peer.  Cross-CTA signalling: producers and epilogue warps of the peer
// arrive on the LEADER's mbarriers through `mapa` + `mbarrier.arrive.shared::cluster`; the leader's
// `tcgen05.commit ... multicast::cluster` arrives on the same barrier offset in BOTH CTAs.
#pragma once
#include "mlp_tc_h.cuh"

namespace cql {
namespace tc {

// ---- cluster / cta_group::2 PTX wrappers
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster (the CUTLASS ClusterBarrier form).
// No cluster-scope release/acquire qualifiers on purpose: what the barriers order here lives in tensor memory and in
// the async proxy (tcgen05.st / tcgen05.mma / bulk copies, ordered by tcgen05.wait + tcgen05.fence), and an
// `.acquire.cluster` wait makes ptxas emit CCTL.IVALL -- an L1 invalidation -- after EVERY wait (measured: the pair
// kernel was slower than the one-CTA kernel with them).
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_slot, uint32_t ncols) {   // same warp id in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem, 256 x N over the pair] (+)= A[tmem, 128 rows per CTA] * B[smem, N/2 rows per CTA]^T ; leader CTA issues
__device__ __forceinline__ void umma_ts2(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  const uint32_t z = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z)
      : "memory");
}
// all MMAs issued so far arrive (once complete) on the barrier at this offset in the CTAs of `mask`
__device__ __forceinline__ void umma_commit2(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
// x (scaled; ReLU NOT yet applied) -> fp16 hi and lo of relu(x): hi = x truncated to 11 significant bits (mask), lo =
// x - hi (same sign as x: truncation is toward zero), both converted with .relu -- a negative x gives hi = lo = +0, so
// the two FMNMX of the plain path are folded into the conversions (the ALU pipe is the producers' busiest).
__device__ __forceinline__ void split_h2_trunc_relu(float2 x, uint32_t& hi, uint32_t& lo) {
  const float h0 = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
  const float h1 = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
  float2 l;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "sub.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(l.x), "=f"(l.y)
      : "f"(x.x), "f"(x.y), "f"(h0), "f"(h1));
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(h1), "f"(h0));     // first source -> upper half
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(l.y), "f"(l.x));
}

struct H2Cfg {
  static constexpr int NPW = 16, NEW = 8;
  static constexpr int KC = 64, STAGES = 4, NCHUNK = H / KC, UK = 16;
  static constexpr int KPW = KC / (NPW / 4);             // 16 K elements per producer warp per stage
  static constexpr int NP = 128;                         // output columns per pass (UMMA N)
  static constexpr int NLOC = NP / 2;                    // operand rows of a pass held by ONE CTA
  static constexpr int PASSES = H / NP;                  // 2
  static constexpr int PARTS = 2 * PASSES;               // layer-3 partial sums per row: (pass, column half)
  static constexpr int TMP = 2 * TM;                     // rows per pair tile (UMMA M)
  static constexpr int MMA_WARP = NEW + NPW;
  static constexpr int THREADS = (NEW + NPW + 1) * 32;   // 800
  static constexpr int PROD_THREADS = NPW * 32;
  static constexpr uint32_t B_TERM_BYTES = NLOC * H * 2;             // 32 KB
  static constexpr uint32_t B_PASS_BYTES = 2 * B_TERM_BYTES;         // 64 KB (hi | lo)
  static constexpr uint32_t B_BYTES = PASSES * B_PASS_BYTES;         // 128 KB per CTA
  // packed net (global): [cta rank 2][pass 2][term 2][kchunk 32][64 rows][16 B], then HMeta
  static constexpr size_t META_OFF = 2 * (size_t)B_BYTES;
  static constexpr size_t PACKED_NET_BYTES = META_OFF + 2048;
  static constexpr uint32_t A_COL0 = 256, A_STAGE_COLS = KC, A_LO_COLS = KC / 2;
  static constexpr uint32_t OFF_B = 0;
  static constexpr uint32_t OFF_W1 = B_BYTES;                        // float4[256] pair-packed W1|b1
  static constexpr uint32_t OFF_EB = OFF_W1 + H * 16;                // float4[2 passes][128]: b2, w3_0, w3_1, 1/s_n
  static constexpr uint32_t OFF_EF = OFF_EB + PASSES * NP * 16;      // float2[2 passes][128] folded constants
  static constexpr uint32_t OFF_BAR = OFF_EF + PASSES * NP * 8;
  static constexpr uint32_t N_BARS = 2 * STAGES + 2 + 2 + 3;         // full, empty, tfull, tempty, bload, bready, drain
  static constexpr uint32_t OFF_SLOT = OFF_BAR + N_BARS * 8;
  static constexpr uint32_t SMEM_BYTES = OFF_SLOT + 16;
};

// byte offset of the 16-byte chunk (operand row n of 256, K chunk kc, term) inside a pair-packed net
__host__ __device__ constexpr size_t pair_chunk_off(int n, int kc, int term) {
  return (size_t)((n & 127) >> 6) * H2Cfg::B_BYTES + (size_t)(n >> 7) * H2Cfg::B_PASS_BYTES +
         (size_t)term * H2Cfg::B_TERM_BYTES + chunk_off(H2Cfg::NLOC, n & 63, kc);
}

// Same packing as k_pack_multi_h (one warp per operand row: row maximum -> exact power-of-two scale, fp16 hi|lo) into
// the pair layout.  transpose: 0 -> B[n][k] = W2[n][k] (forward), 1 -> B[n][k] = W2[k][n] (dH1 = dZ2 W2).
__global__ void __launch_bounds__(256) k_pack_pair_h(const PackJobs jobs, int out_dim_actor) {
  grid_dep_wait();
  using C = H2Cfg;
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
  *reinterpret_cast<uint4*>(jb.dst + pair_chunk_off(n, kc, 0)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(jb.dst + pair_chunk_off(n, kc, 1)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  HMeta* meta = reinterpret_cast<HMeta*>(jb.dst + C::META_OFF);
  if (kc == 0) meta->inv_s[n] = inv_s;
  if (blockIdx.x == 0) {                                      // maxima of the small layers (scales of the A rows)
    __shared__ int wm[8];
    if (threadIdx.x < 8) wm[threadIdx.x] = 0;
    __syncthreads();
    const int out_dim = jb.in_dim == 2 ? out_dim_actor : 1;
    const int k = threadIdx.x;
    const float* W1 = jb.net + off_W1(jb.in_dim);
    for (int cc = 0; cc < jb.in_dim; ++cc) atomicMax(&wm[cc], __float_as_int(fabsf(W1[k * jb.in_dim + cc])));
    atomicMax(&wm[3], __float_as_int(fabsf(jb.net[off_b1(jb.in_dim) + k])));
    for (int o = 0; o < out_dim; ++o) atomicMax(&wm[4 + o], __float_as_int(fabsf(jb.net[off_W3(jb.in_dim) + o * H + k])));
    __syncthreads();
    if (threadIdx.x < 8) meta->wmax[threadIdx.x] = __int_as_float(wm[threadIdx.x]);
  }
}

// pair items: (job, net, pair tile of 256 rows); a cluster takes a contiguous, cost-balanced range
struct H2Item { int job, net, tp, netkey; };
__device__ __forceinline__ int pair_tiles(int rows) { return (rows + H2Cfg::TMP - 1) / H2Cfg::TMP; }
__device__ __forceinline__ H2Item decode_item_h2(const TcFwdJobs& jobs, const int* pbeg, int item) {
  H2Item it;
  it.job = 0;
  while (it.job + 1 < jobs.n && item >= pbeg[it.job + 1]) ++it.job;
  const int local = item - pbeg[it.job];
  const int tiles = pair_tiles(jobs.j[it.job].rows);
  it.net = local / tiles;
  it.tp = local % tiles;
  it.netkey = it.job * 64 + it.net;
  return it;
}

template <int IN, int OUT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(H2Cfg::THREADS, 1) tc_fwd_h2_kernel(const TcFwdJobs jobs, int swap_b) {
  using C = H2Cfg;
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + C::OFF_B;
  float4* w1p = reinterpret_cast<float4*>(sm + C::OFF_W1);
  float4* ebs = reinterpret_cast<float4*>(sm + C::OFF_EB);
  float2* efs = reinterpret_cast<float2*>(sm + C::OFF_EF);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* full = bars;                         // [STAGES] leader: 2 x NPW producer warps
  uint64_t* empty = bars + C::STAGES;            // [STAGES] both CTAs: multicast commit
  uint64_t* tfull = bars + 2 * C::STAGES;        // [2] both CTAs: multicast commit
  uint64_t* tempty = tfull + 2;                  // [2] leader: 2 x 8 epilogue warps
  uint64_t* bload = tempty + 2;                  // own W2 half landed
  uint64_t* bready = bload + 1;                  // leader: both halves landed
  uint64_t* drain = bready + 1;                  // both CTAs: every MMA issued so far has retired
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  // contiguous pair-item range of this cluster, balanced by cost (items that store H2 are more expensive)
  int pbeg[4];
  int item_lo, item_hi;
  {
    long long cb[4];
    int wj[3];
    cb[0] = 0;
    pbeg[0] = 0;
    for (int j = 0; j < jobs.n; ++j) {
      pbeg[j + 1] = pbeg[j] + jobs.j[j].n_nets * pair_tiles(jobs.j[j].rows);
      wj[j] = jobs.j[j].h2 != nullptr ? (jobs.h2_cost > 0 ? jobs.h2_cost : FWD_H2_COST) : 10;
      cb[j + 1] = cb[j] + (long long)(pbeg[j + 1] - pbeg[j]) * wj[j];
    }
    auto item_at = [&](long long cost) {
      int j = 0;
      while (j + 1 < jobs.n && cost >= cb[j + 1]) ++j;
      const int it = pbeg[j] + (int)((cost - cb[j]) / wj[j]);
      return it < pbeg[j + 1] ? it : pbeg[j + 1];
    };
    const long long total_cost = cb[jobs.n];
    item_lo = cluster_id == 0 ? 0 : item_at(total_cost * cluster_id / n_clusters);
    item_hi = cluster_id == n_clusters - 1 ? pbeg[jobs.n] : item_at(total_cost * (cluster_id + 1) / n_clusters);
  }

  if (warp == C::MMA_WARP) {
    tmem_alloc2(slot, 512);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 2 * C::NPW); mbar_init(&empty[s], 1); }
      for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * C::NEW); }
      mbar_init(bload, 1);
      mbar_init(bready, 2);
      mbar_init(drain, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();           // both CTAs' barriers are initialised before anyone arrives remotely
  tc_fence_after();
  const uint32_t tmem = *slot;
  grid_dep_wait();              // everything above overlapped the predecessor's tail (programmatic dependent launch)

  if (warp == C::MMA_WARP) {
    // ============ leader: W2-half loader + MMA issuer;  peer: W2-half loader ============
    const uint32_t idesc = instr_desc(FMT_F16, C::TMP, C::NP);
    const uint32_t b_lbo = C::NLOC * 16;
    const uint32_t b_base = smem_u32(Bs);
    int cur_key = -1;
    uint32_t nb = 0, nd = 0, tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const H2Item ii = decode_item_h2(jobs, pbeg, item);
      if (ii.netkey != cur_key) {
        if (cur_key >= 0) {                         // the old W2 must not be overwritten while MMAs still read it
          if (leader && elect_one()) umma_commit2(drain, 3);
          __syncwarp();
          mbar_wait_cluster(drain, nd & 1);
          ++nd;
        }
        const TcFwdJob& jb = jobs.j[ii.job];
        const uint8_t* src = jb.packed + (size_t)ii.net * C::PACKED_NET_BYTES + (size_t)(rank ^ (uint32_t)swap_b) * C::B_BYTES;
        if (elect_one()) {
          mbar_arrive_expect_tx(bload, C::B_BYTES);
          for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bload);
        }
        __syncwarp();
        mbar_wait(bload, nb & 1);
        if (elect_one()) mbar_arrive_cluster(bready, 0);
        __syncwarp();
        if (leader) mbar_wait_cluster(bready, nb & 1);
        ++nb;
        cur_key = ii.netkey;
      }
      if (!leader) continue;
      for (int p = 0; p < C::PASSES; ++p) {
        mbar_wait_cluster(&tempty[p], (tcount & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem + p * C::NP;
        const uint32_t bp = b_base + p * C::B_PASS_BYTES;
        for (int c = 0; c < C::NCHUNK; ++c) {
          if (p == 0) {
            mbar_wait_cluster(&full[c], tcount & 1);
            tc_fence_after();
          }
          if (elect_one()) {
            const uint32_t a_stage = tmem + C::A_COL0 + c * C::A_STAGE_COLS;
#pragma unroll
            for (int j = 0; j < C::KC / C::UK; ++j) {
              const uint32_t g = c * (C::KC / C::UK) + j;
              const uint64_t b_hi = smem_desc(bp + 2 * g * b_lbo, b_lbo, 128);
              const uint64_t b_lo = smem_desc(bp + C::B_TERM_BYTES + 2 * g * b_lbo, b_lbo, 128);
              const uint32_t a_hi = a_stage + j * 8, a_lo = a_hi + C::A_LO_COLS;
              umma_ts2(d_tmem, a_lo, b_hi, idesc, (c == 0 && j == 0) ? 0u : 1u);
              umma_ts2(d_tmem, a_hi, b_lo, idesc, 1u);
              umma_ts2(d_tmem, a_hi, b_hi, idesc, 1u);
            }
            if (p == C::PASSES - 1) umma_commit2(&empty[c], 3);      // stage reusable in both CTAs
            if (c == C::NCHUNK - 1) umma_commit2(&tfull[p], 3);      // accumulator p complete in both CTAs
          }
          __syncwarp();
        }
      }
      ++tcount;
    }
  } else if (warp >= C::NEW) {
    // ============ producers (both CTAs): layer 1 of the CTA's 128 rows -> scaled fp16 hi|lo -> own TMEM ============
    const int pw = warp - C::NEW, ptid = tid - C::NEW * 32;
    const int kq = pw >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + kq * (C::KPW / 2);
    int cur_key = -1;
    float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t tcount = 0;
    auto load_x = [&](const H2Item& ni) {
      const TcFwdJob& nj = jobs.j[ni.job];
      const int r = ni.tp * C::TMP + (int)rank * TM + (warp & 3) * 32 + lane;
      return r < nj.rows ? __ldg(nj.X + r) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    float4 x_next = make_float4(0.f, 0.f, 0.f, 0.f);
    H2Item ii_next = item_lo < item_hi ? decode_item_h2(jobs, pbeg, item_lo) : H2Item{};
    for (int item = item_lo; item < item_hi; ++item, ++tcount) {
      const H2Item ii = ii_next;
      if (item + 1 < item_hi) ii_next = decode_item_h2(jobs, pbeg, item + 1);
      const TcFwdJob& jb = jobs.j[ii.job];
      if (ii.netkey != cur_key) {
        cur_key = ii.netkey;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        const float* net = jb.params + (size_t)ii.net * NET_STRIDE;
        for (int pr = ptid; pr < H / 2; pr += C::PROD_THREADS) {
          const int k = 2 * pr;
          const float* wa = net + off_W1(IN) + k * IN;
          const float* wb = wa + IN;
          w1p[2 * pr] = make_float4(wa[0], wb[0], wa[1], wb[1]);
          w1p[2 * pr + 1] = make_float4(IN == 3 ? wa[2] : 0.f, IN == 3 ? wb[2] : 0.f, net[off_b1(IN) + k], net[off_b1(IN) + k + 1]);
        }
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packed + (size_t)ii.net * C::PACKED_NET_BYTES + C::META_OFF);
        wm = make_float4(__ldg(&meta->wmax[0]), __ldg(&meta->wmax[1]), IN == 3 ? __ldg(&meta->wmax[2]) : 0.f, __ldg(&meta->wmax[3]));
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      }
      const float4 x = (item == item_lo) ? load_x(ii) : x_next;
      if (item + 1 < item_hi) x_next = load_x(ii_next);
      float sa, inv_sa;
      pow2_scale(h1_row_bound(x, wm), sa, inv_sa);
      const float2 xx = make_float2(x.x, x.x), xy = make_float2(x.y, x.y), xz = make_float2(x.z, x.z), ss = make_float2(sa, sa);
      for (int c = 0; c < C::NCHUNK; ++c) {
        uint32_t hi[C::KPW / 2], lo[C::KPW / 2];
#pragma unroll
        for (int pp = 0; pp < C::KPW / 2; ++pp) {
          const int pr = (c * C::KC + kq * C::KPW) / 2 + pp;
          const float4 wA = w1p[2 * pr], wB = w1p[2 * pr + 1];
          float2 v = ffma2(xx, make_float2(wA.x, wA.y), make_float2(wB.z, wB.w));   // chain starts from the bias
          v = ffma2(xy, make_float2(wA.z, wA.w), v);
          if (IN == 3) v = ffma2(xz, make_float2(wB.x, wB.y), v);
          split_h2_trunc_relu(fmul2(v, ss), hi[pp], lo[pp]);                         // exact: power-of-two scale; ReLU in the cvt
        }
        mbar_wait_cluster(&empty[c], (tcount & 1) ^ 1);           // values are ready before the stage is: wait late
        tc_fence_after();
        tmem_st8(lane_base + c * C::A_STAGE_COLS, hi);
        tmem_st8(lane_base + c * C::A_STAGE_COLS + C::A_LO_COLS, lo);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&full[c], 0);
      }
    }
    // the leader's last multicast commits land in THIS CTA's barriers: do not exit before they have
    if (item_hi > item_lo)
      for (int c = 0; c < C::NCHUNK; ++c) mbar_wait_cluster(&empty[c], (tcount & 1) ^ 1);
  } else {
    // ============ epilogue (both CTAs): unscale -> +b2 -> ReLU -> layer 3 (+ H2) ============
    // ALL eight warps drain pass 0's accumulator (warp w: TMEM lane quarter w % 4, column half w / 4 = 64 columns),
    // then pass 1's.  An accumulator is single-buffered (tensor memory: 256 columns of A + 2 x 128 of D), so the MMA of
    // pass p of the NEXT tile waits for this drain; with one 4-warp group per pass the drain of a 128-column
    // accumulator had to fit into the other pass's 3 k clocks (measured 4-5 k on the tiles that store H2: the tensor
    // pipe idled), with eight warps on each accumulator it takes half as long against the same budget.
    const int hh = warp >> 2, qw = warp & 3;
    int cur_key = -1;
    const int row_in_tile = (int)rank * TM + qw * 32 + lane;
    float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t tcount = 0;
    for (int item = item_lo; item < item_hi; ++item, ++tcount) {
      const H2Item ii = decode_item_h2(jobs, pbeg, item);
      const TcFwdJob& jb = jobs.j[ii.job];
      if (ii.netkey != cur_key) {
        cur_key = ii.netkey;
        asm volatile("bar.sync 2, 256;");
        const float* net = jb.params + (size_t)ii.net * NET_STRIDE;
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packed + (size_t)ii.net * C::PACKED_NET_BYTES + C::META_OFF);
        {
          const int col = tid;                       // 256 epilogue threads = 256 output columns
          const float inv_n = __ldg(&meta->inv_s[col]);
          ebs[col] = make_float4(net[off_b2(IN) + col], net[off_W3(IN) + col],
                                 OUT == 2 ? net[off_W3(IN) + H + col] : 0.f, inv_n);
          // folded form for items that do not store H2 (exact, powers of two):
          // relu(v/(s_m s_n) + b2) w3 = relu(v/s_m + b2 s_n) (w3/s_n); pairs of columns (b2'_c, b2'_c+1, w3'_c, w3'_c+1)
          if (OUT == 1) {
            float* ef = reinterpret_cast<float*>(efs) + (col >> 1) * 4 + (col & 1);
            ef[0] = net[off_b2(IN) + col] / inv_n;
            ef[2] = net[off_W3(IN) + col] * inv_n;
          }
        }
        wm = make_float4(__ldg(&meta->wmax[0]), __ldg(&meta->wmax[1]), IN == 3 ? __ldg(&meta->wmax[2]) : 0.f, __ldg(&meta->wmax[3]));
        asm volatile("bar.sync 2, 256;");
      }
      const int row = ii.tp * C::TMP + row_in_tile;
      const float4 x = row < jb.rows ? __ldg(jb.X + row) : make_float4(0.f, 0.f, 0.f, 0.f);
      float sa, inv_sa;
      pow2_scale(h1_row_bound(x, wm), sa, inv_sa);                 // the producers' scale of this row, recomputed
      const bool store_h2 = jb.h2 != nullptr;
      const int tiles64 = (jb.rows + 63) / 64;
#pragma unroll 1
      for (int p = 0; p < C::PASSES; ++p) {
        constexpr int NC = C::NP / 2;                              // 64 columns per warp per pass
        const int cb = p * C::NP + hh * NC;                        // first output column of this warp in this pass
        mbar_wait(&tfull[p], tcount & 1);
        tc_fence_after();
        float* h2row = store_h2 ? jb.h2 + (((size_t)ii.net * tiles64 + (row >> 6)) * H + cb) * 64 + (row & 63) : nullptr;
        const uint32_t t_acc = tmem + ((uint32_t)(qw * 32) << 16) + cb;
        float q0 = 0.f, q1 = 0.f;
        // The per-column constants are warp-uniform shared-memory loads, fetched in BATCHES (issued back to back,
        // together with the TMEM load) before the math of a step: interleaved one by one each LDS exposed its
        // ~30-clock latency inside the dependent chain.
        if (OUT == 1 && !store_h2) {
          const float2 isa2 = make_float2(inv_sa, inv_sa);
          const float4* ef4 = reinterpret_cast<const float4*>(efs) + (cb >> 1);   // (b2'_c, b2'_c+1, w3'_c, w3'_c+1)
          float2 qa = make_float2(0.f, 0.f), qb = make_float2(0.f, 0.f);
#pragma unroll 1
          for (int c0 = 0; c0 < NC; c0 += 16) {
            float v[16];
            float4 e[8];
            tmem_ld16(t_acc + c0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) e[j] = ef4[(c0 >> 1) + j];
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
              float2 ha = ffma2(make_float2(v[2 * j], v[2 * j + 1]), isa2, make_float2(e[j].x, e[j].y));
              float2 hb = ffma2(make_float2(v[2 * j + 2], v[2 * j + 3]), isa2, make_float2(e[j + 1].x, e[j + 1].y));
              ha.x = fmaxf(ha.x, 0.f); ha.y = fmaxf(ha.y, 0.f);
              hb.x = fmaxf(hb.x, 0.f); hb.y = fmaxf(hb.y, 0.f);
              qa = ffma2(ha, make_float2(e[j].z, e[j].w), qa);
              qb = ffma2(hb, make_float2(e[j + 1].z, e[j + 1].w), qb);
            }
          }
          q0 = (qa.x + qa.y) + (qb.x + qb.y);
        } else {
          const float4* ebg = ebs + cb;
          float q0b = 0.f, q1b = 0.f;
#pragma unroll 1
          for (int c0 = 0; c0 < NC; c0 += 8) {
            float v[8];
            float4 e[8];
            tmem_ld8(t_acc + c0, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) e[i] = ebg[c0 + i];
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; i += 2) {
              const float ha = fmaxf(fmaf(v[i] * inv_sa, e[i].w, e[i].x), 0.f);
              const float hb = fmaxf(fmaf(v[i + 1] * inv_sa, e[i + 1].w, e[i + 1].x), 0.f);
              v[i] = ha;
              v[i + 1] = hb;
              q0 = fmaf(ha, e[i].y, q0);
              q0b = fmaf(hb, e[i + 1].y, q0b);
              if (OUT == 2) { q1 = fmaf(ha, e[i].z, q1); q1b = fmaf(hb, e[i + 1].z, q1b); }
            }
            if (store_h2 && (row >> 6) < tiles64) {
#pragma unroll
              for (int i = 0; i < 8; ++i) h2row[(size_t)(c0 + i) * 64] = v[i];
            }
          }
          q0 += q0b;
          q1 += q1b;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&tempty[p], 0);
        if (row < jb.rows) {
          float* o = jb.out_part + (((size_t)ii.net * C::PARTS + p * 2 + hh) * jb.rows + row) * OUT;
          o[0] = q0;
          if (OUT == 2) o[1] = q1;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();           // the peer's TMEM / barriers stay alive until the leader's last MMA has retired
  if (warp == C::MMA_WARP) tmem_dealloc2(tmem, 512);
}


// ---------------------------------------------------------------------------------------------------------------
// Input gradient of the hidden layer on CTA pairs: dH1 = dZ2 W2 (A = the CTA's 128 dZ2 rows, generated ONCE per pair
// tile from dOut, W3 and the stored H2; B = W2^T in the pair layout), then dZ1 = dH1 * relu'(Z1), dW1/db1 column sums
// and (optionally) dx -- the epilogue of tc_bwd1_h_kernel, group g on the columns of pass g.
struct H2B1Cfg : H2Cfg {
  static constexpr uint32_t OFF_W3 = B_BYTES;                        // float2[256] (W3[0][j], W3[1][j])
  static constexpr uint32_t OFF_EB = OFF_W3 + H * 8;                 // float4[2 passes][128]: W1[k][0..2], b1[k]
  static constexpr uint32_t OFF_IV = OFF_EB + PASSES * NP * 16;      // float[2][128] 1/s_n
  static constexpr uint32_t OFF_BAR = OFF_IV + PASSES * NP * 4;
  static constexpr uint32_t OFF_SLOT = OFF_BAR + 128;                // (N_BARS * 8 = 120, rounded up: what follows holds float4)
  static constexpr uint32_t OFF_FLUSH = OFF_SLOT + 16;               // float[2 groups][4 warps][16][32]
  static constexpr uint32_t OFF_RED = OFF_FLUSH + 2 * 4 * 16 * 32 * 4;
  static constexpr int RED_LD = 34;                                  // row stride of the transposed tile: 8-byte aligned pair stores, conflict-free
  static constexpr uint32_t RED_WARP_BYTES = 32 * RED_LD * 4 + 32 * 16;
  static constexpr uint32_t SMEM_BYTES = OFF_RED + NEW * RED_WARP_BYTES;
};

template <int IN, int OUT, bool WGRADS, bool DX>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(H2Cfg::THREADS, 1) tc_bwd1_h2_kernel(const Bwd1Job jb, int swap_b) {
  using C = H2B1Cfg;
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + C::OFF_B;
  float2* w3s = reinterpret_cast<float2*>(sm + C::OFF_W3);
  float4* ebs = reinterpret_cast<float4*>(sm + C::OFF_EB);
  float* invs = reinterpret_cast<float*>(sm + C::OFF_IV);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bload = tempty + 2;
  uint64_t* bready = bload + 1;
  uint64_t* drain = bready + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  const int tiles = pair_tiles(jb.rows);
  const int tiles64 = (jb.rows + 63) / 64;
  const int total = jb.n_nets * tiles;
  const int item_lo = (int)((long long)total * cluster_id / n_clusters);
  const int item_hi = (int)((long long)total * (cluster_id + 1) / n_clusters);

  if (warp == C::MMA_WARP) {
    tmem_alloc2(slot, 512);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 2 * C::NPW); mbar_init(&empty[s], 1); }
      for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * C::NEW); }
      mbar_init(bload, 1);
      mbar_init(bready, 2);
      mbar_init(drain, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *slot;
  grid_dep_wait();
  if (WGRADS) zero_small1_slots<IN>(jb, 2);          // slots (CTA, column half)

  if (warp == C::MMA_WARP) {
    const uint32_t idesc = instr_desc(FMT_F16, C::TMP, C::NP);
    const uint32_t b_lbo = C::NLOC * 16;
    const uint32_t b_base = smem_u32(Bs);
    int cur_net = -1;
    uint32_t nb = 0, nd = 0, tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int net_i = item / tiles;
      if (net_i != cur_net) {
        if (cur_net >= 0) {
          if (leader && elect_one()) umma_commit2(drain, 3);
          __syncwarp();
          mbar_wait_cluster(drain, nd & 1);
          ++nd;
        }
        const uint8_t* src = jb.packedT + (size_t)net_i * C::PACKED_NET_BYTES + (size_t)(rank ^ (uint32_t)swap_b) * C::B_BYTES;
        if (elect_one()) {
          mbar_arrive_expect_tx(bload, C::B_BYTES);
          for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bload);
        }
        __syncwarp();
        mbar_wait(bload, nb & 1);
        if (elect_one()) mbar_arrive_cluster(bready, 0);
        __syncwarp();
        if (leader) mbar_wait_cluster(bready, nb & 1);
        ++nb;
        cur_net = net_i;
      }
      if (!leader) continue;
      for (int p = 0; p < C::PASSES; ++p) {
        mbar_wait_cluster(&tempty[p], (tcount & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem + p * C::NP;
        const uint32_t bp = b_base + p * C::B_PASS_BYTES;
        for (int c = 0; c < C::NCHUNK; ++c) {
          if (p == 0) {
            mbar_wait_cluster(&full[c], tcount & 1);
            tc_fence_after();
          }
          if (elect_one()) {
            const uint32_t a_stage = tmem + C::A_COL0 + c * C::A_STAGE_COLS;
#pragma unroll
            for (int j = 0; j < C::KC / C::UK; ++j) {
              const uint32_t g = c * (C::KC / C::UK) + j;
              const uint64_t b_hi = smem_desc(bp + 2 * g * b_lbo, b_lbo, 128);
              const uint64_t b_lo = smem_desc(bp + C::B_TERM_BYTES + 2 * g * b_lbo, b_lbo, 128);
              const uint32_t a_hi = a_stage + j * 8, a_lo = a_hi + C::A_LO_COLS;
              umma_ts2(d_tmem, a_lo, b_hi, idesc, (c == 0 && j == 0) ? 0u : 1u);
              umma_ts2(d_tmem, a_hi, b_lo, idesc, 1u);
              umma_ts2(d_tmem, a_hi, b_hi, idesc, 1u);
            }
            if (p == C::PASSES - 1) umma_commit2(&empty[c], 3);
            if (c == C::NCHUNK - 1) umma_commit2(&tfull[p], 3);
          }
          __syncwarp();
        }
      }
      ++tcount;
    }
  } else if (warp >= C::NEW) {
    // ---------------- producers: the CTA's 128 dZ2 rows -> scaled fp16 hi|lo -> own TMEM (once per pair tile) ----------------
    const int pw = warp - C::NEW, ptid = tid - C::NEW * 32;
    const int kq = pw >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + kq * (C::KPW / 2);
    int cur_net = -1;
    float w3m0 = 0.f, w3m1 = 0.f;
    uint32_t tcount = 0;
    for (int item = item_lo; item < item_hi; ++item, ++tcount) {
      const int net_i = item / tiles, tp = item % tiles;
      if (net_i != cur_net) {
        cur_net = net_i;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        for (int j = ptid; j < H; j += C::PROD_THREADS)
          w3s[j] = make_float2(net[off_W3(IN) + j], OUT == 2 ? net[off_W3(IN) + H + j] : 0.f);
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packedT + (size_t)net_i * C::PACKED_NET_BYTES + C::META_OFF);
        w3m0 = __ldg(&meta->wmax[4]);
        w3m1 = OUT == 2 ? __ldg(&meta->wmax[5]) : 0.f;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      }
      const int r = tp * C::TMP + (int)rank * TM + (warp & 3) * 32 + lane;
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
      for (int c = 0; c < C::NCHUNK; ++c) {
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
        mbar_wait_cluster(&empty[c], (tcount & 1) ^ 1);
        tc_fence_after();
        tmem_st8(lane_base + c * C::A_STAGE_COLS, hi);
        tmem_st8(lane_base + c * C::A_STAGE_COLS + C::A_LO_COLS, lo);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&full[c], 0);
      }
    }
    if (item_hi > item_lo)
      for (int c = 0; c < C::NCHUNK; ++c) mbar_wait_cluster(&empty[c], (tcount & 1) ^ 1);
  } else {
    // ---------------- epilogue: dZ1 = dH1 * relu'(Z1), dx, dW1/db1 column sums ----------------
    // All eight warps drain pass 0's accumulator, then pass 1's (warp w: lane quarter w % 4, column half w / 4 =
    // 64 columns of each pass) -- see the forward kernel for why.
    constexpr int NC = C::NP / 2;                          // 64 columns per warp per pass
    constexpr int NCH = NC / 32;                           // 2 chunks of 32 columns
    const int hh = warp >> 2, qw = warp & 3, gtid = tid & 127;
    float a_b[C::PASSES][NCH], a_w0[C::PASSES][NCH], a_w1[C::PASSES][NCH], a_w2[C::PASSES][NCH];   // lane l <-> column
#pragma unroll
    for (int p = 0; p < C::PASSES; ++p)
#pragma unroll
      for (int q = 0; q < NCH; ++q) { a_b[p][q] = 0.f; a_w0[p][q] = 0.f; a_w1[p][q] = 0.f; a_w2[p][q] = 0.f; }
    float* flbuf = reinterpret_cast<float*>(sm + C::OFF_FLUSH) + hh * (4 * 16 * 32);
    float* red_t = reinterpret_cast<float*>(sm + C::OFF_RED + warp * C::RED_WARP_BYTES);       // [32][33]
    float4* red_x = reinterpret_cast<float4*>(red_t + 32 * C::RED_LD);                          // [32] this item's input rows
    auto flush = [&](int net_i) {                    // called uniformly by the 4 warps of a column half
      if (!WGRADS || net_i < 0) return;
#pragma unroll
      for (int p = 0; p < C::PASSES; ++p)
#pragma unroll
        for (int q = 0; q < NCH; ++q) {
          float* f = flbuf + (qw * 16 + (p * NCH + q) * 4) * 32 + lane;
          f[0] = a_w0[p][q]; f[32] = a_w1[p][q]; f[64] = a_w2[p][q]; f[96] = a_b[p][q];
          a_b[p][q] = 0.f; a_w0[p][q] = 0.f; a_w1[p][q] = 0.f; a_w2[p][q] = 0.f;
        }
      asm volatile("bar.sync %0, 128;" ::"r"(2 + hh));
      float* o = jb.small1 + ((size_t)net_i * jb.slots + blockIdx.x * 2 + hh) * SMALL_STRIDE;
      {
        const int pq = qw;                           // warp w sums chunk (p, q) = w over the four warps (order 0..3)
        float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float* f = flbuf + (w * 16 + pq * 4) * 32 + lane;
          t0 += f[0]; t1 += f[32]; t2 += f[64]; t3 += f[96];
        }
        const int k = (pq / NCH) * C::NP + hh * NC + (pq % NCH) * 32 + lane;
        o[k * IN + 0] = t0;
        o[k * IN + 1] = t1;
        if (IN == 3) o[k * IN + 2] = t2;
        o[H * IN + k] = t3;
      }
      asm volatile("bar.sync %0, 128;" ::"r"(2 + hh));
    };
    int cur_net = -1;
    float w3m0 = 0.f, w3m1 = 0.f;
    uint32_t tcount = 0;
    for (int item = item_lo; item < item_hi; ++item, ++tcount) {
      const int net_i = item / tiles, tp = item % tiles;
      if (net_i != cur_net) {
        flush(cur_net);
        cur_net = net_i;
        asm volatile("bar.sync 4, 256;");
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        const HMeta* meta = reinterpret_cast<const HMeta*>(jb.packedT + (size_t)net_i * C::PACKED_NET_BYTES + C::META_OFF);
        {
          const int k = tid;                          // 256 epilogue threads = 256 hidden units
          // column PAIRS (k even, k + 1): ebs[k] = (wx_k, wx_k1, wy_k, wy_k1), ebs[k + 1] = (wz_k, wz_k1, b_k, b_k1)
          float* e = reinterpret_cast<float*>(ebs) + (k >> 1) * 8 + (k & 1);
          e[0] = net[off_W1(IN) + k * IN];
          e[2] = net[off_W1(IN) + k * IN + 1];
          e[4] = IN == 3 ? net[off_W1(IN) + k * IN + 2] : 0.f;
          e[6] = net[off_b1(IN) + k];
          invs[k] = __ldg(&meta->inv_s[k]);
        }
        w3m0 = __ldg(&meta->wmax[4]);
        w3m1 = OUT == 2 ? __ldg(&meta->wmax[5]) : 0.f;
        asm volatile("bar.sync 4, 256;");
      }
      const int row = tp * C::TMP + (int)rank * TM + qw * 32 + lane;
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
        red_x[lane] = make_float4(x.x, x.y, x.z, 1.f);                        // rows beyond jb.rows: x = 0, dZ1 = 0
      }
#pragma unroll
      for (int p = 0; p < C::PASSES; ++p) {
        const int cb = p * C::NP + hh * NC;
        const float4* ebg = ebs + cb;
        const float* ivg = invs + cb;
        mbar_wait(&tfull[p], tcount & 1);
        tc_fence_after();
        const uint32_t t_acc = tmem + ((uint32_t)(qw * 32) << 16) + cb;
        float dx0 = 0.f, dx1 = 0.f, dx2 = 0.f;
#pragma unroll
        for (int q = 0; q < NCH; ++q) {                   // (unrolled: a_w*[p][q] must stay in registers)
          if (WGRADS) __syncwarp();                       // the previous chunk's column sums have read red_t
          // 8 columns per step: the TMEM load and the step's constants (warp-uniform LDS) are issued together, then the
          // math -- one LDS per column inside the dependent chain made this epilogue latency-bound (ncu r02)
#pragma unroll 1
          for (int c8 = 0; c8 < 32; c8 += 8) {
            float v[8];
            float4 w[8];                                  // 4 column pairs x {(wx, wx', wy, wy'), (wz, wz', b, b')}
            float iv[8];
            tmem_ld8(t_acc + q * 32 + c8, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = ebg[q * 32 + c8 + i];
            if (DX) {
              const float4 i0 = *reinterpret_cast<const float4*>(ivg + q * 32 + c8);
              const float4 i1 = *reinterpret_cast<const float4*>(ivg + q * 32 + c8 + 4);
              iv[0] = i0.x; iv[1] = i0.y; iv[2] = i0.z; iv[3] = i0.w; iv[4] = i1.x; iv[5] = i1.y; iv[6] = i1.z; iv[7] = i1.w;
            }
            tmem_ld_wait();
            const float2 xx2 = make_float2(x.x, x.x), xy2 = make_float2(x.y, x.y), xz2 = make_float2(x.z, x.z);
            const float2 isa2 = make_float2(inv_sa, inv_sa);
#pragma unroll
            for (int i = 0; i < 8; i += 2) {              // columns c8 + i, c8 + i + 1: packed fp32x2 arithmetic
              const float4 wa = w[i], wb = w[i + 1];
              // layer-1 pre-activation in the FORWARD's order (chain starts from the bias): same ReLU mask bit for bit
              float2 z = ffma2(xy2, make_float2(wa.z, wa.w), ffma2(xx2, make_float2(wa.x, wa.y), make_float2(wb.z, wb.w)));
              if (IN == 3) z = ffma2(xz2, make_float2(wb.x, wb.y), z);
              // without dx the column scale 1/s_n is applied once per column sum instead of once per element
              float2 vs = fmul2(make_float2(v[i], v[i + 1]), isa2);
              if (DX) vs = fmul2(vs, make_float2(iv[i], iv[i + 1]));
              const float2 d = make_float2(z.x > 0.f ? vs.x : 0.f, z.y > 0.f ? vs.y : 0.f);
              if (DX) {
                dx0 = fmaf(d.x, wa.x, dx0); dx0 = fmaf(d.y, wa.y, dx0);
                dx1 = fmaf(d.x, wa.z, dx1); dx1 = fmaf(d.y, wa.w, dx1);
                if (IN == 3) { dx2 = fmaf(d.x, wb.x, dx2); dx2 = fmaf(d.y, wb.y, dx2); }
              }
              if (WGRADS) *reinterpret_cast<float2*>(red_t + lane * C::RED_LD + c8 + i) = d;
            }
          }
          if (WGRADS) {
            // column sums over the warp's 32 rows through the transposed shared-memory tile (fixed row order); packed
            // FMAs on (x0, x1) and (x2, 1)
            __syncwarp();
            float2 s01 = make_float2(0.f, 0.f), s2b = make_float2(0.f, 0.f);
#pragma unroll 8
            for (int r = 0; r < 32; ++r) {
              const float dv = red_t[r * C::RED_LD + lane];
              const float4 xr = red_x[r];
              const float2 dd = make_float2(dv, dv);
              s01 = ffma2(dd, make_float2(xr.x, xr.y), s01);
              s2b = ffma2(dd, make_float2(xr.z, xr.w), s2b);
            }
            const float cs = DX ? 1.f : ivg[q * 32 + lane];
            a_w0[p][q] = fmaf(s01.x, cs, a_w0[p][q]); a_w1[p][q] = fmaf(s01.y, cs, a_w1[p][q]);
            a_w2[p][q] = fmaf(s2b.x, cs, a_w2[p][q]); a_b[p][q] = fmaf(s2b.y, cs, a_b[p][q]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&tempty[p], 0);
        if (DX && ok)
          jb.dX_part[((size_t)net_i * C::PARTS + p * 2 + hh) * jb.rows + row] = make_float4(dx0, dx1, dx2, 0.f);
      }
    }
    flush(cur_net);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == C::MMA_WARP) tmem_dealloc2(tmem, 512);
}


// ---------------------------------------------------------------------------------------------------------------
// Weight gradient of the hidden layer on CTA pairs: dW2[j][k] = sum_r dZ2[r][j] H1[r][k], contraction over batch rows.
// The one-CTA kernel (tc_bwd2_h_kernel) reads BOTH operands from shared memory -- an SS-mode MMA of N = 256 takes
// 171 clocks instead of 128 (cql_mma_bench, profiles/r02_mma_issue_rate.txt) and the port also carries the producers'
// stores: tensor pipe 21 %.  Here the 256 x 256 accumulator is split over a pair: CTA c owns the output rows
// j in [128c, 128c + 128) (its 128 TMEM lanes, all 256 columns = 256 of its 512 TMEM columns) and holds the operand rows
// k in [128c, 128c + 128) of B = H1^T in shared memory; `tcgen05.mma.cta_group::2` (M = 256, N = 256) reads both halves.
// That frees 256 TMEM columns for the A operand (dZ2^T: lane = j, columns = batch rows, two fp16 each), so the MMA runs
// in TS mode at its 128-clock floor, and each CTA generates only HALF of either operand: producer thread (unit u, row
// group g) owns hidden unit 128c + u for 8 of a stage's 32 rows and writes dZ2[.][unit] to tensor memory and
// H1[.][unit] to shared memory, as scaled fp16 hi|lo (scales per hidden unit, as in tc_bwd2_h_kernel).
struct B2PCfg {
  static constexpr int RS = 32;                             // batch rows (K extent) per stage
  static constexpr int STAGES = 4;
  static constexpr int PROD_WARPS = 16;                     // 4 lane quarters x 4 row groups of 8 rows
  static constexpr int PROD_THREADS = PROD_WARPS * 32;
  static constexpr int MMA_WARP = PROD_WARPS;
  static constexpr int THREADS = PROD_THREADS + 32;
  static constexpr int HU = H / 2;                          // hidden units per CTA (128)
  static constexpr uint32_t B_TERM_BYTES = HU * RS * 2;     // 8 KB
  static constexpr uint32_t B_STAGE_BYTES = 2 * B_TERM_BYTES;   // hi | lo
  static constexpr uint32_t A_COL0 = 256, A_STAGE_COLS = RS, A_LO_COLS = RS / 2;
  static constexpr int SS_ROWS = 4 * RS;                         // rows of a super-stage (x / dOut staged 4 stages at a time)
  static constexpr uint32_t OFF_X = STAGES * B_STAGE_BYTES;     // float[3][2][SS_ROWS]: x.x | x.y | x.z, double-buffered
  static constexpr uint32_t OFF_SS = OFF_X + 3 * 2 * SS_ROWS * 4;   // float[2][2][SS_ROWS]: dOut[.][0] | dOut[.][1]
  static constexpr uint32_t OFF_INV = OFF_SS + 2 * 2 * SS_ROWS * 4; // float invA[128] (own units) | invB[256]
  static constexpr uint32_t OFF_SMALL = OFF_INV + (HU + H) * 4; // float4[3][128]: row groups 1..3: db2 | dW3[0..1] | db3_0
  static constexpr uint32_t OFF_MAX = OFF_SMALL + 3 * HU * 16;  // int[8] row maxima (float bits)
  static constexpr uint32_t OFF_BAR = OFF_MAX + 32;
  static constexpr uint32_t OFF_SLOT = OFF_BAR + (2 * STAGES + 1) * 8 + 8;
  static constexpr uint32_t BYTES = OFF_SLOT + 16;
};

template <int IN, int OUT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(B2PCfg::THREADS, 1) tc_bwd2_h2_kernel(const Bwd2Job jb) {
  using C = B2PCfg;
  extern __shared__ __align__(1024) uint8_t sm[];
  float4* xs = reinterpret_cast<float4*>(sm + C::OFF_X);
  float* invA = reinterpret_cast<float*>(sm + C::OFF_INV);
  float* invB = invA + C::HU;
  float4* small_g = reinterpret_cast<float4*>(sm + C::OFF_SMALL);
  int* rmax = reinterpret_cast<int*>(sm + C::OFF_MAX);
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);     // leader: 2 x PROD_WARPS
  uint64_t* empty = full + C::STAGES;                                // both CTAs: multicast commit
  uint64_t* done = empty + C::STAGES;                                // both CTAs: multicast commit
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int split = blockIdx.x >> 1, net_i = blockIdx.y;
  const float* net = jb.params + (size_t)net_i * NET_STRIDE;
  const int tiles64 = (jb.rows + 63) / 64;
  const int n_stage_total = (jb.rows + C::RS - 1) / C::RS;
  const int st_lo = (int)((long long)n_stage_total * split / jb.splits);
  const int st_hi = (int)((long long)n_stage_total * (split + 1) / jb.splits);

  if (warp == C::MMA_WARP) {
    tmem_alloc2(slot, 512);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 2 * C::PROD_WARPS); mbar_init(&empty[s], 1); }
      mbar_init(done, 1);
      fence_mbar_init();
    }
  }
  if (tid < 8) rmax[tid] = 0;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *slot;
  grid_dep_wait();

  if (warp == C::MMA_WARP) {
    if (leader) {
      const uint32_t idesc = instr_desc(FMT_F16, 256, 256);
      const uint32_t lbo = C::HU * 16;
      uint32_t it = 0;
      for (int sg = st_lo; sg < st_hi; ++sg, ++it) {
        const uint32_t s = it % C::STAGES;
        mbar_wait(&full[s], (it / C::STAGES) & 1);
        tc_fence_after();
        const uint32_t b_base = smem_u32(sm + s * C::B_STAGE_BYTES);
        const uint32_t a_stage = tmem + C::A_COL0 + s * C::A_STAGE_COLS;
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < C::RS / 16; ++j) {
            const uint64_t b_hi = smem_desc(b_base + 2 * j * lbo, lbo, 128);
            const uint64_t b_lo = smem_desc(b_base + C::B_TERM_BYTES + 2 * j * lbo, lbo, 128);
            const uint32_t a_hi = a_stage + j * 8, a_lo = a_hi + C::A_LO_COLS;
            umma_ts2(tmem, a_lo, b_hi, idesc, (it == 0 && j == 0) ? 0u : 1u);
            umma_ts2(tmem, a_hi, b_lo, idesc, 1u);
            umma_ts2(tmem, a_hi, b_hi, idesc, 1u);
          }
          umma_commit2(&empty[s], 3);
          if (sg == st_hi - 1) umma_commit2(done, 3);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------- producers: thread (u, g): hidden unit 128 rank + u, rows 8g .. 8g + 8 of every stage ----------------
    const int u = (warp & 3) * 32 + lane, g = warp >> 2;
    const int t = (int)rank * C::HU + u;                      // global hidden unit: A row j = t, B row k = t
    float w3[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) w3[o] = net[off_W3(IN) + o * H + t];
    const float w1x = net[off_W1(IN) + t * IN], w1y = net[off_W1(IN) + t * IN + 1];
    const float w1z = IN == 3 ? net[off_W1(IN) + t * IN + 2] : 0.f;
    const float b1v = net[off_b1(IN) + t];
    // pre-pass: maxima of |x| and |dOut| components over the pair's rows -> per-unit scales (identical in both CTAs)
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
      if (g == 0) { invA[u] = ia; invB[t] = ib; }
      if (g == 1) {                                         // the PEER's units: their B scales unscale my columns
        const int tp = (int)(rank ^ 1u) * C::HU + u;
        const float px = net[off_W1(IN) + tp * IN], py = net[off_W1(IN) + tp * IN + 1];
        const float pz = IN == 3 ? net[off_W1(IN) + tp * IN + 2] : 0.f;
        const float pb = fmaf(fabsf(px), __int_as_float(rmax[0]), fmaf(fabsf(py), __int_as_float(rmax[1]),
                         fmaf(fabsf(pz), __int_as_float(rmax[2]), fabsf(net[off_b1(IN) + tp]))));
        float ps, pi;
        pow2_scale(pb, ps, pi);
        invB[tp] = pi;
      }
    }
    // Row PAIRS are processed with packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2: the FMA pipe issues one warp
    // instruction per two clocks either way), the layer-1 ReLU is folded into the fp16 conversion, the x / dOut rows of
    // FOUR stages are staged in shared memory at once (structure of arrays, so that a row pair is one 8-byte load; one
    // block barrier per 128 rows instead of one per 32) and the H2 values are fetched two stages ahead -- the
    // operand generators, not the tensor pipe, bound this kernel (ncu r02: tensor pipe 25 %, top stalls = the per-stage
    // barrier and the H2 loads).
    float2 s_db2 = make_float2(0.f, 0.f), s_dw3[OUT];
    float s_db3[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) { s_dw3[o] = make_float2(0.f, 0.f); s_db3[o] = 0.f; }
    const uint32_t a_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + g * 4;    // 8 rows = 4 columns
    float* sxx = reinterpret_cast<float*>(xs);                // [2][128] x.x | [2][128] x.y | [2][128] x.z  (OFF_X region: 3 KB of 2 KB + OFF_DO 1 KB)
    float* sxy = sxx + 2 * C::SS_ROWS;
    float* sxz = sxy + 2 * C::SS_ROWS;
    float* sd0 = reinterpret_cast<float*>(sm + C::OFF_SS);    // [2][128] dOut[.][0] | [2][128] dOut[.][1]
    float* sd1 = sd0 + 2 * C::SS_ROWS;
    auto h2_ptr = [&](int sg) {
      const int row0 = sg * C::RS + g * 8;
      return jb.h2 + (((size_t)net_i * tiles64 + (row0 >> 6)) * H + t) * 64 + (row0 & 63);
    };
    const float2 w1x2 = make_float2(w1x, w1x), w1y2 = make_float2(w1y, w1y), w1z2 = make_float2(w1z, w1z), b12 = make_float2(b1v, b1v);
    const float2 sA2 = make_float2(sA, sA), sB2 = make_float2(sB, sB);
    // x / dOut rows of a super-stage (4 stages = 128 rows): thread tid < 128 fetches one row, one super-stage ahead
    float4 xr = make_float4(0.f, 0.f, 0.f, 0.f);
    float dr[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) dr[o] = 0.f;
    const int r_end = min(jb.rows, st_hi * C::RS);
    auto fetch_rows = [&](int k) {
      if (tid < C::SS_ROWS) {
        const int r = (st_lo + 4 * k) * C::RS + tid;
        const bool ok = r < r_end;
        xr = ok ? __ldg(jb.X + r) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int o = 0; o < OUT; ++o) dr[o] = ok ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + o) : 0.f;
      }
    };
    const int n_st = st_hi - st_lo, n_ss = (n_st + 3) / 4;
    // H2 values of this thread's 8 rows, two stages ahead
    // (two register sets used alternately -- slot = stage parity inside the super-stage, static after unrolling -- so
    // that a set is refilled right after its values were copied out, never moved while a load is in flight)
    constexpr int AH = 2;                                   // (4 stages ahead measured: no gain, registers spill)
    float4 hs[AH][2];
#pragma unroll
    for (int i = 0; i < AH; ++i) hs[i][0] = hs[i][1] = make_float4(0.f, 0.f, 0.f, 0.f);
    auto fetch_h2 = [&](int sg, float4& a, float4& b) {
      const float* h2p = h2_ptr(sg);
      a = __ldg(reinterpret_cast<const float4*>(h2p));
      b = __ldg(reinterpret_cast<const float4*>(h2p) + 1);
    };
    if (n_st > 0) fetch_rows(0);
#pragma unroll
    for (int i = 0; i < AH; ++i)
      if (n_st > i) fetch_h2(st_lo + i, hs[i][0], hs[i][1]);
    uint32_t it = 0;
    for (int k = 0; k < n_ss; ++k) {
      const int buf = (k & 1) * C::SS_ROWS;
      if (tid < C::SS_ROWS) {
        sxx[buf + tid] = xr.x; sxy[buf + tid] = xr.y; sxz[buf + tid] = xr.z;
        sd0[buf + tid] = dr[0];
        if (OUT == 2) sd1[buf + tid] = dr[OUT - 1];
      }
      if (k + 1 < n_ss) fetch_rows(k + 1);
      asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));      // (the buffer was last read two super-stages ago)
#pragma unroll
      for (int q = 0; q < 4; ++q, ++it) {
        const int sg = st_lo + 4 * k + q;
        if (sg >= st_hi) break;
        const uint32_t s = it % C::STAGES;
        float4& h0 = hs[q % AH][0];
        float4& h1r = hs[q % AH][1];
        const float hv[8] = {h0.x, h0.y, h0.z, h0.w, h1r.x, h1r.y, h1r.z, h1r.w};
        if (sg + AH < st_hi) fetch_h2(sg + AH, h0, h1r);
        uint32_t ahi[4], alo[4], bhi[4], blo[4];
        const int rl0 = buf + q * C::RS + g * 8;
#pragma unroll
        for (int e = 0; e < 4; ++e) {                               // rows rl0 + 2e, rl0 + 2e + 1
          const float2 d0 = *reinterpret_cast<const float2*>(sd0 + rl0 + 2 * e);
          const float2 hp = make_float2(hv[2 * e], hv[2 * e + 1]);
          float2 gs = fmul2(d0, make_float2(w3[0], w3[0]));
          s_dw3[0] = ffma2(d0, hp, s_dw3[0]);
          if (t == 0) s_db3[0] += d0.x + d0.y;
          if (OUT == 2) {
            const float2 d1 = *reinterpret_cast<const float2*>(sd1 + rl0 + 2 * e);
            gs = ffma2(d1, make_float2(w3[OUT - 1], w3[OUT - 1]), gs);
            s_dw3[OUT - 1] = ffma2(d1, hp, s_dw3[OUT - 1]);
            if (t == 0) s_db3[OUT - 1] += d1.x + d1.y;
          }
          const float2 dz = make_float2(hp.x > 0.f ? gs.x : 0.f, hp.y > 0.f ? gs.y : 0.f);
          s_db2.x += dz.x; s_db2.y += dz.y;
          const float2 xxp = *reinterpret_cast<const float2*>(sxx + rl0 + 2 * e);
          const float2 xyp = *reinterpret_cast<const float2*>(sxy + rl0 + 2 * e);
          float2 z = ffma2(xyp, w1y2, ffma2(xxp, w1x2, b12));       // the forward's order: chain starts from the bias
          if (IN == 3) z = ffma2(*reinterpret_cast<const float2*>(sxz + rl0 + 2 * e), w1z2, z);
          split_h2_trunc(fmul2(dz, sA2), ahi[e], alo[e]);
          split_h2_trunc_relu(fmul2(z, sB2), bhi[e], blo[e]);      // H1 = relu(z): folded into the conversions
        }
        mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);          // values are ready before the stage is: wait late
        tc_fence_after();
        tmem_st4(a_lane + s * C::A_STAGE_COLS, ahi);
        tmem_st4(a_lane + s * C::A_STAGE_COLS + C::A_LO_COLS, alo);
        uint8_t* Bst = sm + s * C::B_STAGE_BYTES + chunk_off(C::HU, u, g);
        *reinterpret_cast<uint4*>(Bst) = make_uint4(bhi[0], bhi[1], bhi[2], bhi[3]);
        *reinterpret_cast<uint4*>(Bst + C::B_TERM_BYTES) = make_uint4(blo[0], blo[1], blo[2], blo[3]);
        tmem_st_wait();
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&full[s], 0);
      }
    }
    const float s_db2s = s_db2.x + s_db2.y;
    float s_dw3s[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) s_dw3s[o] = s_dw3[o].x + s_dw3[o].y;
    // small gradients of unit t: the four row groups are added in a fixed order (group 0 + 1 + 2 + 3)
    if (g > 0) small_g[(g - 1) * C::HU + u] = make_float4(s_db2s, s_dw3s[0], OUT == 2 ? s_dw3s[OUT - 1] : 0.f, s_db3[0]);
    if (OUT == 2 && t == 0 && g > 0) rmax[4 + g] = __float_as_int(s_db3[OUT - 1]);       // (plain bit copies; slots 5..7)
    asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
    if (g == 0) {
      float db3_1 = s_db3[OUT - 1];
      float a0 = s_db2s, a1 = s_dw3s[0], a2 = OUT == 2 ? s_dw3s[OUT - 1] : 0.f, a3 = s_db3[0];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const float4 o2 = small_g[q * C::HU + u];
        a0 += o2.x; a1 += o2.y; a2 += o2.z; a3 += o2.w;
        if (OUT == 2 && t == 0) db3_1 += __int_as_float(rmax[5 + q]);
      }
      float* sm2 = jb.small2 + ((size_t)net_i * jb.splits + split) * SMALL_STRIDE;
      sm2[H * IN + H + t] = a0;
      sm2[H * IN + 2 * H + t] = a1;
      if (OUT == 2) sm2[H * IN + 2 * H + H + t] = a2;
      if (t == 0) {
        sm2[H * IN + 2 * H + OUT * H] = a3;
        if (OUT == 2) sm2[H * IN + 2 * H + OUT * H + 1] = db3_1;
      }
    }
    // the leader's last multicast commits land in THIS CTA's barriers: do not exit before they have
    if (st_hi > st_lo) {
      mbar_wait(done, 0);
      tc_fence_after();
    }
    // ---------------- epilogue: unscale and dump this CTA's 128 x 256 half of the accumulator as the split's partial ----------------
    // warp w reads TMEM lane quarter w % 4 and every fourth 32-column chunk
    float* out = jb.pw2 + ((size_t)net_i * jb.splits + split) * H * H;
    {
      const int qw = warp & 3, part = warp >> 2;
      const int jl = qw * 32 + lane;
      const float ia = invA[jl];
      float* orow = out + (size_t)((int)rank * C::HU + jl) * H;
#pragma unroll 1
      for (int c0 = part * 32; c0 < H; c0 += 32 * (C::PROD_WARPS / 4)) {
        float v[32];
        if (st_hi > st_lo) {
          tmem_ld32(tmem + ((uint32_t)(qw * 32) << 16) + c0, v);
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
  cluster_sync_all();
  if (warp == C::MMA_WARP) tmem_dealloc2(tmem, 512);
}

}  // namespace tc
}  // namespace cql
