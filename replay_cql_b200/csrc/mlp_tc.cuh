// mlp_tc.cuh -- tensor-core (tcgen05 / TMEM) forward of the 3-layer MLPs.
//
// One persistent, warp-specialised CTA per SM:
//   warps 0-3   epilogue : TMEM -> registers (thread = row), +b2, ReLU, layer-3 dot, optional H2 store
//   warps 4-11  producers: layer 1 on CUDA cores, written straight into the UMMA operand layout
//                          (bf16, or tf32 hi/lo for the 3-term split) -- H1 never touches HBM
//   warp 12     MMA      : bulk-copies the resident W2 slice, issues tcgen05.mma, commits to mbarriers
// W2 stays RESIDENT in shared memory (128 KB): bf16 -> all 256 output columns; tf32x3 -> a 64-column
// slice (hi + lo), so four CTAs share a row tile and the layer-3 partial sums are added afterwards.
// A-operand K-chunks flow through a small smem ring; two TMEM accumulators overlap MMA and epilogue.
#pragma once
#include "tc_common.cuh"
#include "engine.cuh"

namespace cql {
namespace tc {

constexpr int TM = 128;                  // rows per tile (UMMA M)

template <bool TF32>
struct Cfg {
  static constexpr int ES = TF32 ? 4 : 2;            // operand element bytes
  static constexpr int EPC = 16 / ES;                // elements per 16-byte chunk
  static constexpr int UK = 32 / ES;                 // K per tcgen05.mma
  static constexpr int TERMS = TF32 ? 2 : 1;         // operand copies (hi, lo)
  static constexpr int NS = TF32 ? 64 : 256;         // output columns per CTA
  static constexpr int SLICES = H / NS;
  static constexpr uint32_t B_TERM_BYTES = NS * H * ES;
  static constexpr uint32_t B_BYTES = TERMS * B_TERM_BYTES;         // 128 KB
  static constexpr uint32_t TMEM_COLS = 2 * NS < 32 ? 32 : 2 * NS;
  static constexpr size_t PACKED_NET_BYTES = (size_t)SLICES * B_BYTES;
};

// pipeline shape: NPW producer warps (CUDA-core operand generation is issue-bound, so the forward runs 16)
template <bool TF32, int NPW>
struct Pipe : Cfg<TF32> {
  using C = Cfg<TF32>;
  static constexpr int KC = TF32 ? 16 : 64;                    // K elements per ring stage
  static constexpr int STAGES = TF32 ? 5 : 4;
  static constexpr int PIECES = KC / C::EPC;                   // 16-byte K pieces per row per stage (one warp each)
  static constexpr int GROUPS = NPW / PIECES;                  // warp group g fills stages with it % GROUPS == g
  static constexpr int NCHUNK = H / KC;                        // stages per tile
  static constexpr uint32_t A_TERM_BYTES = TM * KC * C::ES;
  static constexpr uint32_t A_STAGE_BYTES = C::TERMS * A_TERM_BYTES;
  static constexpr int MMA_WARP = 4 + NPW;
  static constexpr int THREADS = (5 + NPW) * 32;
  static constexpr int PROD_THREADS = NPW * 32;
};
constexpr int FWD_NPW = 16;
constexpr int BWD1_NPW = 8;

// packed weights: per net, per slice: [term][kchunk16][n_local/8][8][16 B]  (chunk_off with rows = NS)
// TRANSPOSE=false: B[n][k] = W2[n][k] (forward);  true: B[n][k] = W2[k][n] (backward dH1 = dZ2 * W2)
template <bool TF32, bool TRANSPOSE>
__global__ void k_pack_w2(const float* __restrict__ params, int in_dim, int n_nets, uint8_t* __restrict__ packed) {
  using C = Cfg<TF32>;
  const int net = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;        // 16-byte chunk id: n * (H/EPC) + kc
  if (net >= n_nets || c >= H * (H / C::EPC)) return;
  const int n = c / (H / C::EPC), kc = c % (H / C::EPC);
  const float* W2 = params + (size_t)net * NET_STRIDE + off_W2(in_dim);
  float v[C::EPC];
#pragma unroll
  for (int i = 0; i < C::EPC; ++i) {
    const int k = kc * C::EPC + i;
    v[i] = TRANSPOSE ? W2[(size_t)k * H + n] : W2[(size_t)n * H + k];
  }
  const int slice = n / C::NS, nl = n % C::NS;
  uint8_t* base = packed + (size_t)net * C::PACKED_NET_BYTES + (size_t)slice * C::B_BYTES + chunk_off(C::NS, nl, kc);
  if (TF32) {
    float4 h, l;
    split_tf32(v[0], h.x, l.x); split_tf32(v[1], h.y, l.y); split_tf32(v[2], h.z, l.z); split_tf32(v[3], h.w, l.w);
    *reinterpret_cast<float4*>(base) = h;
    *reinterpret_cast<float4*>(base + C::B_TERM_BYTES) = l;
  } else {
    __nv_bfloat162 p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(base) = *reinterpret_cast<uint4*>(p);
  }
}

// several networks / orientations in ONE launch (after an Adam step: critics fwd + critics^T + targets fwd)
struct PackJobs {
  struct J { const float* net; uint8_t* dst; int in_dim, transpose; } j[3 * CQL_MAX_CRITICS];   // C critics (2 orientations) + C targets
  int n;
};
template <bool TF32>
__global__ void k_pack_multi(const PackJobs jobs) {
  using C = Cfg<TF32>;
  const PackJobs::J jb = jobs.j[blockIdx.y];
  const int c = blockIdx.x * blockDim.x + threadIdx.x;        // 16-byte chunk id: n * (H/EPC) + kc
  if (c >= H * (H / C::EPC)) return;
  const int n = c / (H / C::EPC), kc = c % (H / C::EPC);
  const float* W2 = jb.net + off_W2(jb.in_dim);
  float v[C::EPC];
#pragma unroll
  for (int i = 0; i < C::EPC; ++i) {
    const int k = kc * C::EPC + i;
    v[i] = jb.transpose ? W2[(size_t)k * H + n] : W2[(size_t)n * H + k];
  }
  const int slice = n / C::NS, nl = n % C::NS;
  uint8_t* base = jb.dst + (size_t)slice * C::B_BYTES + chunk_off(C::NS, nl, kc);
  if constexpr (TF32) {
    float4 h, l;
    split_tf32(v[0], h.x, l.x); split_tf32(v[1], h.y, l.y); split_tf32(v[2], h.z, l.z); split_tf32(v[3], h.w, l.w);
    *reinterpret_cast<float4*>(base) = h;
    *reinterpret_cast<float4*>(base + C::B_TERM_BYTES) = l;
  } else {
    __nv_bfloat162 p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(base) = *reinterpret_cast<uint4*>(p);
  }
}

struct TcFwdJob {
  const float4* X;        // [rows]
  const float* params;    // fp32 slot of the first net (W1, b1, b2, W3, b3 are read from here)
  const uint8_t* packed;  // packed W2 of the first net
  float* out_part;        // [n_nets][SLICES][rows][OUT] partial layer-3 sums (b3 NOT added)
  float* h2;              // post-ReLU hidden for the backward kernels, or nullptr.  Layout = the CUDA-core
                          // kernels' tile-blocked transposed form [n_nets][ceil(rows/64)][256][64] (mlp_simt.cuh)
  int rows, n_nets;
};
struct TcFwdJobs {
  TcFwdJob j[3];
  int n;
  int item_begin[4];      // prefix sums of items per job; item = (net, slice, tile)
  int h2_cost = 0;        // f16x3 kernel: relative cost of an item that stores H2 (plain item = 10); 0 = default
};

struct ItemInfo { int job, net, slice, tile, pair_id; };

template <bool TF32>
__device__ __forceinline__ ItemInfo decode_item(const TcFwdJobs& jobs, int item) {
  using C = Cfg<TF32>;
  ItemInfo it;
  it.job = 0;
  while (it.job + 1 < jobs.n && item >= jobs.item_begin[it.job + 1]) ++it.job;
  const int local = item - jobs.item_begin[it.job];
  const int tiles = (jobs.j[it.job].rows + TM - 1) / TM;
  const int pair = local / tiles;
  it.tile = local % tiles;
  it.net = pair / C::SLICES;
  it.slice = pair % C::SLICES;
  it.pair_id = it.job * 64 + pair;
  return it;
}

template <bool TF32, int NPW>
struct FwdSmem {
  using C = Pipe<TF32, NPW>;
  static constexpr uint32_t OFF_B = 0;
  static constexpr uint32_t OFF_A = C::B_BYTES;
  static constexpr uint32_t OFF_W1 = OFF_A + C::STAGES * C::A_STAGE_BYTES;   // float4[256]: w0,w1,w2,b1
  static constexpr uint32_t OFF_EB = OFF_W1 + H * 16;                        // float4[NS]: b2,w3_0,w3_1,-
  static constexpr uint32_t OFF_BAR = OFF_EB + C::NS * 16;
  static constexpr uint32_t N_BARS = 2 * C::STAGES + 4 + 2;                  // full/empty, tmem full/empty x2, bload, drain
  static constexpr uint32_t OFF_SLOT = OFF_BAR + N_BARS * 8;
  static constexpr uint32_t BYTES = OFF_SLOT + 16;
};

// packed fp32x2 FMA (sm_100a): d = a * b + c on two lanes of a 64-bit register pair
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
// cheap split for the producers: hi rounded to nearest tf32, lo = exact remainder (the MMA truncates it to tf32:
// <= 2^-23 |x|, negligible next to the accumulation error)
__device__ __forceinline__ void split_tf32_fast(float x, float& hi, float& lo) {
  hi = rn_tf32(x);
  lo = x - hi;
}

template <bool TF32, int IN, int OUT>
__global__ void __launch_bounds__(Pipe<TF32, FWD_NPW>::THREADS, 1) tc_fwd_kernel(const TcFwdJobs jobs) {
  using C = Pipe<TF32, FWD_NPW>;
  using S = FwdSmem<TF32, FWD_NPW>;
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + S::OFF_B;
  uint8_t* As = sm + S::OFF_A;
  float4* w1s = reinterpret_cast<float4*>(sm + S::OFF_W1);
  float4* ebs = reinterpret_cast<float4*>(sm + S::OFF_EB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + S::OFF_BAR);
  uint64_t* full = bars;                       // [STAGES] producers -> MMA
  uint64_t* empty = bars + C::STAGES;          // [STAGES] MMA -> producers
  uint64_t* tfull = bars + 2 * C::STAGES;      // [2] MMA -> epilogue
  uint64_t* tempty = tfull + 2;                // [2] epilogue -> MMA
  uint64_t* bload = tempty + 2;                // W2 slice landed
  uint64_t* drain = bload + 1;                 // all issued MMAs retired
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + S::OFF_SLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int total = jobs.item_begin[jobs.n];
  const int item_lo = (int)((long long)total * blockIdx.x / gridDim.x);
  const int item_hi = (int)((long long)total * (blockIdx.x + 1) / gridDim.x);

  if (warp == C::MMA_WARP) {
    tmem_alloc(slot, C::TMEM_COLS);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], C::PIECES); mbar_init(&empty[s], 1); }
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

  if (warp == C::MMA_WARP) {
    // =============================== MMA issuer (whole warp, one elected lane issues) ===============================
    {
      const uint32_t idesc = instr_desc(TF32 ? FMT_TF32 : FMT_BF16, TM, C::NS);
      const uint32_t a_lbo = TM * 16, b_lbo = C::NS * 16;
      const uint32_t b_base = smem_u32(Bs);
      int cur_pair = -1;
      uint32_t it = 0, nb = 0, nd = 0, tcount = 0;
      for (int item = item_lo; item < item_hi; ++item) {
        const ItemInfo ii = decode_item<TF32>(jobs, item);
        if (ii.pair_id != cur_pair) {
          if (cur_pair >= 0) {              // old W2 slice must not be overwritten while MMAs still read it
            if (elect_one()) umma_commit(drain);
            __syncwarp();
            mbar_wait(drain, nd & 1);
            ++nd;
          }
          const TcFwdJob& jb = jobs.j[ii.job];
          const uint8_t* src = jb.packed + (size_t)ii.net * C::PACKED_NET_BYTES + (size_t)ii.slice * C::B_BYTES;
          if (elect_one()) {
            mbar_arrive_expect_tx(bload, C::B_BYTES);
            for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bload);
          }
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
          const uint32_t a_base = smem_u32(As + s * C::A_STAGE_BYTES);
          if (elect_one()) {
#pragma unroll
          for (int j = 0; j < C::KC / C::UK; ++j) {
            const uint32_t g = c * (C::KC / C::UK) + j;
            const uint64_t a_hi = smem_desc(a_base + 2 * j * a_lbo, a_lbo, 128);
            const uint64_t b_hi = smem_desc(b_base + 2 * g * b_lbo, b_lbo, 128);
            const uint32_t first = (c == 0 && j == 0) ? 0u : 1u;
            if constexpr (TF32) {
              const uint64_t a_lo = smem_desc(a_base + C::A_TERM_BYTES + 2 * j * a_lbo, a_lbo, 128);
              const uint64_t b_lo = smem_desc(b_base + C::B_TERM_BYTES + 2 * g * b_lbo, b_lbo, 128);
              umma<TF32>(d_tmem, a_lo, b_hi, idesc, first);
              umma<TF32>(d_tmem, a_hi, b_lo, idesc, 1u);
              umma<TF32>(d_tmem, a_hi, b_hi, idesc, 1u);
            } else {
              umma<TF32>(d_tmem, a_hi, b_hi, idesc, first);
            }
          }
          umma_commit(&empty[s]);           // stage reusable once these MMAs have read it
          if (c == C::NCHUNK - 1) umma_commit(&tfull[acc]);   // accumulator complete
          }
          __syncwarp();
        }
        ++tcount;
      }
    }
  } else if (warp >= 4) {
    // =============================== producers: layer 1 -> operand ring ===============================
    const int pw = warp - 4, ptid = tid - 128;
    int cur_pair = -1, cur_netkey = -1;
    uint32_t it = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const ItemInfo ii = decode_item<TF32>(jobs, item);
      const TcFwdJob& jb = jobs.j[ii.job];
      const int netkey = ii.job * 64 + ii.net;
      if (ii.pair_id != cur_pair) {
        cur_pair = ii.pair_id;
        if (netkey != cur_netkey) {         // (re)load W1|b1 of this net
          cur_netkey = netkey;
          asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
          const float* net = jb.params + (size_t)ii.net * NET_STRIDE;
          for (int k = ptid; k < H; k += C::PROD_THREADS)
            w1s[k] = make_float4(net[off_W1(IN) + k * IN], net[off_W1(IN) + k * IN + 1],
                                 IN == 3 ? net[off_W1(IN) + k * IN + 2] : 0.f, net[off_b1(IN) + k]);
          asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        }
      }
      float4 x[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = ii.tile * TM + lane + 32 * i;
        x[i] = r < jb.rows ? __ldg(jb.X + r) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        if ((int)(it % C::GROUPS) != pw / C::PIECES) continue;     // the other warp group fills this stage
        const uint32_t s = it % C::STAGES;
        mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
        uint8_t* stage = As + s * C::A_STAGE_BYTES;
        // this warp owns one 16-byte K-piece of the chunk, for all 128 rows (4 per lane)
        const int p = pw % C::PIECES;
        {
          float z[4][C::EPC];
#pragma unroll
          for (int e = 0; e < C::EPC; ++e) {
            const float4 w = w1s[c * C::KC + p * C::EPC + e];
            const float2 bw = make_float2(w.w, w.w), wx = make_float2(w.x, w.x), wy = make_float2(w.y, w.y),
                         wz = make_float2(w.z, w.z);
#pragma unroll
            for (int i = 0; i < 4; i += 2) {     // two rows per packed FMA; chain starts from the bias
              float2 v = ffma2(make_float2(x[i].x, x[i + 1].x), wx, bw);
              v = ffma2(make_float2(x[i].y, x[i + 1].y), wy, v);
              if (IN == 3) v = ffma2(make_float2(x[i].z, x[i + 1].z), wz, v);
              z[i][e] = fmaxf(v.x, 0.f);
              z[i + 1][e] = fmaxf(v.y, 0.f);
            }
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t off = chunk_off(TM, lane + 32 * i, p);
            if constexpr (TF32) {
              float4 hi, lo;
              split_tf32_fast(z[i][0], hi.x, lo.x); split_tf32_fast(z[i][1], hi.y, lo.y);
              split_tf32_fast(z[i][2], hi.z, lo.z); split_tf32_fast(z[i][3], hi.w, lo.w);
              *reinterpret_cast<float4*>(stage + off) = hi;
              *reinterpret_cast<float4*>(stage + C::A_TERM_BYTES + off) = lo;
            } else {
              __nv_bfloat162 q[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) q[e] = __floats2bfloat162_rn(z[i][2 * e], z[i][2 * e + 1]);
              *reinterpret_cast<uint4*>(stage + off) = *reinterpret_cast<uint4*>(q);
            }
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
  } else {
    // =============================== epilogue: TMEM -> layer 3 (+ H2) ===============================
    int cur_pair = -1;
    uint32_t tcount = 0;
    const int row_in_tile = warp * 32 + lane;
    for (int item = item_lo; item < item_hi; ++item) {
      const ItemInfo ii = decode_item<TF32>(jobs, item);
      const TcFwdJob& jb = jobs.j[ii.job];
      if (ii.pair_id != cur_pair) {
        cur_pair = ii.pair_id;
        asm volatile("bar.sync 2, 128;");
        const float* net = jb.params + (size_t)ii.net * NET_STRIDE;
        for (int cidx = tid; cidx < C::NS; cidx += 128) {
          const int col = ii.slice * C::NS + cidx;
          ebs[cidx] = make_float4(net[off_b2(IN) + col], net[off_W3(IN) + col],
                                  OUT == 2 ? net[off_W3(IN) + H + col] : 0.f, 0.f);
        }
        asm volatile("bar.sync 2, 128;");
      }
      const uint32_t acc = tcount & 1;
      mbar_wait(&tfull[acc], (tcount >> 1) & 1);
      tc_fence_after();
      const int row = ii.tile * TM + row_in_tile;
      const bool store_h2 = jb.h2 != nullptr;     // padded rows are stored too (finite; masked by dOut = 0)
      const int tiles64 = (jb.rows + 63) / 64;
      float* h2row = store_h2 ? jb.h2 + (((size_t)ii.net * tiles64 + (row >> 6)) * H + ii.slice * C::NS) * 64 + (row & 63)
                              : nullptr;
      float q0 = 0.f, q1 = 0.f;
#pragma unroll 1
      for (int c0 = 0; c0 < C::NS; c0 += 32) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + acc * C::NS + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float4 e = ebs[c0 + i];
          const float hv = fmaxf(v[i] + e.x, 0.f);
          v[i] = hv;
          q0 = fmaf(hv, e.y, q0);
          if (OUT == 2) q1 = fmaf(hv, e.z, q1);
        }
        if (store_h2 && (row >> 6) < tiles64) {
#pragma unroll
          for (int i = 0; i < 32; ++i) h2row[(size_t)(c0 + i) * 64] = v[i];   // lanes = consecutive rows: coalesced
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
      ++tcount;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::MMA_WARP) tmem_dealloc(tmem, C::TMEM_COLS);
}

// out[net][row][o] = b3[o] + sum over slices of the partial layer-3 sums (fixed order)
template <int IN, int OUT>
__global__ void k_sum_partials(const float* __restrict__ part, const float* __restrict__ params, int rows, int n_nets,
                               int slices, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_nets * rows * OUT) return;
  const int o = i % OUT, r = (i / OUT) % rows, net = i / (OUT * rows);
  float s = 0.f;
  for (int sl = 0; sl < slices; ++sl) s += part[(((size_t)net * slices + sl) * rows + r) * OUT + o];
  out[i] = s + params[(size_t)net * NET_STRIDE + off_b3(IN, OUT) + o];
}

struct SumJobs {
  struct J { const float* part; const float* params; float* out; int rows, n_nets; } j[4];
  int n;
};
template <int IN, int OUT>
__global__ void k_sum_partials_multi(const SumJobs jobs, int slices) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
 
  const SumJobs::J jb = jobs.j[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= jb.n_nets * jb.rows * OUT) return;
  const int o = i % OUT, r = (i / OUT) % jb.rows, net = i / (OUT * jb.rows);
  float s = 0.f;
  for (int sl = 0; sl < slices; ++sl) s += jb.part[(((size_t)net * slices + sl) * jb.rows + r) * OUT + o];
  jb.out[i] = s + jb.params[(size_t)net * NET_STRIDE + off_b3(IN, OUT) + o];
}

}  // namespace tc
}  // namespace cql
