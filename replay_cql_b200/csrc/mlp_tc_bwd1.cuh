// mlp_tc_bwd1.cuh -- tensor-core input gradient of the hidden layer:  dH1 = dZ2 W2, then
// dZ1 = dH1 * relu'(Z1), dW1, db1 and (optionally) dx.  Same warp-specialised pipeline as the forward
// (mlp_tc.cuh): W2^T resident in shared memory, the A operand (dZ2) generated per K-chunk by the
// producer warps from (dOut, W3, H2 > 0), two TMEM accumulators.  In the epilogue a thread owns one row:
// dx is a thread-local dot product; dW1/db1 need a sum over rows, done with a 31-shuffle butterfly
// reduce-scatter per 32-column chunk and then kept in registers across all tiles of the CTA.
#pragma once
#include "mlp_tc.cuh"
#include "mlp_tc_ts.cuh"

namespace cql {
namespace tc {

struct Bwd1Job {
  const float4* X;        // [rows]
  const float* dOut;      // [n_nets][rows][OUT]
  const float* h2;        // [n_nets][tiles64][256][64]
  const float* params;    // first net slot (fp32)
  const uint8_t* packedT; // packed W2^T of the first net (B[n=k][kk=j] = W2[j][k])
  float* small1;          // [n_nets][slots][SMALL_STRIDE]: only W1 | b1 entries written; slots = 4*gridDim.x, zeroed by caller
                          // (or by the kernel itself: zero_small1)
  float4* dX_part;        // [n_nets][SLICES][rows] or nullptr
  int rows, n_nets, slots;
  // dx-only launch of the actor step (f16x3): dOut = d(actor loss)/dQ through the min over the critics, taken by the
  // producers themselves from the forward's layer-3 partial sums -- the former one-CTA k_actor_dq launch (4 us on the
  // critical path).  q_parts > 0 switches it on (OUT == 1); the sums are added in q_at()'s order.
  const float* q_part = nullptr;   // [n_nets][q_parts][rows]
  int q_parts = 0;
  float dq_scale = 0.f;            // -1 / B
  // f16x3 kernels: every CTA zeroes its own slots (W1 | b1 of every network) before its first flush, so that no memset
  // node sits between this launch and its predecessor in the step graph (which would cost the programmatic edge)
  int zero_small1 = 0;
};
// (zero_small1) slots [blockIdx.x * per_cta, + per_cta) of every network, W1 | b1 entries; ends with a CTA barrier
template <int IN>
__device__ __forceinline__ void zero_small1_slots(const Bwd1Job& jb, int per_cta) {
  if (!jb.zero_small1) return;
  constexpr int NF4 = off_W2(IN) / 4;
  for (int net = 0; net < jb.n_nets; ++net)
    for (int s = 0; s < per_cta; ++s) {
      float4* o = reinterpret_cast<float4*>(jb.small1 + ((size_t)net * jb.slots + (size_t)blockIdx.x * per_cta + s) * SMALL_STRIDE);
      for (int f = threadIdx.x; f < NF4; f += blockDim.x) o[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  __syncthreads();
}
// d(actor loss)/dQ of row r for network net_i: dq_scale on the critic with the smallest Q (first one on ties), else 0
template <int IN, int OUT>
__device__ __forceinline__ float actor_dq_of(const Bwd1Job& jb, int net_i, int r) {
  // (a critic's parts and bias are requested before the first addition: one L2 round trip per critic, not per part)
  constexpr int MAXP = 8;
  int arg = 0;
  float qm = 0.f;
  for (int c = 0; c < jb.n_nets; ++c) {
    float part[MAXP];
#pragma unroll
    for (int p = 0; p < MAXP; ++p)
      if (p < jb.q_parts) part[p] = __ldg(jb.q_part + ((size_t)c * jb.q_parts + p) * jb.rows + r);
    const float bias = __ldg(jb.params + (size_t)c * NET_STRIDE + off_b3(IN, OUT));
    float v = 0.f;
#pragma unroll
    for (int p = 0; p < MAXP; ++p)
      if (p < jb.q_parts) v += part[p];
    const float q = v + bias;
    if (c == 0 || q < qm) { qm = q; arg = c; }
  }
  return net_i == arg ? jb.dq_scale : 0.f;
}

// after the call lane l holds sum over the warp's 32 lanes of v[l]
__device__ __forceinline__ float warp_reduce_scatter32(float (&v)[32]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = upper ? v[i] : v[i + off];
      const float keep = upper ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

template <bool TF32, int IN, int OUT, bool WGRADS, bool DX>
__global__ void __launch_bounds__(Pipe<TF32, BWD1_NPW>::THREADS, 1) tc_bwd1_kernel(const Bwd1Job jb) {
  using C = Pipe<TF32, BWD1_NPW>;
  using S = FwdSmem<TF32, BWD1_NPW>;
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + S::OFF_B;
  uint8_t* As = sm + S::OFF_A;
  float2* w3s = reinterpret_cast<float2*>(sm + S::OFF_W1);    // [256] (W3[0][j], W3[1][j])
  float4* ebs = reinterpret_cast<float4*>(sm + S::OFF_EB);    // [NS]  (W1[k][0..2], b1[k]) of the slice's columns
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + S::OFF_BAR);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* bload = tempty + 2;
  uint64_t* drain = bload + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + S::OFF_SLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles = (jb.rows + TM - 1) / TM;
  const int tiles64 = (jb.rows + 63) / 64;
  const int total = jb.n_nets * C::SLICES * tiles;             // item = (net, slice, tile), pair-major
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
    {
      const uint32_t idesc = instr_desc(TF32 ? FMT_TF32 : FMT_BF16, TM, C::NS);
      const uint32_t a_lbo = TM * 16, b_lbo = C::NS * 16;
      const uint32_t b_base = smem_u32(Bs);
      int cur_pair = -1;
      uint32_t it = 0, nb = 0, nd = 0, tcount = 0;
      for (int item = item_lo; item < item_hi; ++item) {
        const int pair = item / tiles;
        if (pair != cur_pair) {
          if (cur_pair >= 0) { if (elect_one()) umma_commit(drain); __syncwarp(); mbar_wait(drain, nd & 1); ++nd; }
          const uint8_t* src = jb.packedT + (size_t)(pair / C::SLICES) * C::PACKED_NET_BYTES + (size_t)(pair % C::SLICES) * C::B_BYTES;
          if (elect_one()) {
            mbar_arrive_expect_tx(bload, C::B_BYTES);
            for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bload);
          }
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
          umma_commit(&empty[s]);
          if (c == C::NCHUNK - 1) umma_commit(&tfull[acc]);
          }
          __syncwarp();
        }
        ++tcount;
      }
    }
  } else if (warp >= 4) {
    // ---------------- producers: dZ2 tile -> operand ring ----------------
    const int pw = warp - 4, ptid = tid - 128;
    int cur_net = -1;
    uint32_t it = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles, tile = item % tiles, net_i = pair / C::SLICES;
      if (net_i != cur_net) {
        cur_net = net_i;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        w3s[ptid] = make_float2(net[off_W3(IN) + ptid], OUT == 2 ? net[off_W3(IN) + H + ptid] : 0.f);
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      }
      float d0[4], d1[4];
      const float* h2r[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = tile * TM + lane + 32 * i;
        const bool ok = r < jb.rows;
        d0[i] = ok ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT) : 0.f;
        d1[i] = (ok && OUT == 2) ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + 1) : 0.f;
        const int rc = ok ? r : 0;     // clamp: the value is multiplied by dOut = 0 anyway
        h2r[i] = jb.h2 + ((size_t)net_i * tiles64 + (rc >> 6)) * H * 64 + (rc & 63);
      }
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        if ((int)(it % C::GROUPS) != pw / C::PIECES) continue;     // the other warp group fills this stage
        const uint32_t s = it % C::STAGES;
        mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
        uint8_t* stage = As + s * C::A_STAGE_BYTES;
        const int p = pw % C::PIECES;
        const int j0 = c * C::KC + p * C::EPC;
        float z[4][C::EPC];
#pragma unroll
        for (int e = 0; e < C::EPC; ++e) {
          const float2 w = w3s[j0 + e];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float hv = __ldg(h2r[i] + (size_t)(j0 + e) * 64);
            float g = d0[i] * w.x;
            if (OUT == 2) g = fmaf(d1[i], w.y, g);
            z[i][e] = hv > 0.f ? g : 0.f;
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t off = chunk_off(TM, lane + 32 * i, p);
          if constexpr (TF32) {
            float4 hi, lo;
            split_tf32(z[i][0], hi.x, lo.x); split_tf32(z[i][1], hi.y, lo.y);
            split_tf32(z[i][2], hi.z, lo.z); split_tf32(z[i][3], hi.w, lo.w);
            *reinterpret_cast<float4*>(stage + off) = hi;
            *reinterpret_cast<float4*>(stage + C::A_TERM_BYTES + off) = lo;
          } else {
            __nv_bfloat162 q[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) q[e] = __floats2bfloat162_rn(z[i][2 * e], z[i][2 * e + 1]);
            *reinterpret_cast<uint4*>(stage + off) = *reinterpret_cast<uint4*>(q);
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
  } else {
    // ---------------- epilogue: dZ1, dx, dW1/db1 ----------------
    constexpr int NCH = C::NS / 32;
    float a_b[NCH], a_w0[NCH], a_w1[NCH], a_w2[NCH];      // lane l <-> column chunk*32 + l of the current slice
#pragma unroll
    for (int q = 0; q < NCH; ++q) { a_b[q] = 0.f; a_w0[q] = 0.f; a_w1[q] = 0.f; a_w2[q] = 0.f; }
    auto flush = [&](int pair) {
      if (!WGRADS || pair < 0) return;
      const int net_i = pair / C::SLICES, slice = pair % C::SLICES;
      float* o = jb.small1 + ((size_t)net_i * jb.slots + blockIdx.x * 4 + warp) * SMALL_STRIDE;
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        const int k = slice * C::NS + q * 32 + lane;
        o[k * IN + 0] = a_w0[q];
        o[k * IN + 1] = a_w1[q];
        if (IN == 3) o[k * IN + 2] = a_w2[q];
        o[H * IN + k] = a_b[q];
        a_b[q] = 0.f; a_w0[q] = 0.f; a_w1[q] = 0.f; a_w2[q] = 0.f;
      }
    };
    int cur_pair = -1;
    uint32_t tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles, tile = item % tiles, net_i = pair / C::SLICES, slice = pair % C::SLICES;
      if (pair != cur_pair) {
        flush(cur_pair);
        cur_pair = pair;
        asm volatile("bar.sync 2, 128;");
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        for (int cidx = tid; cidx < C::NS; cidx += 128) {
          const int k = slice * C::NS + cidx;
          ebs[cidx] = make_float4(net[off_W1(IN) + k * IN], net[off_W1(IN) + k * IN + 1],
                                  IN == 3 ? net[off_W1(IN) + k * IN + 2] : 0.f, net[off_b1(IN) + k]);
        }
        asm volatile("bar.sync 2, 128;");
      }
      const uint32_t acc = tcount & 1;
      const int row = tile * TM + warp * 32 + lane;
      const float4 x = row < jb.rows ? __ldg(jb.X + row) : make_float4(0.f, 0.f, 0.f, 0.f);
      mbar_wait(&tfull[acc], (tcount >> 1) & 1);
      tc_fence_after();
      float dx0 = 0.f, dx1 = 0.f, dx2 = 0.f;
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + acc * C::NS + q * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float4 w = ebs[q * 32 + i];
          float z = fmaf(x.y, w.y, x.x * w.x);
          if (IN == 3) z = fmaf(x.z, w.z, z);
          z += w.w;
          const float d = z > 0.f ? v[i] : 0.f;
          v[i] = d;
          if (DX) {
            dx0 = fmaf(d, w.x, dx0);
            dx1 = fmaf(d, w.y, dx1);
            if (IN == 3) dx2 = fmaf(d, w.z, dx2);
          }
        }
        if (WGRADS) {
          float t[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) t[i] = v[i] * x.x;
          a_w0[q] += warp_reduce_scatter32(t);
#pragma unroll
          for (int i = 0; i < 32; ++i) t[i] = v[i] * x.y;
          a_w1[q] += warp_reduce_scatter32(t);
          if (IN == 3) {
#pragma unroll
            for (int i = 0; i < 32; ++i) t[i] = v[i] * x.z;
            a_w2[q] += warp_reduce_scatter32(t);
          }
          a_b[q] += warp_reduce_scatter32(v);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (DX && row < jb.rows)
        jb.dX_part[((size_t)net_i * C::SLICES + slice) * jb.rows + row] = make_float4(dx0, dx1, dx2, 0.f);
      ++tcount;
    }
    flush(cur_pair);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::MMA_WARP) tmem_dealloc(tmem, C::TMEM_COLS);
}

// ---- FP32-grade variant with the A operand (dZ2 tile) staged in tensor memory, see mlp_tc_ts.cuh ------------
template <int IN, int OUT, bool WGRADS, bool DX>
__global__ void __launch_bounds__(TsCfg::THREADS, 1) tc_bwd1_ts_kernel(const Bwd1Job jb) {
  using C = TsCfg;
  constexpr bool TF32 = true;
  extern __shared__ __align__(1024) uint8_t sm[];
  uint8_t* Bs = sm + C::OFF_B;
  float2* w3s = reinterpret_cast<float2*>(sm + C::OFF_W1);    // [256] (W3[0][j], W3[1][j])
  float4* ebs = reinterpret_cast<float4*>(sm + C::OFF_EB);    // [NS]  (W1[k][0..2], b1[k]) of the slice's columns
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

  if (warp == C::MMA_WARP) {
    const uint32_t idesc = instr_desc(FMT_TF32, TM, C::NS);
    const uint32_t b_lbo = C::NS * 16;
    const uint32_t b_base = smem_u32(Bs);
    int cur_pair = -1;
    uint32_t it = 0, nb = 0, nd = 0, tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles;
      if (pair != cur_pair) {
        if (cur_pair >= 0) { if (elect_one()) umma_commit(drain); __syncwarp(); mbar_wait(drain, nd & 1); ++nd; }
        const uint8_t* src = jb.packedT + (size_t)(pair / C::SLICES) * C::PACKED_NET_BYTES + (size_t)(pair % C::SLICES) * C::B_BYTES;
        if (elect_one()) {
          mbar_arrive_expect_tx(bload, C::B_BYTES);
          for (uint32_t o = 0; o < C::B_BYTES; o += 32768) bulk_g2s(Bs + o, src + o, 32768, bload);
        }
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
            const uint32_t a_hi = a_stage + j * C::UK, a_lo = a_hi + C::KC;
            umma_ts<true>(d_tmem, a_lo, b_hi, idesc, (c == 0 && j == 0) ? 0u : 1u);
            umma_ts<true>(d_tmem, a_hi, b_lo, idesc, 1u);
            umma_ts<true>(d_tmem, a_hi, b_hi, idesc, 1u);
          }
          umma_commit(&empty[s]);
          if (c == C::NCHUNK - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
      }
      ++tcount;
    }
  } else if (warp >= 4) {
    // ---------------- producers: dZ2 row -> TMEM ----------------
    const int pw = warp - 4, ptid = tid - 128;
    const int kq = pw >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + C::A_COL0 + kq * C::KPW;
    int cur_net = -1;
    uint32_t it = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles, tile = item % tiles, net_i = pair / C::SLICES;
      if (net_i != cur_net) {
        cur_net = net_i;
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        for (int j = ptid; j < H; j += C::PROD_THREADS)
          w3s[j] = make_float2(net[off_W3(IN) + j], OUT == 2 ? net[off_W3(IN) + H + j] : 0.f);
        asm volatile("bar.sync 1, %0;" ::"n"(C::PROD_THREADS));
      }
      const int r = tile * TM + (warp & 3) * 32 + lane;
      const bool ok = r < jb.rows;
      const float d0 = ok ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT) : 0.f;
      const float d1 = (ok && OUT == 2) ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + 1) : 0.f;
      const int rc = ok ? r : 0;
      const float* h2r = jb.h2 + ((size_t)net_i * tiles64 + (rc >> 6)) * H * 64 + (rc & 63);
      for (int c = 0; c < C::NCHUNK; ++c, ++it) {
        const uint32_t s = it % C::STAGES;
        const int j0 = c * C::KC + kq * C::KPW;
        float hv[C::KPW];
#pragma unroll
        for (int e = 0; e < C::KPW; ++e) hv[e] = __ldg(h2r + (size_t)(j0 + e) * 64);
        uint32_t hi[C::KPW], lo[C::KPW];
#pragma unroll
        for (int e = 0; e < C::KPW; ++e) {
          const float2 w = w3s[j0 + e];
          float g = d0 * w.x;
          if (OUT == 2) g = fmaf(d1, w.y, g);
          float h, l;
          split_tf32_fast(hv[e] > 0.f ? g : 0.f, h, l);
          hi[e] = __float_as_uint(h); lo[e] = __float_as_uint(l);
        }
        mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
        tc_fence_after();
#pragma unroll
        for (int q = 0; q < C::KPW; q += 8) {
          tmem_st8(lane_base + s * C::A_STAGE_COLS + q, *reinterpret_cast<const uint32_t(*)[8]>(&hi[q]));
          tmem_st8(lane_base + s * C::A_STAGE_COLS + C::KC + q, *reinterpret_cast<const uint32_t(*)[8]>(&lo[q]));
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
  } else {
    // ---------------- epilogue: dZ1, dx, dW1/db1 ----------------
    constexpr int NCH = C::NS / 32;
    float a_b[NCH], a_w0[NCH], a_w1[NCH], a_w2[NCH];      // lane l <-> column chunk*32 + l of the current slice
#pragma unroll
    for (int q = 0; q < NCH; ++q) { a_b[q] = 0.f; a_w0[q] = 0.f; a_w1[q] = 0.f; a_w2[q] = 0.f; }
    auto flush = [&](int pair) {
      if (!WGRADS || pair < 0) return;
      const int net_i = pair / C::SLICES, slice = pair % C::SLICES;
      float* o = jb.small1 + ((size_t)net_i * jb.slots + blockIdx.x * 4 + warp) * SMALL_STRIDE;
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        const int k = slice * C::NS + q * 32 + lane;
        o[k * IN + 0] = a_w0[q];
        o[k * IN + 1] = a_w1[q];
        if (IN == 3) o[k * IN + 2] = a_w2[q];
        o[H * IN + k] = a_b[q];
        a_b[q] = 0.f; a_w0[q] = 0.f; a_w1[q] = 0.f; a_w2[q] = 0.f;
      }
    };
    int cur_pair = -1;
    uint32_t tcount = 0;
    for (int item = item_lo; item < item_hi; ++item) {
      const int pair = item / tiles, tile = item % tiles, net_i = pair / C::SLICES, slice = pair % C::SLICES;
      if (pair != cur_pair) {
        flush(cur_pair);
        cur_pair = pair;
        asm volatile("bar.sync 2, 128;");
        const float* net = jb.params + (size_t)net_i * NET_STRIDE;
        for (int cidx = tid; cidx < C::NS; cidx += 128) {
          const int k = slice * C::NS + cidx;
          ebs[cidx] = make_float4(net[off_W1(IN) + k * IN], net[off_W1(IN) + k * IN + 1],
                                  IN == 3 ? net[off_W1(IN) + k * IN + 2] : 0.f, net[off_b1(IN) + k]);
        }
        asm volatile("bar.sync 2, 128;");
      }
      const uint32_t acc = tcount & 1;
      const int row = tile * TM + warp * 32 + lane;
      const float4 x = row < jb.rows ? __ldg(jb.X + row) : make_float4(0.f, 0.f, 0.f, 0.f);
      mbar_wait(&tfull[acc], (tcount >> 1) & 1);
      tc_fence_after();
      float dx0 = 0.f, dx1 = 0.f, dx2 = 0.f;
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + acc * C::NS + q * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float4 w = ebs[q * 32 + i];
          float z = fmaf(x.y, w.y, x.x * w.x);
          if (IN == 3) z = fmaf(x.z, w.z, z);
          z += w.w;
          const float d = z > 0.f ? v[i] : 0.f;
          v[i] = d;
          if (DX) {
            dx0 = fmaf(d, w.x, dx0);
            dx1 = fmaf(d, w.y, dx1);
            if (IN == 3) dx2 = fmaf(d, w.z, dx2);
          }
        }
        if (WGRADS) {
          float t[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) t[i] = v[i] * x.x;
          a_w0[q] += warp_reduce_scatter32(t);
#pragma unroll
          for (int i = 0; i < 32; ++i) t[i] = v[i] * x.y;
          a_w1[q] += warp_reduce_scatter32(t);
          if (IN == 3) {
#pragma unroll
            for (int i = 0; i < 32; ++i) t[i] = v[i] * x.z;
            a_w2[q] += warp_reduce_scatter32(t);
          }
          a_b[q] += warp_reduce_scatter32(v);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (DX && row < jb.rows)
        jb.dX_part[((size_t)net_i * C::SLICES + slice) * jb.rows + row] = make_float4(dx0, dx1, dx2, 0.f);
      ++tcount;
    }
    flush(cur_pair);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C::MMA_WARP) tmem_dealloc(tmem, C::TMEM_ALLOC);
}

// grads[net][idx] from the tensor-core partials: W2 <- pw2 (bwd2 splits); b2|W3|b3 <- small2 (bwd2 splits);
// W1|b1 <- small1 (bwd1 warp slots).  Fixed summation order.  One thread per 4 consecutive parameters,
// 16-byte loads, 4 partials in flight (the partials were just written: L2-resident, latency-bound).
__device__ __forceinline__ float4 sum_strided4(const float* __restrict__ p, int n, size_t stride) {
  float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
  int i = 0;
  for (; i + 4 <= n; i += 4) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p + (size_t)i * stride));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + (size_t)(i + 1) * stride));
    const float4 c = __ldg(reinterpret_cast<const float4*>(p + (size_t)(i + 2) * stride));
    const float4 d = __ldg(reinterpret_cast<const float4*>(p + (size_t)(i + 3) * stride));
    s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += a.w;
    s1.x += b.x; s1.y += b.y; s1.z += b.z; s1.w += b.w;
    s2.x += c.x; s2.y += c.y; s2.z += c.z; s2.w += c.w;
    s3.x += d.x; s3.y += d.y; s3.z += d.z; s3.w += d.w;
  }
  for (; i < n; ++i) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p + (size_t)i * stride));
    s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += a.w;
  }
  return make_float4((s0.x + s1.x) + (s2.x + s3.x), (s0.y + s1.y) + (s2.y + s3.y), (s0.z + s1.z) + (s2.z + s3.z),
                     (s0.w + s1.w) + (s2.w + s3.w));
}

// The same sums for one or two components of sum_strided4's float4 (per component they are the same additions in the same
// order, so the results are bit-identical), with every load of a chunk of at most NPRE partials issued before the first
// addition.  reduce8 = k_reduce_grads_tc's whole reduction of n partials: 8 chunks of ceil(n/8), combined in chunk order.
__device__ __forceinline__ void vacc(float& s, float a) { s += a; }
__device__ __forceinline__ void vacc(float2& s, float2 a) { s.x += a.x; s.y += a.y; }
__device__ __forceinline__ float vfold(float a, float b, float c, float d) { return (a + b) + (c + d); }
__device__ __forceinline__ float2 vfold(float2 a, float2 b, float2 c, float2 d) {
  return make_float2((a.x + b.x) + (c.x + d.x), (a.y + b.y) + (c.y + d.y));
}
template <typename V> __device__ __forceinline__ V vld(const float* p);
template <> __device__ __forceinline__ float vld<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float2 vld<float2>(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
template <typename V, int NPRE>
__device__ __forceinline__ V sum_strided_pre(const float* __restrict__ p, int n, size_t stride) {
  static_assert(NPRE % 4 == 0, "groups of four");
  V s0{}, s1{}, s2{}, s3{};
  if (n <= NPRE) {
    V a[NPRE];
#pragma unroll
    for (int i = 0; i < NPRE; ++i)
      if (i < n) a[i] = vld<V>(p + (size_t)i * stride);
#pragma unroll
    for (int i = 0; i < NPRE; i += 4)
      if (i + 4 <= n) { vacc(s0, a[i]); vacc(s1, a[i + 1]); vacc(s2, a[i + 2]); vacc(s3, a[i + 3]); }
#pragma unroll
    for (int i = 0; i < NPRE; ++i)
      if (i >= (n & ~3) && i < n) vacc(s0, a[i]);
  } else {
    int i = 0;
    for (; i + 4 <= n; i += 4) {
      const V a = vld<V>(p + (size_t)i * stride), b = vld<V>(p + (size_t)(i + 1) * stride);
      const V c = vld<V>(p + (size_t)(i + 2) * stride), d = vld<V>(p + (size_t)(i + 3) * stride);
      vacc(s0, a); vacc(s1, b); vacc(s2, c); vacc(s3, d);
    }
    for (; i < n; ++i) vacc(s0, vld<V>(p + (size_t)i * stride));
  }
  return vfold(s0, s1, s2, s3);
}
template <typename V, int NPRE>
__device__ __forceinline__ V chunk_sum8(const float* __restrict__ p, int n, size_t stride, int chunk) {
  const int per = (n + 7) / 8, lo = chunk * per, hi = min(n, lo + per);
  return hi > lo ? sum_strided_pre<V, NPRE>(p + (size_t)lo * stride, hi - lo, stride) : V{};
}
template <typename V, int NPRE>
__device__ __forceinline__ V reduce8(const float* __restrict__ p, int n, size_t stride) {
  V t = chunk_sum8<V, NPRE>(p, n, stride, 0);
#pragma unroll
  for (int c = 1; c < 8; ++c) vacc(t, chunk_sum8<V, NPRE>(p, n, stride, c));
  return t;
}

// block = 32 float4 groups (128 consecutive parameters) x 8 slot-chunks; chunk partials combined through shared
// memory in chunk order, so the result is independent of scheduling
__global__ void __launch_bounds__(256) k_reduce_grads_tc(const float* __restrict__ small1, int slots1,
                                                         const float* __restrict__ small2, const float* __restrict__ pw2,
                                                         int splits, int in_dim, int out_dim, float* __restrict__ grads,
                                                         const DpPeer dp = DpPeer{}, int dp_group = 0,
                                                         long long dp_off = 0) {
  tc::grid_dep_wait();   /* programmatic dependent launch: the predecessor's results are needed from here on */
 
  __shared__ float4 part[8][32];
  const int net = blockIdx.y;
  const int g = threadIdx.x & 31, chunk = threadIdx.x >> 5;
  const int idx = (blockIdx.x * 32 + g) * 4;                          // every region boundary is a multiple of 4
  const int w2_lo = off_W2(in_dim), w2_hi = w2_lo + H * H, total = net_floats(in_dim, out_dim);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (idx < NET_STRIDE) {
    const float* base = nullptr;
    int n = 0;
    size_t stride = 0;
    if (idx >= w2_lo && idx < w2_hi) {
      base = pw2 + (size_t)net * splits * H * H + (idx - w2_lo); n = splits; stride = (size_t)H * H;
    } else if (idx < w2_lo) {
      base = small1 + (size_t)net * slots1 * SMALL_STRIDE + idx; n = slots1; stride = SMALL_STRIDE;
    } else if (idx < total) {         // tail: (idx - H*H) keeps 16-byte alignment; entries past `total` are zero
      base = small2 + (size_t)net * splits * SMALL_STRIDE + (idx - H * H); n = splits; stride = SMALL_STRIDE;
    }
    const int per = (n + 7) / 8, lo = chunk * per, hi = min(n, lo + per);
    if (base != nullptr && hi > lo) s = sum_strided4(base + (size_t)lo * stride, hi - lo, stride);
  }
  part[chunk][g] = s;
  __syncthreads();
  if (chunk == 0 && idx < NET_STRIDE) {
    float4 t = part[0][g];
#pragma unroll
    for (int c = 1; c < 8; ++c) { const float4 v = part[c][g]; t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w; }
    *reinterpret_cast<float4*>(grads + (size_t)net * NET_STRIDE + idx) = t;
    // data-parallel (fused exchange): the local sum is pushed into every peer's staging buffer, tagged with the epoch
    if (dp.world > 1)
      dp_ll_push4(dp, dp_group, dp_slices(dp, dp_off, (long long)gridDim.y * NET_STRIDE), dp_off + (long long)net * NET_STRIDE + idx, t);
  }
}

}  // namespace tc
}  // namespace cql
