// mlp_tc_bwd2.cuh -- tensor-core weight gradient of the hidden layer:  dW2 = dZ2^T H1  (256 x 256 x rows).
//
// Both operands are *generated on chip* per K-stage (K = rows): thread t owns hidden unit t and writes
//   A[j=t][r] = dZ2[r][j] = (sum_o dOut[r][o] W3[o][j]) * (H2[r][j] > 0)        (needs H2, 4 B/elt from HBM/L2)
//   B[k=t][r] = H1[r][k]  = relu(W1[k].x[r] + b1[k])                              (recomputed, 3 FMAs)
// straight into the UMMA K-major operand layout, so neither dZ2 nor H1 ever exists in memory.
// The 256x256 FP32 accumulator occupies the whole TMEM (2 M-halves x 256 columns) and stays there
// across ALL row tiles of the CTA; it is written out once, as one split-partial.
// Because thread t sees every row of unit t, the same pass yields db2, dW3 and db3 for free.
#pragma once
#include "tc_common.cuh"
#include "mlp_simt.cuh"

namespace cql {
namespace tc {

constexpr int B2_PROD_WARPS = 8;
constexpr int B2_THREADS = (B2_PROD_WARPS + 1) * 32;   // 8 producer warps + 1 MMA warp

template <bool TF32>
struct B2Cfg {
  static constexpr int ES = TF32 ? 4 : 2;
  static constexpr int EPC = 16 / ES;
  static constexpr int UK = 32 / ES;
  static constexpr int TERMS = TF32 ? 2 : 1;
  static constexpr int RS = TF32 ? 16 : 64;              // rows (K extent) per stage
  static constexpr int STAGES = 3;
  static constexpr uint32_t OP_TERM_BYTES = H * RS * ES;  // 16 KB / 32 KB
  static constexpr uint32_t OP_BYTES = TERMS * OP_TERM_BYTES;   // 32 KB
  static constexpr uint32_t STAGE_BYTES = 2 * OP_BYTES;         // A then B: 64 KB
  static constexpr uint32_t OFF_X = STAGES * STAGE_BYTES;       // float4[STAGES][RS]
  static constexpr uint32_t OFF_DO = OFF_X + STAGES * RS * 16;  // float[STAGES][RS][2]
  static constexpr uint32_t OFF_BAR = OFF_DO + STAGES * RS * 8;
  static constexpr uint32_t OFF_SLOT = OFF_BAR + (2 * STAGES + 1) * 8;
  static constexpr uint32_t BYTES = OFF_SLOT + 16;
};

struct Bwd2Job {
  const float4* X;      // [rows]
  const float* dOut;    // [n_nets][rows][OUT]
  const float* h2;      // [n_nets][tiles64][256][64]
  const float* params;  // first net slot (fp32)
  float* pw2;           // [n_nets][splits][256*256]
  float* small2;        // [n_nets][splits][SMALL_STRIDE]: only b2 | W3 | b3 entries written (same offsets as `small`)
  int rows, n_nets, splits;
};

template <bool TF32, int IN, int OUT>
__global__ void __launch_bounds__(B2_THREADS, 1) tc_bwd2_kernel(const Bwd2Job jb) {
  using C = B2Cfg<TF32>;
  extern __shared__ __align__(1024) uint8_t sm[];
  float4* xs = reinterpret_cast<float4*>(sm + C::OFF_X);
  float* dos = reinterpret_cast<float*>(sm + C::OFF_DO);
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + C::OFF_BAR);
  uint64_t* empty = full + C::STAGES;
  uint64_t* done = empty + C::STAGES;
  uint32_t* slot = reinterpret_cast<uint32_t*>(sm + C::OFF_SLOT);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = blockIdx.x, net_i = blockIdx.y;
  const float* net = jb.params + (size_t)net_i * NET_STRIDE;
  const int tiles64 = (jb.rows + 63) / 64;
  const int n_stage_total = (jb.rows + C::RS - 1) / C::RS;      // K stages over all rows of the net
  // contiguous share of the stages for this split
  const int st_lo = (int)((long long)n_stage_total * split / jb.splits);
  const int st_hi = (int)((long long)n_stage_total * (split + 1) / jb.splits);

  if (warp == B2_PROD_WARPS) {
    tmem_alloc(slot, 512);
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], B2_PROD_WARPS); mbar_init(&empty[s], 1); }
      mbar_init(done, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *slot;

  if (warp == B2_PROD_WARPS) {
    {
      const uint32_t idesc = instr_desc(TF32 ? FMT_TF32 : FMT_BF16, 128, 256);
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
            const uint32_t d = tmem + half * 256;
            if constexpr (TF32) {
              const uint64_t a_lo = smem_desc(a_base + C::OP_TERM_BYTES + half * 2048 + 2 * j * lbo, lbo, 128);
              const uint64_t b_lo = smem_desc(b_base + C::OP_TERM_BYTES + 2 * j * lbo, lbo, 128);
              umma<TF32>(d, a_lo, b_hi, idesc, acc);
              umma<TF32>(d, a_hi, b_lo, idesc, 1u);
              umma<TF32>(d, a_hi, b_hi, idesc, 1u);
            } else {
              umma<TF32>(d, a_hi, b_hi, idesc, acc);
            }
          }
        }
        umma_commit(&empty[s]);
        if (sg == st_hi - 1) umma_commit(done);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------- producers: thread t = hidden unit t (A row j = t, B row k = t) ----------------
    const int t = tid;   // 0..255
    float w3[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) w3[o] = net[off_W3(IN) + o * H + t];
    const float w1x = net[off_W1(IN) + t * IN], w1y = net[off_W1(IN) + t * IN + 1];
    const float w1z = IN == 3 ? net[off_W1(IN) + t * IN + 2] : 0.f;
    const float b1v = net[off_b1(IN) + t];
    float s_db2 = 0.f, s_dw3[OUT], s_db3[OUT];
#pragma unroll
    for (int o = 0; o < OUT; ++o) { s_dw3[o] = 0.f; s_db3[o] = 0.f; }
    uint32_t it = 0;
    constexpr int NV = C::RS / 4;                      // float4 loads of H2 per thread per stage
    constexpr bool PREFETCH = NV <= 4;                 // keep next stage's H2 in registers (tf32: 16 regs)
    float4 hnext[PREFETCH ? NV : 1];
    auto h2_ptr = [&](int sg) {
      const int row0 = sg * C::RS;
      return jb.h2 + (((size_t)net_i * tiles64 + (row0 >> 6)) * H + t) * 64 + (row0 & 63);
    };
    if (PREFETCH && st_lo < st_hi) {
      const float* hp = h2_ptr(st_lo);
#pragma unroll
      for (int q = 0; q < NV; ++q) hnext[q] = __ldg(reinterpret_cast<const float4*>(hp) + q);
    }
    for (int sg = st_lo; sg < st_hi; ++sg, ++it) {
      const uint32_t s = it % C::STAGES;
      float4 hcur[PREFETCH ? NV : 1];
      if (PREFETCH) {
#pragma unroll
        for (int q = 0; q < NV; ++q) hcur[q] = hnext[q];
        if (sg + 1 < st_hi) {
          const float* hp = h2_ptr(sg + 1);
#pragma unroll
          for (int q = 0; q < NV; ++q) hnext[q] = __ldg(reinterpret_cast<const float4*>(hp) + q);
        }
      }
      mbar_wait(&empty[s], ((it / C::STAGES) & 1) ^ 1);
      const int row0 = sg * C::RS;
      float4* xst = xs + s * C::RS;
      float* dost = dos + s * C::RS * 2;
      if (t < C::RS) {
        const int r = row0 + t;
        xst[t] = r < jb.rows ? __ldg(jb.X + r) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int o = 0; o < OUT; ++o)
          dost[t * 2 + o] = r < jb.rows ? __ldg(jb.dOut + ((size_t)net_i * jb.rows + r) * OUT + o) : 0.f;
      }
      asm volatile("bar.sync 1, 256;");
      uint8_t* Ast = sm + s * C::STAGE_BYTES;
      uint8_t* Bst = Ast + C::OP_BYTES;
      const float* h2p = h2_ptr(sg);
#pragma unroll
      for (int kc = 0; kc < C::RS / C::EPC; ++kc) {
        float hv[C::EPC], dz[C::EPC], h1[C::EPC];
        if constexpr (C::EPC == 8) {
          const float4 p0 = __ldg(reinterpret_cast<const float4*>(h2p + kc * 8));
          const float4 p1 = __ldg(reinterpret_cast<const float4*>(h2p + kc * 8 + 4));
          hv[0] = p0.x; hv[1] = p0.y; hv[2] = p0.z; hv[3] = p0.w;
          hv[4] = p1.x; hv[5] = p1.y; hv[6] = p1.z; hv[7] = p1.w;
        } else {
          const float4 p0 = PREFETCH ? hcur[kc % NV] : __ldg(reinterpret_cast<const float4*>(h2p + kc * 4));
          hv[0] = p0.x; hv[1] = p0.y; hv[2] = p0.z; hv[3] = p0.w;
        }
#pragma unroll
        for (int e = 0; e < C::EPC; ++e) {
          const int rl = kc * C::EPC + e;
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
          float z = fmaf(x.y, w1y, x.x * w1x);
          if (IN == 3) z = fmaf(x.z, w1z, z);
          h1[e] = fmaxf(z + b1v, 0.f);
        }
        const uint32_t off = chunk_off(H, t, kc);
        if constexpr (TF32) {
          float4 hi, lo;
          split_tf32(dz[0], hi.x, lo.x); split_tf32(dz[1], hi.y, lo.y); split_tf32(dz[2], hi.z, lo.z); split_tf32(dz[3], hi.w, lo.w);
          *reinterpret_cast<float4*>(Ast + off) = hi;
          *reinterpret_cast<float4*>(Ast + C::OP_TERM_BYTES + off) = lo;
          split_tf32(h1[0], hi.x, lo.x); split_tf32(h1[1], hi.y, lo.y); split_tf32(h1[2], hi.z, lo.z); split_tf32(h1[3], hi.w, lo.w);
          *reinterpret_cast<float4*>(Bst + off) = hi;
          *reinterpret_cast<float4*>(Bst + C::OP_TERM_BYTES + off) = lo;
        } else {
          __nv_bfloat162 q[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) q[e] = __floats2bfloat162_rn(dz[2 * e], dz[2 * e + 1]);
          *reinterpret_cast<uint4*>(Ast + off) = *reinterpret_cast<uint4*>(q);
#pragma unroll
          for (int e = 0; e < 4; ++e) q[e] = __floats2bfloat162_rn(h1[2 * e], h1[2 * e + 1]);
          *reinterpret_cast<uint4*>(Bst + off) = *reinterpret_cast<uint4*>(q);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
    }
    // small gradients owned by this unit (same offsets as the CUDA-core kernels' `small` block)
    float* sm2 = jb.small2 + ((size_t)net_i * jb.splits + split) * SMALL_STRIDE;
    sm2[H * IN + H + t] = s_db2;
#pragma unroll
    for (int o = 0; o < OUT; ++o) sm2[H * IN + 2 * H + o * H + t] = s_dw3[o];
    if (t == 0) {
#pragma unroll
      for (int o = 0; o < OUT; ++o) sm2[H * IN + 2 * H + OUT * H + o] = s_db3[o];
    }
  }
  // ---------------- epilogue: dump the 256x256 accumulator as this split's partial ----------------
  float* out = jb.pw2 + ((size_t)net_i * jb.splits + split) * H * H;
  if (warp < 4) {
    if (st_hi > st_lo) {
      mbar_wait(done, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      float* orow = out + (size_t)(half * 128 + warp * 32 + lane) * H;
#pragma unroll 1
      for (int c0 = 0; c0 < H; c0 += 32) {
        float v[32];
        if (st_hi > st_lo) {
          tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + half * 256 + c0, v);
          tmem_ld_wait();
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
  if (warp == B2_PROD_WARPS) tmem_dealloc(tmem, 512);
}

}  // namespace tc
}  // namespace cql
