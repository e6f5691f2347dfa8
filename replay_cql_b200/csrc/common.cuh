// common.cuh -- layout constants, error handling, warp helpers, Philox RNG.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>
#include "../../include/cql_b200.h"

namespace cql {

constexpr int H = CQL_HIDDEN;            // 256
constexpr int NET_STRIDE = 67136;        // floats per network slot (>= 67074, multiple of 64)
constexpr int SCALAR_SLOT = 64;          // [0]=log_temp [1]=log_alpha

// offsets inside one network slot (floats); PyTorch (out,in) row-major
__host__ __device__ constexpr int off_W1(int) { return 0; }
__host__ __device__ constexpr int off_b1(int in) { return H * in; }
__host__ __device__ constexpr int off_W2(int in) { return H * in + H; }
__host__ __device__ constexpr int off_b2(int in) { return H * in + H + H * H; }
__host__ __device__ constexpr int off_W3(int in) { return H * in + H + H * H + H; }
__host__ __device__ constexpr int off_b3(int in, int out) { return H * in + H + H * H + H + out * H; }
__host__ __device__ constexpr int net_floats(int in, int out) { return H * in + H + H * H + H + out * H + out; }

// "small" gradient block of a net = everything except W2, packed [W1|b1|b2|W3|b3]
__host__ __device__ constexpr int small_floats(int in, int out) { return H * in + H + H + out * H + out; }
constexpr int SMALL_STRIDE = 1856;       // >= small_floats(3,1)=1537 and small_floats(2,2)=1794, mult of 64

// slot indices in the flat state
__host__ __device__ inline int slot_actor() { return 0; }
__host__ __device__ inline int slot_critic(int c) { return 1 + c; }
__host__ __device__ inline int slot_targ_actor(int C) { return 1 + C; }
__host__ __device__ inline int slot_targ_critic(int C, int c) { return 2 + C + c; }
__host__ __device__ inline int64_t scalars_off(int C) { return (int64_t)(2 + 2 * C) * NET_STRIDE; }
__host__ __device__ inline int64_t state_floats(int C) { return scalars_off(C) + SCALAR_SLOT; }
// trainable gradient buffer: [actor | critics | scalars]
__host__ __device__ inline int64_t grad_floats(int C) { return (int64_t)(1 + C) * NET_STRIDE + SCALAR_SLOT; }

// ---------------------------------------------------------------- errors
struct Error { std::string msg; };
struct ArgError : Error {};          // a rejected argument or call sequence (CQL_REQUIRE): the C API returns 3
#define CQL_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      throw ::cql::Error{std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" +      \
                         __FILE__ + ":" + std::to_string(__LINE__) + ")"};               \
  } while (0)
#define CQL_REQUIRE(cond, text)                                                          \
  do {                                                                                   \
    if (!(cond)) throw ::cql::ArgError{{std::string(text)}};                             \
  } while (0)

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Philox4x32-10 (Salmon et al. 2011), counter-based: no state in memory.
struct Philox {
  __host__ __device__ static inline void round(uint32_t (&c)[4], uint32_t (&k)[2]) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k[0];
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k[1];
    uint32_t n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
  }
  // 4 x 32 random bits for (seed, stream, index)
  __host__ __device__ static inline void gen(uint64_t seed, uint64_t stream, uint64_t index, uint32_t (&out)[4]) {
    uint32_t c[4] = {(uint32_t)index, (uint32_t)(index >> 32), (uint32_t)stream, (uint32_t)(stream >> 32)};
    uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
    for (int i = 0; i < 10; ++i) round(c, k);
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
  }
};
// (0, 1] from 32 bits: the float32 sum rounds to even from x >> 8 = 2^23 on, so x >> 8 = 2^24 - 1 gives exactly 1
__host__ __device__ inline float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

}  // namespace cql
