// common.cuh -- shared helpers for libbarvae (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/barvae.h"

typedef __nv_bfloat16 bf16;

namespace bvae {

void set_error(const char* fmt, ...);
int check_launch(const char* what);   // cudaGetLastError -> BVAE_ERR_CUDA (+message), counts the launch
void count_launch(int n = 1);
void note_kernel(const char* fmt, ...);   // remembered per host thread for bvae_last_kernel()
bool deterministic();                     // bvae_set_deterministic / BVAE_DETERMINISTIC
int option(const char* name, int dflt);   // bvae_set_option override, else getenv(name), else dflt (kernel-variant switches)

#define BVAE_REQUIRE(cond, code, ...)            \
  do {                                           \
    if (!(cond)) {                               \
      bvae::set_error(__VA_ARGS__);              \
      return (code);                             \
    }                                            \
  } while (0)

__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ float bf2f(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ bf16 f2bf(float v) { return __float2bfloat16_rn(v); }

// 8 bf16 <-> 8 floats through ONE 16-byte memory transaction.  The carrier is a plain uint4: a struct of
// __nv_bfloat162 members gets copied member-wise by nvcc and is split into 4-byte LDG/STG (measured: 8x the sectors).
typedef uint4 bf16x8;
__device__ __forceinline__ void unpack8(const bf16x8& p, float* f) {
  const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);            // bf16 -> fp32 is a 16-bit shift
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ bf16x8 pack8(const float* f) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
__device__ __forceinline__ bf16x8 ldg8(const bf16* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void stg8(bf16* p, const bf16x8& v) { *reinterpret_cast<uint4*>(p) = v; }
// 8 consecutive fp32 (two float4)
__device__ __forceinline__ void ldg8f(const float* p, float* f) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
  f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123 constants)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// The decoder's probability of a logit, with the accurate expf (no fast math).  fit_sigmoid_fwd_kernel, the Bernoulli
// draw and the bar score all use this one expression, so at temperature 1 they agree with the decoder bit for bit.
__device__ __forceinline__ float prob_of_logit(float l) { return 1.f / (1.f + expf(-l)); }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }
__device__ __forceinline__ float act_fwd(float v, float slope) { return v > 0.f ? v : v * slope; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// order-preserving float -> uint32 map (larger float -> larger uint)
__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
  uint32_t b = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  return __uint_as_float(b);
}
// key for "max value, smallest index wins ties"
__device__ __forceinline__ unsigned long long make_key(float v, uint32_t idx) {
  return ((unsigned long long)f2ord(v) << 32) | (unsigned long long)(0xffffffffu - idx);
}
__device__ __forceinline__ float key_val(unsigned long long k) { return ord2f((uint32_t)(k >> 32)); }
__device__ __forceinline__ uint32_t key_idx(unsigned long long k) { return 0xffffffffu - (uint32_t)(k & 0xffffffffu); }

}  // namespace bvae
