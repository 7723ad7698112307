// Shared helpers for the mmbidaf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/mmbidaf_b200.h"

namespace mmb {

void set_error(const char* fmt, ...);

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return MMB_ERR_CUDA;
  }
  return MMB_OK;
}

#define MMB_REQUIRE(cond, code, ...)      \
  do {                                    \
    if (!(cond)) {                        \
      ::mmb::set_error(__VA_ARGS__);      \
      return code;                        \
    }                                     \
  } while (0)

#define MMB_CUDA(call)                                                        \
  do {                                                                        \
    cudaError_t e_ = (call);                                                  \
    if (e_ != cudaSuccess) {                                                  \
      ::mmb::set_error("%s failed: %s", #call, cudaGetErrorString(e_));       \
      return MMB_ERR_CUDA;                                                    \
    }                                                                         \
  } while (0)

constexpr float kNegFill = -1e30f;   // layers/attention.py:94

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
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
// Branch-free gate non-linearities for the serial LSTM chain: act_k(x) = 1 - k / (1 + e^{kx}) is tanh for
// k = 2 and the logistic sigmoid for k = 1.  __expf / __fdividef keep the absolute error near 1e-7
// (measured against the fp64 oracle in tests/test_lstm_gpu.py), which is what the gates need.
// Counter-based keep mask for dropout applied INSIDE a kernel: element `idx` of a tensor is kept iff hash(idx, key) < keep_prob 2^32.
// A 32-bit avalanche hash (two multiplies and three xor-shifts around the two key halves): nine integer instructions, the same bits
// wherever they are recomputed (the forward store, the backward load, mmb_dropout_mask in the tests).  Not ATen's Philox stream:
// bit-parity of the random stream with the reference is not a goal (DESIGN.md section 1), parity GIVEN the mask is tested.
__device__ __forceinline__ uint32_t hash32(uint32_t idx, uint32_t k0, uint32_t k1) {
  uint32_t x = idx ^ k0;
  x *= 0x9E3779B1u;
  x ^= x >> 16;
  x *= 0x85EBCA6Bu;
  x ^= k1;
  x ^= x >> 13;
  x *= 0xC2B2AE35u;
  x ^= x >> 16;
  return x;
}
__device__ __forceinline__ bool dropout_keep(uint32_t idx, uint32_t k0, uint32_t k1, uint32_t thresh) {
  return hash32(idx, k0, k1) < thresh;
}
// The Gumbel-max score of a sampled pick (the rule at mmb_decoder_sample_fused): z = logf(p) inv_t - logf(-logf(u)) with the uniform
// u = ((hash32(c, key) >> 9) + 0.5) 2^-23 of counter c.  Every step of u is exact in fp32 (23 bits plus the half), so u lies in
// [2^-24, 1 - 2^-24] and -logf(-logf(u)) is finite: z is -inf for p = 0 and finite for p > 0.  (With 24 bits the top value would round
// to u = 1 and give z = +inf.)  The roll-out kernel and mmb_sample_pick both call this one function, so both give the same bits.
__device__ __forceinline__ float sample_score(float p, float inv_t, uint32_t c, uint32_t k0, uint32_t k1) {
  const float u = ((float)(hash32(c, k0, k1) >> 9) + 0.5f) * 1.1920928955078125e-7f;
  return logf(p) * inv_t - logf(-logf(u));
}
__host__ __device__ __forceinline__ uint32_t dropout_thresh(float keep_prob) {
  const double t = (double)keep_prob * 4294967296.0;
  return t >= 4294967295.0 ? 0xffffffffu : (t <= 0.0 ? 0u : (uint32_t)t);
}

__device__ __forceinline__ float gate_act(float x, float k) { return 1.0f - __fdividef(k, 1.0f + __expf(k * x)); }
__device__ __forceinline__ float tanh_fast(float x) { return gate_act(x, 2.0f); }

}  // namespace mmb
