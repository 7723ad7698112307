// The sampled pick of given distribution rows (mmb_sample_pick): steps 1 to 4 of the rule at mmb_decoder_sample_fused in
// include/mmbidaf_b200.h, one CTA per row, with the roll-out kernel's score function (common.cuh::sample_score).  The rule is a top-k
// set (p descending, m ascending) and an arg-max of z with ties to the smaller m: it does not depend on how the rows are split, so
// this kernel gives the cluster kernel's picks bit for bit.  The tests use it as the reference pick of a host loop.
// With top_p < 1 (mmb_sample_pick_nucleus) the draw is over the nucleus of the rule at mmb_decoder_sample_nucleus_fused, found here
// by another algorithm than the roll-out kernel's radix select: the candidates one block-wide "next best" round at a time, their
// integer masses summed until need is reached.
#include <limits.h>
#include <math.h>
#include "common.cuh"

namespace mmb {
namespace {

constexpr int PT = 256;
constexpr int PW = PT / 32;

// a ranks before b: p descending, then m ascending (m = INT_MAX: no entry)
__device__ __forceinline__ bool pick_before(float pa, int ma, float pb, int mb) { return pa != pb ? pa > pb : ma < mb; }

// the block's best (p, m) ranked after (p0, m0), in every thread
__device__ void block_next(float& p, int& m, float* s_p, int* s_m) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float p2 = __shfl_xor_sync(0xffffffffu, p, o);
    const int m2 = __shfl_xor_sync(0xffffffffu, m, o);
    if (pick_before(p2, m2, p, m)) { p = p2; m = m2; }
  }
  __syncthreads();
  if (lane == 0) { s_p[warp] = p; s_m[warp] = m; }
  __syncthreads();
  p = s_p[0];
  m = s_m[0];
  for (int w = 1; w < PW; ++w)
    if (pick_before(s_p[w], s_m[w], p, m)) { p = s_p[w]; m = s_m[w]; }
}

// the integer mass of the nucleus rule: floor(p 2^24), exact from the fp32 p
__device__ __forceinline__ unsigned long long mass(float p) { return __float2uint_rz(p * 16777216.f); }

// P = rint(top_p 2^24); P = 2^24 (top_p = 1): no cut
__global__ void __launch_bounds__(PT) sample_pick_kernel(const float* __restrict__ probs, const uint8_t* __restrict__ eligible,
                                                         const unsigned long long* __restrict__ key_ptr, const int* __restrict__ row_base,
                                                         int M, int S, int s, int N, float T, int top_k, uint32_t P,
                                                         long long* __restrict__ picks) {
  __shared__ float s_p[PW];
  __shared__ int s_m[PW];
  __shared__ unsigned long long s_q[PW];
  const int r = blockIdx.x, tid = threadIdx.x;
  const unsigned long long key = *key_ptr;
  const uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
  const float inv_t = 1.f / T;
  const uint32_t cbase = (((uint32_t)row_base[r] * (uint32_t)N + (uint32_t)(r % N)) * (uint32_t)S + (uint32_t)s) * (uint32_t)M;
  const float* p = probs + (size_t)r * M;
  const uint8_t* el = eligible ? eligible + (size_t)r * M : nullptr;
  float bz = -INFINITY;
  int bm = INT_MAX;                                          // no candidate yet
  if (P < (1u << 24)) {
    // Q: the mass of every candidate (top_k = 0), or of the first top_k
    unsigned long long Q = 0;
    if (top_k == 0) {
      for (int m = tid; m < M; m += PT)
        if (!el || el[m]) Q += mass(p[m]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) Q += __shfl_xor_sync(0xffffffffu, Q, o);
      if ((tid & 31) == 0) s_q[tid >> 5] = Q;
      __syncthreads();
      Q = 0;
      for (int w = 0; w < PW; ++w) Q += s_q[w];
    } else {
      float lp = INFINITY;
      int lm = -1;
      for (int j = 0; j < top_k; ++j) {
        float cp = -INFINITY;
        int cm = INT_MAX;
        for (int m = tid; m < M; m += PT) {
          if (el && !el[m]) continue;
          if (pick_before(lp, lm, p[m], m) && pick_before(p[m], m, cp, cm)) { cp = p[m]; cm = m; }
        }
        block_next(cp, cm, s_p, s_m);
        if (cm == INT_MAX) break;
        Q += mass(cp);
        lp = cp;
        lm = cm;
      }
    }
    const unsigned long long pq = (unsigned long long)P * Q;
    const unsigned long long need = (pq >> 24) + ((pq & 0xffffffull) != 0ull);
    // the candidates in order until their mass reaches need (at least one), each drawn for
    float lp = INFINITY;
    int lm = -1;
    unsigned long long acc = 0;
    for (;;) {
      float cp = -INFINITY;
      int cm = INT_MAX;
      for (int m = tid; m < M; m += PT) {
        if (el && !el[m]) continue;
        if (pick_before(lp, lm, p[m], m) && pick_before(p[m], m, cp, cm)) { cp = p[m]; cm = m; }
      }
      block_next(cp, cm, s_p, s_m);
      if (cm == INT_MAX) break;                              // no candidate left (none at all: -1)
      const float z = sample_score(cp, inv_t, cbase + (uint32_t)cm, k0, k1);
      if (bm == INT_MAX || z > bz || (z == bz && cm < bm)) { bz = z; bm = cm; }
      acc += mass(cp);
      if (acc >= need) break;
      lp = cp;
      lm = cm;
    }
    if (tid == 0) picks[r] = bm == INT_MAX ? -1 : bm;
    return;
  }
  if (top_k == 0) {
    for (int m = tid; m < M; m += PT) {
      if (el && !el[m]) continue;
      const float z = sample_score(p[m], inv_t, cbase + (uint32_t)m, k0, k1);
      if (bm == INT_MAX || z > bz) { bz = z; bm = m; }       // (m ascends within a thread: ties keep the smaller)
    }
  } else {
    // the top_k candidates, one block-wide pick per round, each ranked after the last; the draw among them in every thread
    float lp = INFINITY;
    int lm = -1;
    for (int j = 0; j < top_k; ++j) {
      float cp = -INFINITY;
      int cm = INT_MAX;
      for (int m = tid; m < M; m += PT) {
        if (el && !el[m]) continue;
        if (pick_before(lp, lm, p[m], m) && pick_before(p[m], m, cp, cm)) { cp = p[m]; cm = m; }
      }
      block_next(cp, cm, s_p, s_m);
      if (cm == INT_MAX) break;                              // fewer than top_k candidates
      const float z = sample_score(cp, inv_t, cbase + (uint32_t)cm, k0, k1);
      if (tid == 0 && (bm == INT_MAX || z > bz || (z == bz && cm < bm))) { bz = z; bm = cm; }
      lp = cp;
      lm = cm;
    }
    if (tid == 0) picks[r] = bm == INT_MAX ? -1 : bm;
    return;
  }
  // the largest z, ties to the smaller m: the block's best (z, -m)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float z2 = __shfl_xor_sync(0xffffffffu, bz, o);
    const int m2 = __shfl_xor_sync(0xffffffffu, bm, o);
    if (m2 != INT_MAX && (bm == INT_MAX || z2 > bz || (z2 == bz && m2 < bm))) { bz = z2; bm = m2; }
  }
  if ((tid & 31) == 0) { s_p[tid >> 5] = bz; s_m[tid >> 5] = bm; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < PW; ++w)
      if (s_m[w] != INT_MAX && (bm == INT_MAX || s_p[w] > bz || (s_p[w] == bz && s_m[w] < bm))) { bz = s_p[w]; bm = s_m[w]; }
    picks[r] = bm == INT_MAX ? -1 : bm;
  }
}

static int sample_pick(const float* probs, const uint8_t* eligible, const unsigned long long* key, const int* row_base, int R, int M,
                       int S, int s, int N, float T, int top_k, long long* picks, float top_p, mmb_stream_t stream, const char* who) {
  MMB_REQUIRE(probs && key && row_base && picks, MMB_ERR_INVALID, "%s: null pointer", who);
  MMB_REQUIRE(R > 0 && M > 0 && S > 0 && s >= 0 && s < S && N >= 1 && N <= 64 && T > 0.f && isfinite(T) && top_k >= 0 && top_k <= 8 &&
                  top_p > 0.f && top_p <= 1.f,
              MMB_ERR_INVALID, "%s: R=%d M=%d S=%d s=%d N=%d (1..64) T=%g (finite, > 0) top_k=%d (0..8) top_p=%g (in (0, 1])", who, R, M,
              S, s, N, (double)T, top_k, (double)top_p);
  MMB_REQUIRE(top_p == 1.f || M < 65536, MMB_ERR_UNSUPPORTED, "%s: M=%d (below 65536 with top_p < 1)", who, M);
  const uint32_t P = (uint32_t)rintf(top_p * 16777216.f);
  sample_pick_kernel<<<R, PT, 0, static_cast<cudaStream_t>(stream)>>>(probs, eligible, key, row_base, M, S, s, N, T, top_k, P, picks);
  return check_launch("sample_pick_kernel");
}

}  // namespace
}  // namespace mmb

extern "C" int mmb_sample_pick(const float* probs, const uint8_t* eligible, const unsigned long long* key, const int* row_base, int R,
                               int M, int S, int s, int N, float T, int top_k, long long* picks, mmb_stream_t stream) {
  return mmb::sample_pick(probs, eligible, key, row_base, R, M, S, s, N, T, top_k, picks, 1.f, stream, "mmb_sample_pick");
}

extern "C" int mmb_sample_pick_nucleus(const float* probs, const uint8_t* eligible, const unsigned long long* key, const int* row_base,
                                       int R, int M, int S, int s, int N, float T, int top_k, long long* picks, float top_p,
                                       mmb_stream_t stream) {
  return mmb::sample_pick(probs, eligible, key, row_base, R, M, S, s, N, T, top_k, picks, top_p, stream, "mmb_sample_pick_nucleus");
}
