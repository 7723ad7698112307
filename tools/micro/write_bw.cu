// Micro-benchmark: what the chip sustains for the store side of the BiDAF forward (105 MB of fp32 output per call at config 2,
// as 800-byte blocks inside 3200-byte rows) -- the denominator for "how fast can the epilogues be".
//   mode 0: STG.128, a warp writes one contiguous 800-byte run (50 lanes' worth -> two instructions), grid-stride over runs
//   mode 1: cp.async.bulk shared -> global, one 800-byte run per instruction, 64 runs in flight per CTA
//   mode 2: plain contiguous STG.128 fill (memset-like)
//   mode 3: contiguous copy (LDG.128 + STG.128), read + write bytes counted (the MEASURED_PEAKS definition)
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 tools/micro/write_bw.cu -o tools/micro/write_bw
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

constexpr int ROW_FLOATS = 800, BLK_FLOATS = 200;

__global__ void __launch_bounds__(256) k_runs(float* out, long long nrows, int nblk) {
  const int lane = threadIdx.x & 31;
  const long long warp = (long long)blockIdx.x * 8 + (threadIdx.x >> 5), nwarps = (long long)gridDim.x * 8;
  const float4 v = make_float4(1.f, 2.f, 3.f, 4.f);
  for (long long r = warp; r < nrows; r += nwarps)
    for (int b = 1; b <= nblk; ++b) {
      float* p = out + r * ROW_FLOATS + b * BLK_FLOATS;
      *reinterpret_cast<float4*>(p + lane * 4) = v;
      if (lane < 18) *reinterpret_cast<float4*>(p + 128 + lane * 4) = v;
    }
}
__global__ void __launch_bounds__(256) k_bulk(float* out, long long nrows, int nblk) {
  extern __shared__ __align__(128) float stg[];
  for (int i = threadIdx.x; i < 64 * BLK_FLOATS; i += 256) stg[i] = i;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 64) {
    const uint32_t src = (uint32_t)__cvta_generic_to_shared(stg + threadIdx.x * BLK_FLOATS);
    for (long long r = (long long)blockIdx.x * 64 + threadIdx.x; r < nrows; r += (long long)gridDim.x * 64) {
      for (int b = 1; b <= nblk; ++b) {
        float* dst = out + r * ROW_FLOATS + b * BLK_FLOATS;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(BLK_FLOATS * 4) : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 4;" ::: "memory");
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
}
// mode 4 / 5: the store pattern of the epilogue of bidaf_tc4_kernel, the persistent forward with 32-column tiles that preceded
// bidaf_tc5_kernel: a warp owns 32 rows and sweeps them in
// 32-column chunks; one instruction writes 4 rows x 128 bytes (8 lanes x float4 per row); default (4) or .cs (5) stores.
template <int CS>
__global__ void __launch_bounds__(256) k_epi(float* out, long long nrows, int nblk) {
  const int lane = threadIdx.x & 31;
  const long long warp = (long long)blockIdx.x * 8 + (threadIdx.x >> 5), nwarps = (long long)gridDim.x * 8;
  const int c4 = (lane & 7) * 4, rsub = lane >> 3;
  for (long long g = warp; g < nrows / 32; g += nwarps)
    for (int cc = 0; cc < 7; ++cc) {
      if (cc * 32 + c4 >= BLK_FLOATS) continue;
      float* p = out + (g * 32 + rsub) * ROW_FLOATS + BLK_FLOATS + cc * 32 + c4;
#pragma unroll
      for (int rr = 0; rr < 8; ++rr) {
        for (int b = 0; b < nblk; ++b) {
          if (CS) asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p + b * BLK_FLOATS), "f"(1.f), "f"(2.f), "f"(3.f), "f"(4.f) : "memory");
          else *reinterpret_cast<float4*>(p + b * BLK_FLOATS) = make_float4(1.f, 2.f, 3.f, 4.f);
        }
        p += 4 * ROW_FLOATS;
      }
    }
}
__global__ void __launch_bounds__(256) k_fill(float4* out, long long n4) {
  const float4 v = make_float4(1.f, 2.f, 3.f, 4.f);
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) out[i] = v;
}
__global__ void __launch_bounds__(256) k_copy(float4* out, const float4* in, long long n4) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) out[i] = in[i];
}

int main() {
  const long long nrows = 64LL * 512 * 4;                 // 4 x config 2: 131072 rows x 3200 B = 419 MB (> L2)
  float *out, *in;
  cudaMalloc(&out, nrows * ROW_FLOATS * 4);
  cudaMalloc(&in, nrows * ROW_FLOATS * 4);
  cudaMemset(in, 0, nrows * ROW_FLOATS * 4);
  cudaFuncSetAttribute(k_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * BLK_FLOATS * 4);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int mode = 0; mode < 6; ++mode)
    for (int ctas : {148, 592, 2368}) {
      float best = 1e9f;
      for (int it = 0; it < 4; ++it) {
        cudaEventRecord(e0);
        if (mode == 0) k_runs<<<ctas, 256>>>(out, nrows, 3);
        if (mode == 1) k_bulk<<<ctas, 256, 64 * BLK_FLOATS * 4>>>(out, nrows, 3);
        if (mode == 2) k_fill<<<ctas, 256>>>(reinterpret_cast<float4*>(out), nrows * ROW_FLOATS / 4);
        if (mode == 4) k_epi<0><<<ctas, 256>>>(out, nrows, 3);
        if (mode == 5) k_epi<1><<<ctas, 256>>>(out, nrows, 3);
        if (mode == 3) k_copy<<<ctas, 256>>>(reinterpret_cast<float4*>(out), reinterpret_cast<const float4*>(in), nrows * ROW_FLOATS / 4);
        cudaEventRecord(e1);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); return 1; }
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        if (it > 0 && ms < best) best = ms;
      }
      const double bytes = (mode <= 1 || mode >= 4) ? (double)nrows * 3 * BLK_FLOATS * 4 : (double)nrows * ROW_FLOATS * 4 * (mode == 3 ? 2 : 1);
      printf("mode %d ctas %4d: %.1f us, %.2f TB/s (%s)\n", mode, ctas, best * 1e3, bytes / (best * 1e-3) / 1e12,
             mode == 0 ? "STG.128 800-byte runs x3 per 3200-byte row" : mode == 1 ? "cp.async.bulk 800-byte runs x3 per row"
             : mode == 2 ? "contiguous fill" : mode == 3 ? "contiguous copy, read+write" : mode == 4 ? "epilogue pattern: 4 rows x 128 B per instruction"
             : "epilogue pattern, st.global.cs");
    }
  return 0;
}
