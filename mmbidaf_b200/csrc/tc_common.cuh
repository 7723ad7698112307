// tcgen05 / TMEM / TMA building blocks shared by the tensor-core BiDAF kernels (forward and backward).
// sm_100a only.  Operand layout ("pack"): bf16 rows in UMMA core-matrix order
//     pack[b][row/8][chunk 0..25][row%8][8 x bf16]          (8 rows x 16 bytes = one 128-byte core matrix)
// so any run of consecutive rows (a multiple of 8) is one contiguous block of memory; the same bytes serve as a
// K-major operand (LBO 128, SBO GROUP_BYTES) and as an MN-major operand (LBO GROUP_BYTES, SBO 128).
#pragma once
#include <cuda_bf16.h>
#include "common.cuh"

namespace mmb {
namespace tc {

constexpr int DPAD = 208;                 // K / N padding of d (d <= 200 so that chunk 25 is free for the terms)
constexpr int CHUNKS = DPAD / 8;          // 26 sixteen-byte chunks per row
constexpr int GROUP_BYTES = CHUNKS * 128; // 8 rows
constexpr int TMEM_COLS = 512;
constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;

// ---------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// One lane of a converged warp (1 for the elected lane, 0 for the others).  The single-thread instructions below
// (tcgen05.mma / commit, TMA issue) take it as `leader` and are executed by ALL lanes of the issuing warp with the
// instruction itself predicated on it: their operands are then computed in warp-uniform control flow and ptxas keeps
// them in uniform registers.  Issuing them under `if (tid == 0)` makes it emit a per-instruction ELECT /
// R2UR.BROADCAST loop instead (measured: 63 cycles per tcgen05.mma).
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred;
}
// Warp index as a value the compiler knows to be warp-uniform.
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %2, 0;\n\t"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t"
      "}" ::"r"(bar), "r"(bytes), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  // try_wait suspends for a hardware time slice; the bound turns a protocol bug into a trap instead of a hang.
  // unroll 1: the compiler otherwise unrolls the poll ~30 times at every call site (2 700 of the 6 600 SASS instructions of the
  // cut-5 forward kernel), and these kernels are instruction-cache bound before they are anything else.
#pragma unroll 1
  for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %4, 0;\n\t"
      "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t"
      "}" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ long long globaltimer_ns() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// Inter-CTA ordering inside one launch (producer blocks have lower block indices than their consumers).
__device__ __forceinline__ void signal_counter(int* counter) {
  __threadfence();
  asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(counter) : "memory");
}
__device__ __forceinline__ void wait_counter(const int* counter, int target) {
  // bounded: a scheduling surprise becomes a trap (an error to the caller), not a hang
#pragma unroll 1
  for (uint32_t spin = 0; spin < (1u << 24); ++spin) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    if (v >= target) return;
    __nanosleep(64);
  }
  __trap();
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate.  Executed by a converged warp, issued by its leader.
// The descriptors are given as (low word, high word): the high word (SBO, version) is a constant and the low
// word (address >> 4 | LBO) advances by a constant per K step, so the issue loop is one integer add per operand.
__device__ __forceinline__ void umma_bf16_lh(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                             uint32_t idesc, uint32_t acc, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc), "r"(leader)
      : "memory");
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr, uint32_t lbo_bytes) { return ((addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16); }
constexpr uint32_t desc_hi(uint32_t sbo_bytes) { return (sbo_bytes >> 4) | (1u << 14); }
__device__ __forceinline__ void umma_commit(uint32_t bar, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(bar), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}

// Instruction descriptor: D = F32, A = B = BF16.  M = 128: accumulator row i is TMEM lane i.  M = 64: row i is lane
// (i / 16) * 32 + i % 16 -- sixteen rows in the low half of each 32-lane quarter (tools/micro/umma_m64_layout.cu).
constexpr uint32_t idesc_bf16(int n, int b_mn_major, int m = 128) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// 2^x as one MUFU.EX2: results below 2^-126 flush to zero (exp2f spends three more instructions on them), which for
// soft-max weights that are rounded to bf16 or summed in fp32 next is exact enough.
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Layout of the forward workspace (mmb_bidaf_workspace_bytes): the bf16 packs and mask words the forward pass
// produces and the backward pass re-uses.  Lengths are padded to PACK_ROWS rows.
constexpr int PACK_ROWS = 128;
struct BidafPacks {
  __nv_bfloat16 *cw, *cp;            // text: S operand (dropped, w_cq folded, term chunk) / plain values
  __nv_bfloat16 *qs, *qp;            // modality: S operand (dropped, term chunk) / plain values (== qs without dropout)
  __nv_bfloat16* tp;                 // packed T = s2^T c
  unsigned long long *c_words, *q_words;   // (B, LP/64, 2): [in-range bits, un-masked bits] per 64 rows
  int* ready;                        // (B) Q2C -> C2Q dependency counters of the main launch, then its work-queue head
  int LcP, LqP;
  size_t c_pack, q_pack, bytes;
};
inline BidafPacks bidaf_packs(void* workspace, int B, int Lc, int Lq, bool modality_dropout) {
  BidafPacks p;
  p.LcP = round_up(Lc, PACK_ROWS);
  p.LqP = round_up(Lq, PACK_ROWS);
  p.c_pack = (size_t)B * (p.LcP / 8) * GROUP_BYTES;
  p.q_pack = (size_t)B * (p.LqP / 8) * GROUP_BYTES;
  char* ws = static_cast<char*>(workspace);
  p.cw = reinterpret_cast<__nv_bfloat16*>(ws);
  p.cp = reinterpret_cast<__nv_bfloat16*>(ws + p.c_pack);
  p.qs = reinterpret_cast<__nv_bfloat16*>(ws + 2 * p.c_pack);
  p.tp = reinterpret_cast<__nv_bfloat16*>(ws + 2 * p.c_pack + p.q_pack);
  char* next = ws + 2 * p.c_pack + 2 * p.q_pack;
  p.qp = p.qs;
  if (modality_dropout) {
    p.qp = reinterpret_cast<__nv_bfloat16*>(next);
    next += p.q_pack;
  }
  p.c_words = reinterpret_cast<unsigned long long*>(next);
  p.q_words = p.c_words + (size_t)B * (p.LcP / 64) * 2;
  const size_t used = ((size_t)(next - ws) + 16 * (size_t)B * (p.LcP / 64 + p.LqP / 64) + 255) / 256 * 256;
  p.ready = reinterpret_cast<int*>(ws + used);
  p.bytes = used + ((size_t)(B + 1) * 4 + 255) / 256 * 256;
  return p;
}

}  // namespace tc
}  // namespace mmb
