// Fused BiDAF attention forward, tensor-core tier, cut 5: ONE persistent, warp-specialised CTA per SM, 64-column S tiles,
// P handed to the tensor core through TENSOR MEMORY, a split accumulator, and a staged, row-coalesced drain.
//
// What the earlier cuts measured (profiles/r02_bidaf_fwd.md): a 32-column tile cost 1.4 - 2.4 us against ~0.37 us of tensor
// time because every tile is a chain of barrier round trips (TMA -> MMA -> commit -> tcgen05.ld -> soft-max -> st.shared ->
// proxy fence -> MMA), the S products re-read the 4 KB X operand from shared memory for every 128 x 32 x 16 instruction
// (40 cycles against a floor of 16), S was evaluated three times (Q2C, C2QA, C2QB blocks), and the output went to memory in
// 128-byte runs.  Here
//   * a tile is 128 X rows x 64 Y rows (half the round trips of the 32-column cuts per element, a 128 x 64 x 16 product costs
//     49 cycles against a floor of 32);
//   * P never touches shared memory: the soft-max threads write it as packed bf16 into TMEM and the P V product takes its A
//     operand from there (tcgen05.mma [d], [a], b-desc; layout checked by tools/micro/umma_tmem_a.cu);
//   * the text-side block keeps its X tile for both of its passes (a = s1 q, then b = s1 T);
//   * the 208-column accumulator is split into LO (112 columns, double buffered) and HI (96 columns): 2 x 64 (S) + 2 x 32 (P) +
//     2 x 112 + 96 = 512 TMEM columns, so the drain of pass n runs under the tile loop of pass n + 1;
//   * the drain goes TMEM -> registers -> a padded shared-memory stage -> whole row runs (up to 448 bytes) of `out`, with the
//     c * a / c * b products formed from the fp32 text on the way out.
//
//   warps 0-3    soft-max     one thread per X row (TMEM lane): masked streaming soft-max (base 2, lazy rescale) of a 64-column tile
//   warps 4-7    epilogue     drain: HI first (single buffered), then LO
//   warp 8       MMA issuer   S(t + 1) is issued before P V(t)
//   warp 9       scheduler + TMA producer of the Y tiles (4 slots of 64 rows; a tile takes one slot when its value operand is its
//                S operand, else two)
//   warp 10      X loader
//
// Work items (global atomic queue): Q2C(b, 128 modality rows): T = softmax_i(S)^T c  -> packed bf16 T (+ fp32 T, lse_col);
// C2Q(b, 128 text rows): pass A  a = softmax_j(S) q -> out blocks 1, 2, lse_row;  pass B  b = softmax_j(S) T -> out block 3 (+ bm).
// All Q2C items precede the C2Q items in the queue; pass B waits for its batch row's Q2C items (ready[b]), which were claimed
// earlier by CTAs that are running -- no assumption on block scheduling.
#include <stdlib.h>
#include "tc_common.cuh"

namespace mmb {
using namespace tc;
namespace {

constexpr int TX = 128, TY = 64;
constexpr int X_BYTES = TX / 8 * GROUP_BYTES;       // 53248
constexpr int SLOT_BYTES = TY / 8 * GROUP_BYTES;    // 26624
constexpr int NSLOT = 4;
constexpr int STG_STRIDE = 116;                     // floats per staged row (112 + 4: conflict-free 128-bit accesses by 8 rows)
constexpr int STG_BYTES = TX * STG_STRIDE * 4;      // 59392
constexpr int NSOFT = 4, NEPI = 4;
// 12 warps = 384 threads: 168 registers per thread (with 15 warps the cap was 128 and the epilogue's pointers lived in local
// memory: every phase began with a dozen dependent LDLs that took microseconds under the store stream)
constexpr int EPI_WARP0 = 4, MMA_WARP = 8, TMA_WARP = 9, XLOAD_WARP = 10, NTHREADS = 12 * 32;
constexpr int N_LO = 112, N_HI = DPAD - N_LO;       // 96
constexpr int COL_S = 0, COL_P = 2 * TY, COL_LO = COL_P + TY, COL_HI = COL_LO + 2 * N_LO;
static_assert(COL_HI + N_HI == TMEM_COLS, "TMEM budget");
constexpr int ITEM_SLOTS = 4;
constexpr int N_CONSUMERS = NSOFT + NEPI + 2;       // warps that read an item slot (the scheduler keeps its own copy)
constexpr float TAU2 = 11.0f;
constexpr float NEG2 = kNegFill * LOG2E;

enum Kind { PQ = 0, PA = 1, PB = 2, DONE = 3 };

struct PassArgs {
  const __nv_bfloat16* s_pack;       // Y side: S operand
  const __nv_bfloat16* v_pack;       // Y side: value operand (may equal s_pack)
  const unsigned long long* y_words; // (B, LYP/64, 2)
  int LX, LXP, LY, LYP;
};

struct Args {
  PassArgs p[3];
  const __nv_bfloat16* x_pack[3];    // X side S operand per kind (PB: unused, the tile of pass A stays)
  const __nv_bfloat16* c_pack;       // plain bf16 text pack: the c of c * a, c * b
  float* out;                        // (B, Lc, 4d)
  float* q2c;                        // (B, Lq, d) fp32 T or null
  float* bm;                         // (B, Lc, d) or null
  __nv_bfloat16* t_pack;             // packed T
  float* lse_row;                    // (B, Lc) or null
  float* lse_col;                    // (B, Lq) or null
  const float* bias;
  int* ready;                        // (B) Q2C -> pass B counters, zeroed before the launch
  int* queue;                        // work queue head, zeroed before the launch
  int nq, nc, n_q2c, n_c2q, d;
  long long* trace;                  // debugging aid: 8 x int64 per pass (queue order), or null
  long long* ev;                     // debugging aid: event log of CTA 0, 4 roles x 1024 x (code, clock64), or null
  int dbg;                           // debugging aid (MMB_TC5_DEBUG): 1 no c loads, 2 no stores of out / T
};

struct EvLog {                       // lane 0 of one warp of CTA 0 appends (code, clock64)
  long long* p;
  int n;
  __device__ __forceinline__ void operator()(int code) {
    if (p && n < 1024) {
      p[2 * n] = code;
      p[2 * n + 1] = clock64();
      ++n;
    }
  }
};

// (A back-off variant of mbar_wait -- __nanosleep between polls for the waits that are expected to be long -- was measured: it does not
// free anything the working warps need, and the coarser wake-up costs ~1.5 us per forward; every wait polls.)
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16_u32(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                             uint32_t acc, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "setp.ne.b32 q, %6, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void st_cs_f4(float* p, const float4 v) {      // streaming store: the output is not re-read here
  asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ int4 ld_item(const int4* p) {                   // (ordered by the acquire of the barrier wait before it)
  int4 v;
  asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void signal_release(int* counter) {
  asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(counter) : "memory");
}

constexpr int NBARS = 2 * ITEM_SLOTS + 2 + 2 * NSLOT + 4 * 2 + 2 + 2 + 1 + 2 + 2;
constexpr size_t SMEM_BYTES = (size_t)X_BYTES + NSLOT * SLOT_BYTES + STG_BYTES + 2 * TX * 4 + ITEM_SLOTS * 16 + NBARS * 8 + 16;
static_assert(SMEM_BYTES <= 227 * 1024, "one CTA per SM");

// ---------------------------------------------------------------------------------------------------------------------------------
// Drain.  Everything below is written for CODE SIZE: the first version instantiated the write-out per kind and phase with every
// loop unrolled (11 200 SASS instructions in the kernel, 179 KB against a 32 KB L1.5 / 6 KB L0 instruction cache) and an epilogue
// warp spent 2 500 cycles in a write-out that had all its loads and stores switched off.
// ---------------------------------------------------------------------------------------------------------------------------------

// Fill the stage with columns [16 * ch0, 16 * (ch0 + nch)) of this thread's accumulator row, scaled by 1 / l.
__device__ __noinline__ void stage_fill(float* stg_row, const uint32_t acc, const int ch0, const int nch, const float inv_l) {
#pragma unroll 1
  for (int c = 0; c < nch; ++c) {
    uint32_t raw[16];
    tmem_ld16_nowait(acc + (ch0 + c) * 16, raw);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; i += 4)
      *reinterpret_cast<float4*>(stg_row + (ch0 + c) * 16 + i) =
          make_float4(__uint_as_float(raw[i]) * inv_l, __uint_as_float(raw[i + 1]) * inv_l, __uint_as_float(raw[i + 2]) * inv_l,
                      __uint_as_float(raw[i + 3]) * inv_l);
  }
}

// One phase of the write-out for one epilogue warp: rows e, e + 8, ... (cnt of them, at most 16) of the staged block, this lane's
// four columns.  Pointers advance by eight rows per step (no per-row index arithmetic: the first version spent ~50 instructions
// per row, and a warp that executes a dependent instruction stream alone retires one instruction every 4 - 6 cycles).
//   PA: pa = out block 1 (a, streaming), pb = out block 2 (c * a)      PB: pa = bm or null, pb = out block 3 (c * b)
//   PQ: pa = fp32 T or null, pb = null
// c comes from the plain bf16 text pack (core-matrix order; 8 bytes per lane and row instead of 16, so that two rounds of 16 rows fit
// in registers next to each other): row e + 4 j of the block, columns col0 + 4 * lane -> group j / 2, row-in-group e + 4 (j & 1).
// ONE copy of this code serves all three pass kinds (pa / pb may be null): the epilogue is executed once per pass, and straight-line
// code that is executed once misses the instruction cache line by line (L1.5: 32 KB, the kernel: ~90 KB) -- with the write-out
// instantiated per kind an epilogue warp took 2 000 cycles for a phase that had all its loads and stores switched off.
__device__ __forceinline__ void load_c16(uint2* cv, const char* c, const int cnt) {
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    cv[j] = make_uint2(0u, 0u);
    if (j < cnt) cv[j] = __ldg(reinterpret_cast<const uint2*>(c + (j >> 1) * GROUP_BYTES + (j & 1) * 64));
  }
}
__device__ __forceinline__ float4 bf16x4_to_float4(const uint2 v) {
  return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16),
                     __uint_as_float(v.y & 0xffff0000u));
}
__device__ __forceinline__ void st_f4_if(float* p, const float4 v, const uint32_t plain, const uint32_t streaming) {
  asm volatile(
      "{\n\t"
      ".reg .pred a, b;\n\t"
      "setp.ne.u32 a, %5, 0;\n\t"
      "setp.ne.u32 b, %6, 0;\n\t"
      "@a st.global.v4.f32 [%0], {%1, %2, %3, %4};\n\t"
      "@b st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};\n\t"
      "}" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(plain), "r"(streaming)
      : "memory");
}
//   PA: pa = out block 1 (a, streaming), pb = out block 2 (c * a)      PB: pa = bm or null (plain), pb = out block 3 (c * b)
//   PQ: pa = fp32 T or null (plain), pb = null
__device__ __forceinline__ void store16(const uint2* cv, const float* sp, float* pa, float* pb, const uint32_t a8, const uint32_t b8,
                                        const int cnt, const uint32_t a_plain, const uint32_t a_cs, const uint32_t b_on) {
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    if (j < cnt) {
      const float4 o = *reinterpret_cast<const float4*>(sp + j * (NEPI * STG_STRIDE));
      st_f4_if(pa, o, a_plain, a_cs);
      const float4 c = bf16x4_to_float4(cv[j]);
      st_f4_if(pb, make_float4(c.x * o.x, c.y * o.y, c.z * o.z, c.w * o.w), 0u, b_on);
    }
    pa += a8;
    pb += b8;
  }
}

// Packed bf16 T (value operand of pass B, and of the backward pass) from the staged columns [col0, col0 + ncols): lane = (row % 8,
// chunk % 4); eight lanes write one 128-byte core matrix.  Rows past LX and columns past d are written as zeros (operand padding).
__device__ __noinline__ void write_t_pack(char* tp_block, const float* stg, const int e, const int lane, const int col0, const int ncols,
                                          const int rows, const int d) {
  const int r8 = lane & 7, cq = lane >> 3;
  const int nch = ncols / 8, chunk0 = col0 / 8;
#pragma unroll 1
  for (int rg = e; rg < TX / 8; rg += NEPI) {
    const int row = rg * 8 + r8;
    char* dst = tp_block + (size_t)rg * GROUP_BYTES + r8 * 16;
    const float* src = stg + row * STG_STRIDE;
#pragma unroll 1
    for (int ch = cq; ch < nch; ch += 4) {
      const float4 lo = *reinterpret_cast<const float4*>(src + ch * 8), hi = *reinterpret_cast<const float4*>(src + ch * 8 + 4);
      const bool ok = row < rows && (chunk0 + ch) * 8 < d;          // d % 8 == 0
      __nv_bfloat162 h[4];
      h[0] = __floats2bfloat162_rn(ok ? lo.x : 0.f, ok ? lo.y : 0.f);
      h[1] = __floats2bfloat162_rn(ok ? lo.z : 0.f, ok ? lo.w : 0.f);
      h[2] = __floats2bfloat162_rn(ok ? hi.x : 0.f, ok ? hi.y : 0.f);
      h[3] = __floats2bfloat162_rn(ok ? hi.z : 0.f, ok ? hi.w : 0.f);
      *reinterpret_cast<uint4*>(dst + (chunk0 + ch) * 128) = *reinterpret_cast<uint4*>(h);
    }
  }
}

__global__ void __launch_bounds__(NTHREADS, 1) bidaf_tc5_kernel(const Args f) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* const sX = smem_raw;
  unsigned char* const sY = sX + X_BYTES;
  float* const sStage = reinterpret_cast<float*>(sY + NSLOT * SLOT_BYTES);
  float* const sStat = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(sStage) + STG_BYTES);    // [2][TX] row sums
  int4* const sItems = reinterpret_cast<int4*>(sStat + 2 * TX);
  uint64_t* const sBars = reinterpret_cast<uint64_t*>(sItems + ITEM_SLOTS);
  uint32_t* const sTmem = reinterpret_cast<uint32_t*>(sBars + NBARS);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp_u = uniform_warp_idx();
  const uint32_t leader = elect_one();

  const uint32_t b0 = smem_u32(sBars);
  const uint32_t item_full0 = b0, item_empty0 = item_full0 + 8 * ITEM_SLOTS;
  const uint32_t x_full = item_empty0 + 8 * ITEM_SLOTS, x_free = x_full + 8;
  const uint32_t slot_full0 = x_free + 8, slot_free0 = slot_full0 + 8 * NSLOT;
  const uint32_t s_full0 = slot_free0 + 8 * NSLOT, s_free0 = s_full0 + 16;
  const uint32_t p_full0 = s_free0 + 16, p_free0 = p_full0 + 16;
  const uint32_t o_full0 = p_free0 + 16, lo_free0 = o_full0 + 16, hi_free = lo_free0 + 16;
  const uint32_t st_full0 = hi_free + 8, st_free0 = st_full0 + 16;

  if (tid == 0) {
    for (int i = 0; i < ITEM_SLOTS; ++i) {
      mbar_init(item_full0 + 8 * i, 1);
      mbar_init(item_empty0 + 8 * i, N_CONSUMERS);
    }
    mbar_init(x_full, 1);
    mbar_init(x_free, 1);
    for (int i = 0; i < NSLOT; ++i) {
      mbar_init(slot_full0 + 8 * i, 1);
      mbar_init(slot_free0 + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(s_full0 + 8 * i, 1);
      mbar_init(s_free0 + 8 * i, NSOFT);
      mbar_init(p_full0 + 8 * i, NSOFT);
      mbar_init(p_free0 + 8 * i, 1);
      mbar_init(o_full0 + 8 * i, 1);
      mbar_init(lo_free0 + 8 * i, 1);
      mbar_init(st_full0 + 8 * i, NSOFT);
      mbar_init(st_free0 + 8 * i, NEPI);
    }
    mbar_init(hi_free, 1);
    fence_barrier_init();
  }
  if (warp_u == 0) tmem_alloc(smem_u32(sTmem), TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(sTmem);
  const int n_items = f.n_q2c + 2 * f.n_c2q;

  if (warp_u == TMA_WARP) {
    // =========================================== scheduler + TMA producer ===========================================
    // Programmatic dependent launch: this grid may have started while bidaf_pack_kernel was still running (its CTAs are placed as
    // SMs free up and get here through their prologue); nothing of the pack kernel's output -- the operand packs, the mask words, the
    // zeroed queue head and dependency counters -- is touched before this wait, and every other role starts from an item published below.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    uint32_t g = 0;                                                 // slots used so far (ring position)
    EvLog ev{(f.ev && blockIdx.x == 0 && lane == 0) ? f.ev + 2 * 2048 : nullptr, 0};
    for (uint32_t n = 0;; ++n) {                                    // n: passes published so far
      int item = 0;
      if (leader) item = atomicAdd(f.queue, 1);
      item = __shfl_sync(0xffffffffu, item, __ffs(__ballot_sync(0xffffffffu, leader)) - 1);
      int kind = DONE, b = 0, xblk = 0, nty = 0, canon = 0;         // canon: kind-major pass number (trace index)
      if (item < n_items) {
        // Queue order: Q2C and pass-A items interleaved in proportion (neither depends on anything, and only the A items write
        // `out`: the store stream starts with the kernel), then the pass-B items.
        const int n1 = f.n_q2c + f.n_c2q;
        if (item < n1) {
          const int qb = (int)((long long)item * f.n_q2c / n1), qa = (int)((long long)(item + 1) * f.n_q2c / n1);
          if (qa > qb) { kind = PQ; b = qb / f.nq; xblk = qb - b * f.nq; canon = qb; }
          else { kind = PA; const int i = item - qb; b = i / f.nc; xblk = i - b * f.nc; canon = f.n_q2c + i; }
        } else {
          kind = PB;
          const int i = item - n1;
          b = i / f.nc;
          xblk = i - b * f.nc;
          canon = item;
        }
        const PassArgs& a = f.p[kind];
        // tiles past the last un-masked Y row contribute exp(-1e30 - m) = 0 to every soft-max: stop there.  (If nothing at
        // all is un-masked the soft-max is uniform over the whole range, attention.py:94, and every tile is needed.)
        nty = (a.LY + TY - 1) / TY;
        int last = 0;
        for (int w = lane; w < nty; w += 32)
          if (a.y_words[((size_t)b * (a.LYP / 64) + w) * 2 + 1] != 0ull) last = w + 1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
        if (last > 0) nty = min(nty, last);
      }
      const int slot = n & (ITEM_SLOTS - 1);
      mbar_wait(item_empty0 + 8 * slot, ((n / ITEM_SLOTS) & 1) ^ 1);
      if (lane == 0) {
        sItems[slot] = make_int4(kind, b, xblk, nty);
        if (f.trace && kind != DONE) {
          long long* tr = f.trace + (size_t)canon * 8;
          tr[0] = globaltimer_ns();
          tr[3] = kind;
          tr[5] = nty;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(item_full0 + 8 * slot);            // release semantics: the slot contents are visible
      ev(kind);
      if (kind == DONE) break;
      const PassArgs& a = f.p[kind];
      const size_t y_batch = (size_t)b * (a.LYP / 8) * GROUP_BYTES;
      if (kind == PB) {                                             // the value operand is T: wait for this batch row's Q2C items
        wait_counter(f.ready + b, f.nq * NEPI);
        fence_proxy_async_all();                                    // their generic-proxy stores -> our async-proxy (TMA) loads
      }
      const bool same_v = a.v_pack == a.s_pack;
#pragma unroll 1
      for (int t = 0; t < nty; ++t) {
        const size_t off = y_batch + (size_t)t * SLOT_BYTES;
#pragma unroll 1
        for (int part = 0; part < (same_v ? 1 : 2); ++part, ++g) {
          const int s = g % NSLOT;
          mbar_wait(slot_free0 + 8 * s, ((g / NSLOT) & 1) ^ 1);
          if (part == 0) ev(100 + t);
          mbar_expect_tx(slot_full0 + 8 * s, SLOT_BYTES, leader);
          tma_bulk_g2s(smem_u32(sY + s * SLOT_BYTES), reinterpret_cast<const char*>(part == 0 ? a.s_pack : a.v_pack) + off, SLOT_BYTES,
                       slot_full0 + 8 * s, leader);
        }
      }
    }
  } else if (warp_u == MMA_WARP) {
    // ================================================= MMA issuer ==================================================
    constexpr uint32_t IDESC_S = idesc_bf16(TY, 0), IDESC_LO = idesc_bf16(N_LO, 1), IDESC_HI = idesc_bf16(N_HI, 1);
    uint32_t g = 0;                                                 // slots consumed so far
    uint32_t gt = 0;                                                // tiles so far (S / P buffer position)
    uint32_t nx = 0;                                                // X tiles so far
    const uint32_t xs_lo = desc_lo(smem_u32(sX), 128);
    EvLog ev{(f.ev && blockIdx.x == 0 && lane == 0) ? f.ev : nullptr, 0};
    for (uint32_t n = 0;; ++n) {
      const int slot = n & (ITEM_SLOTS - 1);
      mbar_wait(item_full0 + 8 * slot, (n / ITEM_SLOTS) & 1);
      const int4 it = ld_item(sItems + slot);
      __syncwarp();
      if (lane == 0) mbar_arrive(item_empty0 + 8 * slot);
      const int kind = it.x, nty = it.w;
      if (kind == DONE) break;
      const bool same_v = f.p[kind].v_pack == f.p[kind].s_pack;
      const uint32_t per = same_v ? 1u : 2u;
      const int ob = n & 1;
      ev(kind);
      mbar_wait(x_full, nx & 1);
      ++nx;
      ev(10);
      tc_fence_after();
      if (f.trace && lane == 0)
        f.trace[(size_t)(kind == PQ ? it.y * f.nq + it.z : f.n_q2c + f.n_c2q * (kind == PB ? 1 : 0) + it.y * f.nc + it.z) * 8 + 7] = globaltimer_ns();
      auto issue_s = [&](int t) {                                   // S(t) = X Y_t^T into S buffer (gt + t) & 1
        const uint32_t gg = g + per * t, tt = gt + t;
        const int s = gg % NSLOT, sb = tt & 1;
        mbar_wait(slot_full0 + 8 * s, (gg / NSLOT) & 1);
        ev(200 + t);
        mbar_wait(s_free0 + 8 * sb, ((tt >> 1) & 1) ^ 1);
        ev(300 + t);
        tc_fence_after();
        const uint32_t y_lo = desc_lo(smem_u32(sY + s * SLOT_BYTES), 128);
#pragma unroll
        for (int k = 0; k < DPAD / 16; ++k)
          umma_bf16_lh(tmem + COL_S + sb * TY, xs_lo + k * 16, desc_hi(GROUP_BYTES), y_lo + k * 16, desc_hi(GROUP_BYTES), IDESC_S,
                       k > 0, leader);
        umma_commit(s_full0 + 8 * sb, leader);
        if (!same_v) umma_commit(slot_free0 + 8 * s, leader);       // the S operand's slot is dead; the value operand has its own
        if (t == nty - 1) umma_commit(x_free, leader);             // the X tile is dead after the pass's last S product
      };
      int s_issued = 0;
      for (int t = 0; t < nty; ++t) {
        while (s_issued < nty && s_issued < t + 2) issue_s(s_issued++);
        const uint32_t gg = g + per * t + (per - 1), tt = gt + t;
        const int s = gg % NSLOT, pb = tt & 1;
        if (t == 0) {                                               // the accumulators this pass writes have been drained
          mbar_wait(lo_free0 + 8 * ob, ((n >> 1) & 1) ^ 1);
          mbar_wait(hi_free, (n & 1) ^ 1);
        }
        if (!same_v) mbar_wait(slot_full0 + 8 * s, (gg / NSLOT) & 1);
        mbar_wait(p_full0 + 8 * pb, (tt >> 1) & 1);
        ev(400 + t);
        tc_fence_after();
        const uint32_t v_lo = desc_lo(smem_u32(sY + s * SLOT_BYTES), GROUP_BYTES);
        const uint32_t p_addr = tmem + COL_P + pb * (TY / 2);
#pragma unroll
        for (int k = 0; k < TY / 16; ++k) {                         // O += P V (A = P from TMEM; V MN-major: LBO = group stride)
          const uint32_t acc = (t > 0) || (k > 0);
          umma_bf16_ts(tmem + COL_LO + ob * N_LO, p_addr + k * 8, v_lo + k * (2 * GROUP_BYTES / 16), desc_hi(128), IDESC_LO, acc, leader);
          umma_bf16_ts(tmem + COL_HI, p_addr + k * 8, v_lo + k * (2 * GROUP_BYTES / 16) + (N_LO / 8) * (128 / 16), desc_hi(128), IDESC_HI,
                       acc, leader);
        }
        umma_commit(slot_free0 + 8 * s, leader);
        umma_commit(p_free0 + 8 * pb, leader);
        if (t == nty - 1) umma_commit(o_full0 + 8 * ob, leader);
      }
      g += per * nty;
      gt += nty;
    }
  } else if (warp_u == XLOAD_WARP) {
    // ================================================== X loader ===================================================
    uint32_t nx = 0;
    for (uint32_t n = 0;; ++n) {
      const int slot = n & (ITEM_SLOTS - 1);
      mbar_wait(item_full0 + 8 * slot, (n / ITEM_SLOTS) & 1);
      const int4 it = ld_item(sItems + slot);
      __syncwarp();
      if (lane == 0) mbar_arrive(item_empty0 + 8 * slot);
      if (it.x == DONE) break;
      const PassArgs& a = f.p[it.x];
      const size_t x_off = ((size_t)it.y * (a.LXP / 8) + (size_t)it.z * (TX / 8)) * GROUP_BYTES;
      mbar_wait(x_free, (nx & 1) ^ 1);                              // the previous item's last S product has read the tile
      ++nx;
      mbar_expect_tx(x_full, X_BYTES, leader);
      tma_bulk_g2s(smem_u32(sX), reinterpret_cast<const char*>(f.x_pack[it.x]) + x_off, X_BYTES, x_full, leader);
    }
  } else if (warp_u < NSOFT) {
    // ================================================ soft-max warps ================================================
    const int row = warp_u * 32 + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(warp_u * 32) << 16);
    const float bias2 = f.bias[0] * LOG2E;
    uint32_t gt = 0;
    EvLog ev{(f.ev && blockIdx.x == 0 && tid == 0) ? f.ev + 2048 : nullptr, 0};
    for (uint32_t n = 0;; ++n) {
      const int slot = n & (ITEM_SLOTS - 1);
      mbar_wait(item_full0 + 8 * slot, (n / ITEM_SLOTS) & 1);
      const int4 it = ld_item(sItems + slot);
      __syncwarp();
      if (lane == 0) mbar_arrive(item_empty0 + 8 * slot);
      const int kind = it.x, b = it.y, xblk = it.z, nty = it.w;
      if (kind == DONE) break;
      const PassArgs& a = f.p[kind];
      const int ob = n & 1;
      const unsigned long long* words_b = a.y_words + (size_t)b * (a.LYP / 64) * 2;
      float m_ref = -INFINITY, l_run = 0.f;                         // log2 domain
      ulonglong2 words = *reinterpret_cast<const ulonglong2*>(words_b);
#pragma unroll 1
      for (int t = 0; t < nty; ++t, ++gt) {
        const int sb = gt & 1;
        const uint32_t sk = (gt >> 1) & 1;                          // parity of this use of S / P buffer sb
        const unsigned long long wvalid = words.x, wopen = words.y;
        const bool all_open = (wvalid & wopen) == ~0ull;
        if (t + 1 < nty) words = *reinterpret_cast<const ulonglong2*>(words_b + (size_t)(t + 1) * 2);   // next tile's masks
        mbar_wait(s_full0 + 8 * sb, sk);
        ev(200 + t);
        tc_fence_after();
        const uint32_t s_addr = lane_base + COL_S + sb * TY;
        // pass 1 over the tile (two halves of 32 columns; small loop bodies -- see the note on code size above): the maximum
        float tile_max = -INFINITY;
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          uint32_t raw[32];
          tmem_ld16_nowait(s_addr + h * 32, raw);
          tmem_ld16_nowait(s_addr + h * 32 + 16, raw + 16);
          tmem_wait_ld();
          float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
          if (all_open) {
#pragma unroll
            for (int c = 0; c < 32; ++c) mx[c & 3] = fmaxf(mx[c & 3], __uint_as_float(raw[c]));
          } else {
            const uint32_t wv = (uint32_t)(wvalid >> (32 * h)), wo = (uint32_t)(wopen >> (32 * h));
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              const float v = ((wo >> c) & 1u) ? fmaf(__uint_as_float(raw[c]), LOG2E, bias2) : NEG2;     // attention.py:94
              if ((wv >> c) & 1u) mx[c & 3] = fmaxf(mx[c & 3], v);
            }
          }
          tile_max = fmaxf(tile_max, fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])));
        }
        if (all_open) tile_max = fmaf(tile_max, LOG2E, bias2);      // log2 domain (monotone: the maximum commutes with it)
        float alpha = 1.f;
        const bool bump = tile_max > m_ref + TAU2;                  // first tile: m_ref = -inf -> always
        if (bump) {
          alpha = fast_exp2(m_ref - tile_max);                      // 0 on the first tile
          m_ref = tile_max;
        }
        const float shift = bias2 - m_ref;
        ev(400 + t);
        mbar_wait(p_free0 + 8 * sb, sk ^ 1);                        // P V(t - 2) has read this P buffer
        ev(500 + t);
        tc_fence_after();
        // pass 2: P = 2^(s log2 e + bias2 - m_ref) as packed bf16 into TMEM, and its row sum
        float psum = 0.f;
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          uint32_t raw[32];
          tmem_ld16_nowait(s_addr + h * 32, raw);
          tmem_ld16_nowait(s_addr + h * 32 + 16, raw + 16);
          tmem_wait_ld();
          if (h == 1) {                                             // S(t + 2) may overwrite the buffer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(s_free0 + 8 * sb);
          }
          uint32_t packed[16];
          float ps[2] = {0.f, 0.f};
          if (all_open) {
#pragma unroll
            for (int c = 0; c < 32; c += 2) {
              const float p0 = fast_exp2(fmaf(__uint_as_float(raw[c]), LOG2E, shift));
              const float p1 = fast_exp2(fmaf(__uint_as_float(raw[c + 1]), LOG2E, shift));
              ps[0] += p0;
              ps[1] += p1;
              const __nv_bfloat162 pk = __floats2bfloat162_rn(p0, p1);
              packed[c / 2] = *reinterpret_cast<const uint32_t*>(&pk);
            }
          } else {
            const uint32_t wv = (uint32_t)(wvalid >> (32 * h)), wo = (uint32_t)(wopen >> (32 * h));
#pragma unroll
            for (int c = 0; c < 32; c += 2) {
              // a masked logit is the literal -1e30 (log2 domain: NEG2); NEG2 - m_ref is exactly 0 when everything is masked
              const float s0 = ((wo >> c) & 1u) ? fmaf(__uint_as_float(raw[c]), LOG2E, bias2) : NEG2;
              const float s1 = ((wo >> (c + 1)) & 1u) ? fmaf(__uint_as_float(raw[c + 1]), LOG2E, bias2) : NEG2;
              const float p0 = ((wv >> c) & 1u) ? fast_exp2(s0 - m_ref) : 0.f;
              const float p1 = ((wv >> (c + 1)) & 1u) ? fast_exp2(s1 - m_ref) : 0.f;
              ps[0] += p0;
              ps[1] += p1;
              const __nv_bfloat162 pk = __floats2bfloat162_rn(p0, p1);
              packed[c / 2] = *reinterpret_cast<const uint32_t*>(&pk);
            }
          }
          psum += ps[0] + ps[1];
          tmem_st16_u32(lane_base + COL_P + sb * (TY / 2) + h * 16, packed);
        }
        l_run = l_run * alpha + psum;
        if (__any_sync(0xffffffffu, bump && t > 0)) {               // lazy rescale of this warp's rows (alpha = 1 where no bump)
          mbar_wait(p_free0 + 8 * (sb ^ 1), ((gt - 1) >> 1) & 1);   // P V(t - 1) has landed in the accumulators
          tc_fence_after();
#pragma unroll 1
          for (int q = 0; q < DPAD / 16; ++q) {
            const uint32_t addr = lane_base + (q < N_LO / 16 ? COL_LO + ob * N_LO + q * 16 : COL_HI + (q - N_LO / 16) * 16);
            float o[16];
            tmem_ld16(addr, o);
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] *= alpha;
            tmem_st16(addr, o);
          }
        }
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full0 + 8 * sb);
        ev(600 + t);
      }
      // row statistics -> epilogue warps; log-sum-exp of the row (natural log) for the backward pass
      mbar_wait(st_free0 + 8 * ob, ((n >> 1) & 1) ^ 1);
      sStat[ob * TX + row] = l_run;
      __syncwarp();
      if (lane == 0) mbar_arrive(st_full0 + 8 * ob);
      float* lse = kind == PQ ? f.lse_col : (kind == PA ? f.lse_row : nullptr);
      if (lse && xblk * TX + row < a.LX) lse[(size_t)b * a.LX + xblk * TX + row] = (m_ref + log2f(l_run)) * LN2;
    }
  } else if (warp_u < EPI_WARP0 + NEPI) {
    // ================================================ epilogue warps ================================================
    const int e = warp_u - EPI_WARP0, q4 = e & 3;
    const uint32_t lane_base = tmem + ((uint32_t)(q4 * 32) << 16);
    float* const stg_row = sStage + (q4 * 32 + lane) * STG_STRIDE;
    EvLog ev{(f.ev && blockIdx.x == 0 && e == (f.dbg >> 8) && lane == 0) ? f.ev + 3 * 2048 : nullptr, 0};
    for (uint32_t n = 0;; ++n) {
      const int slot = n & (ITEM_SLOTS - 1);
      mbar_wait(item_full0 + 8 * slot, (n / ITEM_SLOTS) & 1);
      const int4 it = ld_item(sItems + slot);
      __syncwarp();
      if (lane == 0) mbar_arrive(item_empty0 + 8 * slot);
      const int kind = it.x, b = it.y, xblk = it.z;
      if (kind == DONE) break;
      ev(20 + kind);
      const int ob = n & 1;
      const uint32_t par = (n >> 1) & 1;
      const int x0 = xblk * TX, LX = f.p[kind].LX, d = f.d;
      const size_t row0 = (size_t)b * LX + x0;
      const int rows = min(TX, LX - x0);                           // valid rows of this block
      const int cnt = rows > e ? (rows - e + NEPI - 1) / NEPI : 0;  // ... of which this warp writes rows e, e + 4, ... (<= 32)
      const int cnt0 = min(cnt, 16), cnt1 = max(cnt - 16, 0);       // two rounds of 16 rows
      const uint32_t d8 = NEPI * d;                                 // row step of this warp, in floats of a d-wide tensor
      // this lane's c: chunk (col0 + 4 * lane) / 8, half (lane & 1), rows e + 4 j (col0 is a multiple of 8)
      const char* c_row = reinterpret_cast<const char*>(f.c_pack) + ((size_t)b * (f.p[PA].LXP / 8) + (size_t)(x0 / 8)) * GROUP_BYTES + e * 16 +
                          (lane >> 1) * 128 + (lane & 1) * 8;
      float* const pa_base = kind == PA ? f.out + d : (kind == PB ? f.bm : f.q2c);
      // null outputs: the pointers stay valid addresses (never dereferenced: the stores are predicated off)
      float* pa_row = (pa_base ? pa_base : f.out) + (row0 + e) * (kind == PA ? 4 * d : d) + 4 * lane;
      float* pb_row = f.out + (row0 + e) * 4 * d + (kind == PA ? 2 : 3) * d + 4 * lane;
      const uint32_t a8 = kind == PA ? 4 * d8 : d8, b8 = 4 * d8;
      const bool dbg_st = (f.dbg & 2) != 0;
      const uint32_t a_plain = (kind != PA && pa_base && !dbg_st) ? 1u : 0u, a_cs = (kind == PA && !dbg_st) ? 1u : 0u;
      const uint32_t b_on = (kind != PQ && !dbg_st) ? 1u : 0u;
      char* const tp_block = reinterpret_cast<char*>(f.t_pack) + ((size_t)b * (f.p[PQ].LXP / 8) + (size_t)(x0 / 8)) * GROUP_BYTES;
      const int n4_hi = max(0, min(N_HI, d - N_LO)) >> 2, n4_lo = min(N_LO, d) >> 2;   // float4s per row in each phase
      const float* const sp = sStage + e * STG_STRIDE + 4 * lane;
      const bool ld_hi = lane < n4_hi && kind != PQ && !(f.dbg & 1), ld_lo = lane < n4_lo && kind != PQ && !(f.dbg & 1);
      uint2 cva[16], cvb[16];
      load_c16(cva, c_row + (N_LO / 8) * 128, ld_hi ? cnt0 : 0);    // in flight while the tile loop of this pass still runs
      mbar_wait(st_full0 + 8 * ob, par);
      const float inv_l = 1.f / sStat[ob * TX + q4 * 32 + lane];
      __syncwarp();
      if (lane == 0) mbar_arrive(st_free0 + 8 * ob);
      mbar_wait(o_full0 + 8 * ob, par);
      tc_fence_after();
      long long t_acc = 0;
      if (f.trace && e == 0 && lane == 0) t_acc = globaltimer_ns();
      ev(31);
#pragma unroll 1
      for (int phase = 0; phase < 2; ++phase) {                     // HI (columns 112..207, single buffered) first, then LO
        const int col0 = phase == 0 ? N_LO : 0, ncols = phase == 0 ? N_HI : N_LO, n4 = phase == 0 ? n4_hi : n4_lo;
        if (!(f.dbg & 8)) stage_fill(stg_row, lane_base + (phase == 0 ? COL_HI : COL_LO + ob * N_LO), 0, ncols / 16, inv_l);
        tc_fence_before();
        named_bar_sync(1, NEPI * 32);
        if (e == 0 && lane == 0) mbar_arrive(phase == 0 ? hi_free : lo_free0 + 8 * ob);
        ev(33 + 4 * phase);
        const bool st = lane < n4, ld = phase == 0 ? ld_hi : ld_lo;
        const int w0 = st ? cnt0 : 0, w1 = st ? cnt1 : 0;           // rows this lane stores in each round
        load_c16(cvb, c_row + (col0 / 8) * 128 + 8 * GROUP_BYTES, ld ? cnt1 : 0);
        if (kind == PQ && !(f.dbg & 8)) write_t_pack(tp_block, sStage, e, lane, col0, ncols, rows, d);
        store16(cva, sp, pa_row + col0, pb_row + col0, a8, b8, w0, a_plain, a_cs, b_on);
        if (phase == 0) load_c16(cva, c_row, ld_lo ? cnt0 : 0);     // LO, round 0: in flight over the barrier and the fill
        store16(cvb, sp + 16 * NEPI * STG_STRIDE, pa_row + col0 + 16 * a8, pb_row + col0 + 16 * b8, a8, b8, w1, a_plain, a_cs, b_on);
        ev(34 + 4 * phase);
        named_bar_sync(1, NEPI * 32);                               // the stage may be refilled
      }
      if (kind == PQ) {                                             // this warp's part of the T rows is in memory: one count per warp
        __syncwarp();
        if (lane == 0) signal_release(f.ready + b);
      }
      if (f.trace && e == 0 && lane == 0) {
        long long* tr = f.trace + (size_t)(kind == PQ ? b * f.nq + xblk : f.n_q2c + f.n_c2q * (kind == PB ? 1 : 0) + b * f.nc + xblk) * 8;
        tr[1] = t_acc;
        tr[2] = globaltimer_ns();
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        tr[4] = smid;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp_u == 0) tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace

// After bidaf_pack_kernel: one launch for all Q2C and C2Q items.  `text` is the fp32 text input (B, Lc, d); q2c, bm, lse_row and
// lse_col may be null (inference: T is kept only in its packed bf16 form).
int bidaf_fwd_tc5_launch(const BidafPacks& pk, const float* text, const float* bias, float* out, float* q2c, float* bm,
                         float* lse_row, float* lse_col, int B, int Lc, int Lq, int d, cudaStream_t stream) {
  static_assert(PACK_ROWS == TX, "pack padding must match the X tile");
  const int LcP = pk.LcP, LqP = pk.LqP;
  Args f{};
  f.p[PQ] = PassArgs{pk.cw, pk.cp, pk.c_words, Lq, LqP, Lc, LcP};
  f.p[PA] = PassArgs{pk.qs, pk.qp, pk.q_words, Lc, LcP, Lq, LqP};
  f.p[PB] = PassArgs{pk.qs, pk.tp, pk.q_words, Lc, LcP, Lq, LqP};
  f.x_pack[PQ] = pk.qs;
  f.x_pack[PA] = pk.cw;
  f.x_pack[PB] = pk.cw;
  f.c_pack = pk.cp;
  (void)text;
  f.out = out;
  f.q2c = q2c;
  f.bm = bm;
  f.t_pack = pk.tp;
  f.lse_row = lse_row;
  f.lse_col = lse_col;
  f.bias = bias;
  f.ready = pk.ready;
  f.queue = pk.ready + B;
  f.nq = LqP / TX;
  f.nc = LcP / TX;
  f.n_q2c = B * f.nq;
  f.n_c2q = B * f.nc;
  f.d = d;
  static const char* trace_env = getenv("MMB_BIDAF_FWD_ITEM_TRACE");     // debugging aid (tools/bidaf_fwd_items.py)
  f.trace = trace_env ? reinterpret_cast<long long*>(strtoull(trace_env, nullptr, 0)) : nullptr;
  static const char* ev_env = getenv("MMB_BIDAF_FWD_EV_TRACE");          // debugging aid (tools/bidaf_fwd_events.py)
  f.ev = ev_env ? reinterpret_cast<long long*>(strtoull(ev_env, nullptr, 0)) : nullptr;
  static const char* dbg_env = getenv("MMB_TC5_DEBUG");
  f.dbg = dbg_env ? atoi(dbg_env) : 0;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    MMB_CUDA(cudaGetDevice(&dev));
    MMB_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    MMB_CUDA(cudaFuncSetAttribute(bidaf_tc5_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
  }
  // (pk.ready[0 .. B] -- the counters and the queue head -- are zeroed by bidaf_pack_kernel)
  const int n_items = f.n_q2c + 2 * f.n_c2q;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(n_items < num_sms ? n_items : num_sms));
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];                                           // programmatic dependent launch (griddepcontrol.wait)
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MMB_CUDA(cudaLaunchKernelEx(&cfg, bidaf_tc5_kernel, f));
  return check_launch("bidaf_tc5_kernel");
}

}  // namespace mmb
