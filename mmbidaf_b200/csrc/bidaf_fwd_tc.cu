// Fused BiDAF attention forward, tensor-core tier (sm_100a: tcgen05.mma + TMEM + TMA bulk copies).
// bf16 operands, fp32 accumulation / soft-max; rel <= 2e-2 tier of north_star.
//
// Same three streaming-soft-max contractions as the fp32 tier (bidaf_fwd_f32.cu), reorganised for the
// 5th-generation tensor cores.  Two launches:
//
//  1. bidaf_pack_kernel   converts c, q (optionally dropped) to bf16 ONCE, in the UMMA "core matrix" order
//       pack[b][row/8][chunk 0..25][row%8][8 x bf16]      (8 rows x 16 bytes = one 128-byte core matrix)
//     so that ANY tile of consecutive rows is one contiguous run of memory: a tile is fetched with a single
//     cp.async.bulk (TMA) that completes on an mbarrier and lands ready for tcgen05.mma -- no swizzle, no
//     register staging.  The same bytes serve as a K-major operand (S = X Y^T: LBO 128, SBO 3328) and as an
//     MN-major operand (O = P V: LBO 3328, SBO 128).  Chunk 25 is K padding (200 -> 208); it carries the
//     additive terms of the trilinear form split into bf16 hi/lo halves: text rows hold
//     [t_hi, t_lo, 1, 1, 0..] and modality rows [1, 1, m_hi, m_lo, 0..], so the GEMM itself adds
//     c~.w_c + q~.w_q to every logit.  w_cq is folded into the text-side S operand.  It also writes block 0 of
//     the output (the text itself) and zeroes the dependency counters and work-queue head of launch 2.
//  2. bidaf_tc5_kernel (bidaf_fwd_tc5.cu)   one persistent, warp-specialised CTA per SM runs the Q2C items
//     (T = softmax_i(S)^T c) and the C2Q items (a = softmax_j(S) q, b = softmax_j(S) T) and writes blocks 1 - 3.
#include "tc_common.cuh"

namespace mmb {
using namespace tc;
namespace {

// ---------------------------------------------------------------------------------------------------------
// 1. pack: fp32 (B, L, d) -> bf16 core-matrix order (+ folded weights, additive terms, mask words)
// ---------------------------------------------------------------------------------------------------------
struct PackArgs {
  const float* src;          // (B, L, d)
  const uint8_t* keep;       // (B, L, d) or null
  const uint8_t* mask;       // (B, L)
  const float* w_term;       // (d): c-side text_weight / q-side modality_weight
  const float* w_fold;       // (d) text_modality_weight for the text side, null for the modality side
  __nv_bfloat16* s_pack;     // S operand (dropped, folded, with term chunk)
  __nv_bfloat16* v_pack;     // plain values (value operand); may equal s_pack when identical (modality side, eval)
  unsigned long long* mask_words;   // (B, LP/64, 2): [valid bits, unmasked bits]
  float* out_copy;           // text side: block 0 of the output (B, L, 4d) <- the text itself (attention.py:52)
  float keep_scale;
  int L, LP, d, text_side;
};

struct PackPair { PackArgs side[2]; };

// (The inputs are read once and block 0 of the output is not re-read by this pass: evict-first loads and streaming stores leave L2 to the
// bf16 packs, which the main kernel streams several times.)
// 256-bit global accesses (sm_100): one instruction per lane and row instead of two 128-bit ones whose halves of every 32-byte
// sector arrived at L2 as separate requests (ncu: 2.3 M read sectors for 1.2 M sectors of input).
__device__ __forceinline__ void ldg256(const float* p, float* v) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
// two adjacent 16-byte pieces of a pack (rows r, r + 1 of one chunk) as ONE 32-byte store: a whole sector per request instead of two
// half sectors that L2 has to merge
__device__ __forceinline__ void stg256_u(void* p, const uint4 a, const uint4 b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x),
               "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void stg256(float* p, const float* v) {
  asm volatile("st.global.cs.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}

// A persistent grid of warps, each streaming over "units" of four consecutive rows of one side (lane = 16-byte chunk = 8 columns): the
// loads of the next unit are in flight while the current one is converted and stored.
// Rounds 1-2: one warp per 8-row group in small blocks (1 536 blocks of 128 threads in 1.7 waves, every block a serial
// load -> convert -> store chain behind a prologue of weight loads): two 128-bit loads per row and lane whose halves of every
// 32-byte sector arrived at L2 as separate requests, the converted group staged in shared memory; 25.7 - 31 us at config 2 for
// 99 MB of traffic.  Now: 256-bit loads / copies, the 16-byte pieces go straight to their place in the pack (a 128-byte core matrix
// is completed by eight rows handled by the same warp back to back, so L2 sees whole lines), no shared memory.
struct PackUnit {
  int side, b, row0;       // four rows row0 .. row0 + 3 of batch row b
};
__device__ __forceinline__ PackUnit pack_unit(const PackPair& pp, const int u, const int units0, const int per_b0, const int per_b1) {
  PackUnit r;
  r.side = u >= units0;
  const int v = r.side ? u - units0 : u, per_b = r.side ? per_b1 : per_b0;
  r.b = v / per_b;
  r.row0 = (v - r.b * per_b) * 4;
  return r;
}
__device__ __forceinline__ void pack_load4(const PackArgs& a, const PackUnit& un, const int lane, float (*v)[8], uint2* kraw) {
  const bool data_lane = lane < (a.d >> 3);
#pragma unroll
  for (int r = 0; r < 4; ++r) {                         // every global load of four rows is issued before any is used
#pragma unroll
    for (int e = 0; e < 8; ++e) v[r][e] = 0.f;
    kraw[r] = make_uint2(0u, 0u);
    const int row = un.row0 + r;
    if (row < a.L && data_lane) {
      const size_t off = ((size_t)un.b * a.L + row) * a.d + lane * 8;
      ldg256(a.src + off, v[r]);
      if (a.keep) kraw[r] = __ldg(reinterpret_cast<const uint2*>(a.keep + off));
    }
  }
}

__global__ void __launch_bounds__(128, 4) bidaf_pack_kernel(const PackPair pp, const int B, int* const zero_ints, const int n_zero) {
  // the main launch may be scheduled as soon as SMs free up (programmatic dependent launch; it waits for this grid before it reads)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (blockIdx.x == 0)                                  // dependency counters / work-queue head of the main launch
    for (int i = threadIdx.x; i < n_zero; i += blockDim.x) zero_ints[i] = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per_b0 = pp.side[0].LP / 4, per_b1 = pp.side[1].LP / 4;          // units per batch row (LP is a multiple of 128)
  const int units0 = B * per_b0, n_units = units0 + B * per_b1;
  const int n_warps = gridDim.x * 4;
  int u = blockIdx.x * 4 + warp;
  if (u >= n_units) return;
  // weights of both sides stay in registers (lane = chunk): 8 + 8 + 8 floats
  float wt0[8], wf0[8], wt1[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const bool in0 = lane < (pp.side[0].d >> 3), in1 = lane < (pp.side[1].d >> 3);
    wt0[e] = in0 ? pp.side[0].w_term[lane * 8 + e] : 0.f;
    wf0[e] = (in0 && pp.side[0].w_fold) ? pp.side[0].w_fold[lane * 8 + e] : 1.f;
    wt1[e] = in1 ? pp.side[1].w_term[lane * 8 + e] : 0.f;
  }
  const __nv_bfloat16 zero = __float2bfloat16_rn(0.f);
  float v[4][8], vn[4][8];
  uint2 kraw[4], kn[4];
  PackUnit un = pack_unit(pp, u, units0, per_b0, per_b1);
  pack_load4(pp.side[un.side], un, lane, v, kraw);
#pragma unroll 1
  for (;;) {
    const int u_next = u + n_warps;
    const bool more = u_next < n_units;
    PackUnit nx = un;
    if (more) {
      nx = pack_unit(pp, u_next, units0, per_b0, per_b1);
      pack_load4(pp.side[nx.side], nx, lane, vn, kn);
    }
    const PackArgs& a = pp.side[un.side];
    const int d = a.d;
    const bool data_lane = lane < (d >> 3);
    const bool two_packs = a.v_pack != a.s_pack;
    const size_t pack_off = ((size_t)un.b * (a.LP / 8) + (un.row0 >> 3)) * GROUP_BYTES + lane * 128 + (un.row0 & 7) * 16;
    char* const s_dst = reinterpret_cast<char*>(a.s_pack) + pack_off;
    char* const v_dst = reinterpret_cast<char*>(a.v_pack) + pack_off;
    float dot[4];
    uint4 vq[4], sq[4];                                 // this lane's four 16-byte pieces of the value pack / the S pack
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int row = un.row0 + r;
      const bool in = row < a.L;
      if (a.out_copy && in && data_lane) stg256(a.out_copy + ((size_t)un.b * a.L + row) * 4 * d + lane * 8, v[r]);   // out[:, :, 0:d] = text
      __nv_bfloat162 vp[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) vp[e] = __floats2bfloat162_rn(v[r][2 * e], v[r][2 * e + 1]);
      vq[r] = lane < CHUNKS - 1 ? *reinterpret_cast<uint4*>(vp) : make_uint4(0u, 0u, 0u, 0u);
      if (a.keep) {                                     // dropout (attention.py:66-67): the S operand sees the dropped values
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const uint32_t word = e < 4 ? kraw[r].x : kraw[r].y;
          v[r][e] = ((word >> (8 * (e & 3))) & 0xffu) ? v[r][e] * a.keep_scale : 0.f;
        }
      }
      float dt = 0.f;
      __nv_bfloat162 sp[4];
      if (un.side == 0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) dt = fmaf(v[r][e], wt0[e], dt);
#pragma unroll
        for (int e = 0; e < 4; ++e) sp[e] = __floats2bfloat162_rn(v[r][2 * e] * wf0[2 * e], v[r][2 * e + 1] * wf0[2 * e + 1]);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) dt = fmaf(v[r][e], wt1[e], dt);
#pragma unroll
        for (int e = 0; e < 4; ++e) sp[e] = __floats2bfloat162_rn(v[r][2 * e], v[r][2 * e + 1]);
      }
      dot[r] = dt;
      sq[r] = *reinterpret_cast<uint4*>(sp);
    }
    if (two_packs && lane < CHUNKS) {
      stg256_u(v_dst, vq[0], vq[1]);
      stg256_u(v_dst + 32, vq[2], vq[3]);
    }
    if (lane < CHUNKS - 1) {
      stg256_u(s_dst, sq[0], sq[1]);
      stg256_u(s_dst + 32, sq[2], sq[3]);
    }
    // the four row sums at once: two exchange steps halve the number of values a lane carries, three more finish them
    {
      const bool up16 = lane & 16, up8 = lane & 8;
      const float a0 = (up16 ? dot[2] : dot[0]) + __shfl_xor_sync(0xffffffffu, up16 ? dot[0] : dot[2], 16);   // rows {0,1} on lanes 0-15, {2,3} on 16-31
      const float a1 = (up16 ? dot[3] : dot[1]) + __shfl_xor_sync(0xffffffffu, up16 ? dot[1] : dot[3], 16);
      float sm = (up8 ? a1 : a0) + __shfl_xor_sync(0xffffffffu, up8 ? a0 : a1, 8);                             // one row per 8-lane group
      sm += __shfl_xor_sync(0xffffffffu, sm, 4);
      sm += __shfl_xor_sync(0xffffffffu, sm, 2);
      sm += __shfl_xor_sync(0xffffffffu, sm, 1);
#pragma unroll
      for (int r = 0; r < 4; ++r) dot[r] = __shfl_sync(0xffffffffu, sm, ((r >> 1) * 16) + ((r & 1) * 8));
    }
    if (lane == CHUNKS - 1) {                           // the K-padding chunk carries the additive term
      uint4 tq[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const bool in = un.row0 + r < a.L;
        const __nv_bfloat16 hi = __float2bfloat16_rn(dot[r]);
        const __nv_bfloat16 lo = __float2bfloat16_rn(dot[r] - __bfloat162float(hi));
        const __nv_bfloat16 one = __float2bfloat16_rn(in ? 1.f : 0.f);
        __nv_bfloat16 t[8] = {zero, zero, zero, zero, zero, zero, zero, zero};
        if (a.text_side) { t[0] = in ? hi : zero; t[1] = in ? lo : zero; t[2] = one; t[3] = one; }
        else             { t[0] = one; t[1] = one; t[2] = in ? hi : zero; t[3] = in ? lo : zero; }
        tq[r] = *reinterpret_cast<uint4*>(t);
      }
      stg256_u(s_dst, tq[0], tq[1]);
      stg256_u(s_dst + 32, tq[2], tq[3]);
    }
    // mask words of the 64-row tile this unit starts
    if ((un.row0 & 63) == 0) {
      const int tile = un.row0 >> 6;
      const int r0 = un.row0 + lane, r1 = r0 + 32;
      const unsigned v0 = __ballot_sync(0xffffffffu, r0 < a.L), v1 = __ballot_sync(0xffffffffu, r1 < a.L);
      const unsigned o0 = __ballot_sync(0xffffffffu, r0 < a.L && a.mask[(size_t)un.b * a.L + min(r0, a.L - 1)] != 0);
      const unsigned o1 = __ballot_sync(0xffffffffu, r1 < a.L && a.mask[(size_t)un.b * a.L + min(r1, a.L - 1)] != 0);
      if (lane == 0) {
        a.mask_words[((size_t)un.b * (a.LP / 64) + tile) * 2 + 0] = ((unsigned long long)v1 << 32) | v0;
        a.mask_words[((size_t)un.b * (a.LP / 64) + tile) * 2 + 1] = ((unsigned long long)o1 << 32) | o0;
      }
    }
    if (!more) break;
    u = u_next;
    un = nx;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      kraw[r] = kn[r];
#pragma unroll
      for (int e = 0; e < 8; ++e) v[r][e] = vn[r][e];
    }
  }
}

}  // namespace

int bidaf_fwd_tc5_launch(const BidafPacks& pk, const float* text, const float* bias, float* out, float* q2c, float* bm,
                         float* lse_row, float* lse_col, int B, int Lc, int Lq, int d, cudaStream_t stream);

// Workspace (bytes): packed operands, mask words (layout: tc_common.cuh::bidaf_packs).
size_t bidaf_tc_workspace_bytes(int B, int Lc, int Lq, int dropout) { return bidaf_packs(nullptr, B, Lc, Lq, dropout != 0).bytes; }

int bidaf_fwd_tc(const float* text, const float* modality, const uint8_t* text_mask, const uint8_t* modality_mask,
                 const float* w_text, const float* w_modality, const float* w_cross, const float* bias,
                 const uint8_t* keep_text, const uint8_t* keep_modality, float keep_scale, float* out, float* q2c,
                 float* bm, float* lse_row, float* lse_col, void* workspace, int B, int Lc, int Lq, int d, cudaStream_t stream) {
  MMB_REQUIRE(d % 8 == 0 && d <= 200, MMB_ERR_UNSUPPORTED, "mmb_bidaf_fwd (bf16 tier): d=%d (need d %% 8 == 0, d <= 200)", d);
  MMB_REQUIRE(workspace, MMB_ERR_INVALID, "mmb_bidaf_fwd (bf16 tier): workspace is null");
  const BidafPacks pk = bidaf_packs(workspace, B, Lc, Lq, keep_modality != nullptr);
  const int LcP = pk.LcP, LqP = pk.LqP;

  PackPair pp;
  pp.side[0] = PackArgs{text, keep_text, text_mask, w_text, w_cross, pk.cw, pk.cp, pk.c_words, out, keep_scale, Lc, LcP, d, 1};
  pp.side[1] = PackArgs{modality, keep_modality, modality_mask, w_modality, nullptr, pk.qs, pk.qp, pk.q_words, nullptr, keep_scale,
                        Lq, LqP, d, 0};
  {
    static int num_sms = 0;
    if (num_sms == 0) {
      int dev = 0;
      MMB_CUDA(cudaGetDevice(&dev));
      MMB_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    }
    const int n_units = B * (LcP + LqP) / 4;
    const int blocks = min((n_units + 3) / 4, num_sms * 4);         // 16 warps per SM, each streaming over its units
    bidaf_pack_kernel<<<blocks, 128, 0, stream>>>(pp, B, pk.ready, B + 1);
  }
  if (int rc = check_launch("bidaf_pack_kernel")) return rc;

  return bidaf_fwd_tc5_launch(pk, text, bias, out, q2c, bm, lse_row, lse_col, B, Lc, Lq, d, stream);
}

}  // namespace mmb
