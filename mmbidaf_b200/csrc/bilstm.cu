// Persistent length-aware LSTM recurrence, forward and backward (BPTT), fp32.
//
// Replaces the nn.LSTM call of layers/encoding.py:96 (and the sort / pack / unpack / unsort
// gathers around it, encoding.py:91-101) for one layer, both directions.  The input projection
// x W_ih^T + b_ih + b_hh is a plain GEMM done by the caller; this kernel owns the serial part.
//
// One CTA = one direction x NB sequences, alive for the whole sequence.  FORWARD kernel: two lanes share a hidden
// unit j: lane kp (0/1) keeps in REGISTERS the recurrent weights of all four gate rows of unit j
// restricted to half of the k range (4 x KS floats, KS = 52 at H = 100), so W_hh never leaves the
// register file between time steps and the CTA is only 2H threads (7 warps at H = 100: <= 2 warps per
// scheduler, 255 registers each -- no spills).  Per step: 4 x KS FMAs against h (broadcast float4
// reads from shared memory), a 2-shuffle reduce-scatter (lane 0 ends with gates i,f; lane 1 with g,o),
// two branch-free activations per lane, a 2-shuffle exchange, the cell update, one __syncthreads.
// Input pre-activations are prefetched RING-1 steps ahead with cp.async; all addressing is by running
// pointers (one add per step).  The BACKWARD kernel uses a different cut (a gate per warp pair), see its header.
//
// Semantics follow torch.nn.LSTM on a PackedSequence: gate order i,f,g,o; zero initial state;
// the reverse direction starts at each sample's own last valid step; outputs past a sample's
// length are exactly zero (pad_packed_sequence, encoding.py:99); h_n / c_n are the states after
// each sample's last valid step.
#include <stdlib.h>
#include "common.cuh"

namespace mmb {
namespace {

constexpr int RING = 8;          // power of two

__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// 1 - k / (1 + 2^z): sigma(x) for k = 1, z = x log2 e; tanh(x) for k = 2, z = 2 x log2 e.  ex2 / rcp in their flush-to-zero forms (one
// MUFU each, no range fix-ups: 2^z -> inf gives 1, 2^z -> 0 gives 1 - k).
__device__ __forceinline__ float gate_act2(float z, float k) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return fmaf(-k, r, 1.0f);
}

// Predicated memory operations: the loop body of the recurrence must stay ONE basic block (ptxas does not schedule across the branches
// that `if (on) *p = v;` compiles to, and every instruction of a step that is not FMA work has to be interleaved with the FMAs).
__device__ __forceinline__ void st_global_if(float* p, float v, bool pred) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.f32 [%0], %1;\n\t}" ::"l"(p), "f"(v), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void st_shared_if(float* p, float v, bool pred) {
  const unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(p));
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.shared.f32 [%0], %1;\n\t}" ::"r"(sa), "f"(v), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void cp_async4_if(float* smem_dst, const float* gsrc, bool pred) {
  const unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q cp.async.ca.shared.global [%0], [%1], 4;\n\t}" ::"r"(sa), "l"(gsrc), "r"((int)pred) : "memory");
}

struct LstmArgs {
  float* gates;            // (B, L, ndir, 4H): in = input pre-activations, out (save) = activated gates / d pre-act
  const float* w_hh;       // (ndir, 4H, H)
  const int* lengths;      // (B)
  const int* order;        // (B) permutation (longest first) or nullptr
  float* out;              // fwd: (B, L, ndir*H)
  float* h_n;              // fwd: (B, ndir, H)
  float* c_n;              // fwd: (B, ndir, H)
  float* cell;             // (B, L, ndir, H) saved cell states (fwd writes when save != 0, bwd reads)
  const float* dout;       // bwd: (B, L, ndir*H)
  const float* dh_n;       // bwd: (B, ndir, H) or nullptr
  const float* dc_n;       // bwd: (B, ndir, H) or nullptr
  int B, L, H, ndir, save;
  long long* trace;        // debugging aid (MMB_LSTM_TRACE, tools/lstm_trace.py): clock64 stamps of CTA (0, 0), or null
  // dropout on the layer's OUTPUT (encoding.py:104, nn.LSTM's inter-layer dropout), applied in the kernel: keep bits from
  // common.cuh::dropout_keep(element index in (B, L, ndir H), key).  fwd: y = keep ? out / keep_prob : 0 is written beside `out`
  // (the recurrence and the weight gradients keep the un-dropped states); bwd: `dout` is d y.
  float* y;                            // fwd: (B, L, ndir*H) or null (no dropout)
  const unsigned long long* rng_key;   // device scalar, or null (no dropout)
  float keep_prob;
};

constexpr int threads_for(int KS) { return (4 * KS + 31) / 32 * 32 < 64 ? 64 : (4 * KS + 31) / 32 * 32; }

// Stamp that cannot be scheduled before the values it names are computed.
__device__ __forceinline__ long long clock_after(float x, float y) {
  long long t;
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "f"(x), "f"(y) : "memory");
  return t;
}
constexpr int TRACE_S0 = 64, TRACE_NS = 32, TRACE_PTS = 5;   // steps [64, 96): 5 stamps per step, lane 0 of each warp

constexpr int pow2_ceil(int x) { int p = 1; while (p < x) p *= 2; return p; }

// The loop body is written for INSTRUCTION COUNT and as one basic block (tools/lstm_trace.py, round 2: a step is issue bound -- two
// warps per scheduler, ~380 instructions each, of which 211 are the FFMAs; the serial tail after them is ~320 cycles):
//  * the weights are PRE-SCALED by log2(e) (2 log2(e) for the tanh gate g) so that the accumulated pre-activation is the argument of
//    ex2 directly: sigma(x) = 1 - 1 / (1 + 2^(x log2 e)), tanh(x) = 1 - 2 / (1 + 2^(2 x log2 e));
//  * a lane keeps its weight rows in the order (kept gate 0, kept gate 1, sent gate 0, sent gate 1) -- lane 0 keeps (i, f), lane 1
//    (g, o) -- so the reduce-scatter over the pair needs no selects, and the input pre-activations SEED the two kept accumulators;
//  * the global stores of a step (out, saved gates, cell state) are issued one step LATE, from registers, inside the next step's FMA
//    stream, and every memory operation is predicated rather than branched around;
//  * the cp.async ring has a power-of-two slot stride: one add + one and per step for both ring positions.
// Measured and not kept (round 2, tools/lstm_trace.py): eight accumulator chains instead of four (no change: a warp alone on its
// scheduler issues an FFMA every ~2 cycles whatever the chain count); packed fma.rn.f32x2 (104 FFMA2 instead of 208 FFMA: a lone warp
// then needs ~7 cycles per FFMA2, two warps ~4 -- the same FMA rate, 0.518 - 0.535 against 0.532 us per step).
template <int KS, int NB, bool TRACE = false, bool DROP = false>
__global__ void __launch_bounds__(threads_for(KS)) bilstm_fwd_kernel(const LstmArgs a) {
  constexpr int HP = 2 * KS;                       // padded hidden size
  constexpr int NT = threads_for(KS);              // == blockDim.x
  constexpr int RSLOT = pow2_ceil(NB * 2 * NT);    // floats per ring slot: [NB][2][NT], padded to a power of two
  constexpr int RMASK = RING * RSLOT - 1;
  const int H = a.H, L = a.L, ndir = a.ndir;
  const int dir = blockIdx.y;
  const int tid = threadIdx.x;
  const int j = tid >> 1, kp = tid & 1;
  const bool live = j < H;
  const int jj = min(j, H - 1);                    // threads past the last unit MIRROR it: same weights, same values, same addresses,
                                                   // so nothing in the loop is predicated on the thread

  extern __shared__ __align__(16) float smem[];
  float* h_s = smem;                               // [2][NB][HP]
  float* ring = h_s + 2 * NB * HP;                 // [RING][RSLOT]

  int seq[NB], len[NB];
  int max_len = 0;
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const int slot = blockIdx.x * NB + n;
    seq[n] = slot < a.B ? (a.order ? a.order[slot] : slot) : -1;
    len[n] = seq[n] >= 0 ? min(max(a.lengths[seq[n]], 0), L) : 0;
    max_len = max(max_len, len[n]);
  }

  // recurrent weights of unit j, k in [kp*KS, kp*KS + KS); slot q of w holds gate (q < 2 ? 2 kp + q : 2 (1 - kp) + q - 2)
  constexpr float LOG2E_F = 1.4426950408889634f;
  float w[4][KS];
  {
    const float* wd = a.w_hh + (size_t)dir * 4 * H * H;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int g = q < 2 ? 2 * kp + q : 2 * (1 - kp) + (q - 2);
      const float sc = g == 2 ? 2.f * LOG2E_F : LOG2E_F;
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        const int k = kp * KS + kk;
        w[q][kk] = k < H ? wd[(size_t)(g * H + jj) * H + k] * sc : 0.f;
      }
    }
  }
  for (int i = tid; i < 2 * NB * HP; i += NT) h_s[i] = 0.f;

  // Running pointers: this lane's two pre-activation / saved-gate slots (gates 2kp, 2kp+1 of unit j), the output slot and the cell slot
  // of sequence n at the step being STORED (one behind the step being computed), and the prefetch pointer RING-1 steps ahead.
  // Forward walks t = 0.., the reverse direction t = len-1 ...
  const long sign = dir ? -1 : 1;
  const long g_stride = sign * (long)ndir * 4 * H, o_stride = sign * (long)ndir * H;
  float *gp[NB], *op[NB], *cp[NB];
  const float* pf[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const size_t bt0 = (size_t)max(seq[n], 0) * L + (dir ? max(len[n] - 1, 0) : 0);
    gp[n] = a.gates + (bt0 * ndir + dir) * 4 * H + (2 * kp) * H + jj;
    op[n] = a.out + bt0 * ndir * H + dir * H + jj;
    cp[n] = (a.cell ? a.cell : a.out) + (bt0 * ndir + dir) * H + jj;   // (never dereferenced without a cell buffer)
    pf[n] = gp[n];
  }
  float* const ring_t = ring + tid;
  auto prefetch = [&](int s, int off) {            // off: float offset of the ring slot
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const bool p = s < len[n];
      cp_async4_if(ring_t + off + (n * 2 + 0) * NT, pf[n], p);
      cp_async4_if(ring_t + off + (n * 2 + 1) * NT, pf[n] + H, p);
      pf[n] += g_stride;
    }
    cp_async_commit();
  };
#pragma unroll 1
  for (int s = 0; s < RING - 1; ++s) prefetch(s, s * RSLOT);
  __syncthreads();

  float c_reg[NB], h_reg[NB], a0_reg[NB], a1_reg[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) c_reg[n] = h_reg[n] = a0_reg[n] = a1_reg[n] = 0.f;
  // output dropout: key halves, threshold, 1 / keep_prob, and the distance from `out` to `y` (one add per store)
  constexpr bool drop = DROP;                      // (compile time: the loop body must stay one basic block)
  const unsigned long long key = drop ? a.rng_key[0] : 0ull;
  const uint32_t key0 = (uint32_t)key, key1 = (uint32_t)(key >> 32), thresh = dropout_thresh(a.keep_prob);
  const float inv_keep = drop ? 1.f / a.keep_prob : 1.f;
  const long y_off = drop ? a.y - a.out : 0;
  const float k_first = kp ? 2.0f : 1.0f;          // lane 0: (i, f) both sigmoid; lane 1: (g = tanh, o = sigmoid)
  const float pre_first = k_first * LOG2E_F;
  const bool save = a.save != 0;
  // (both lanes of a pair hold the same h and c: both store them -- same address, same value -- rather than predicate on the lane)
  int hoff = 0;                                    // float offset of the current h buffer (0 or NB * HP)
  int roff = 0;                                    // float offset of the current ring slot
  __shared__ long long tr_s[TRACE ? TRACE_NS * 8 * TRACE_PTS : 1];
  const bool tr_on = TRACE && blockIdx.x == 0 && blockIdx.y == 0 && (tid & 31) == 0;

#pragma unroll 1
  for (int s = 0; s < max_len; ++s) {
    const bool tr_now = TRACE && tr_on && s >= TRACE_S0 && s < TRACE_S0 + TRACE_NS;
    long long* const tr = tr_s + ((s - TRACE_S0) * 8 + (tid >> 5)) * TRACE_PTS;
    if (tr_now) tr[0] = clock_after(0.f, 0.f);
    prefetch(s + RING - 1, (roff + (RING - 1) * RSLOT) & RMASK);
    cp_async_wait<RING - 1>();
    const float* hk = h_s + hoff + kp * KS;

    // the input pre-activations of this step (scaled like the weights) seed the two kept accumulators.  A sequence that has ended
    // (NB = 2 only) reads a stale ring slot: its values are never stored.
    float acc[NB][4];
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const float* rs = ring_t + roff + n * 2 * NT;
      acc[n][0] = rs[0] * pre_first;
      acc[n][1] = rs[NT] * LOG2E_F;
      acc[n][2] = acc[n][3] = 0.f;
    }
#pragma unroll
    for (int k4 = 0; k4 < KS / 4; ++k4) {
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        const float4 hv = *reinterpret_cast<const float4*>(hk + n * HP + k4 * 4);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          acc[n][g] = fmaf(w[g][k4 * 4 + 0], hv.x, acc[n][g]);
          acc[n][g] = fmaf(w[g][k4 * 4 + 1], hv.y, acc[n][g]);
          acc[n][g] = fmaf(w[g][k4 * 4 + 2], hv.z, acc[n][g]);
          acc[n][g] = fmaf(w[g][k4 * 4 + 3], hv.w, acc[n][g]);
        }
      }
    }
    // the previous step's values go to memory now: independent of this step's chain, interleaved with it by the scheduler
    {
      const bool prev = s > 0;
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        const bool on = prev && (NB == 1 || s - 1 < len[n]), on_sv = on && save;
        st_global_if(op[n], h_reg[n], on);
        if (drop) {                                                 // (uniform)
          const bool keep = dropout_keep((uint32_t)(op[n] - a.out), key0, key1, thresh);
          st_global_if(op[n] + y_off, keep ? h_reg[n] * inv_keep : 0.f, on);
        }
        st_global_if(gp[n], a0_reg[n], on_sv);
        st_global_if(gp[n] + H, a1_reg[n], on_sv);
        st_global_if(cp[n], c_reg[n], on_sv);
        gp[n] += prev ? g_stride : 0;
        op[n] += prev ? o_stride : 0;
        cp[n] += prev ? o_stride : 0;
      }
    }
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const bool on = NB == 1 || s < len[n];                       // uniform over the CTA
      if (tr_now && n == 0) tr[1] = clock_after(acc[n][0] + acc[n][1], acc[n][2] + acc[n][3]);
      // reduce-scatter over the lane pair: lane 0 ends with gates (i, f), lane 1 with (g, o)
      const float m0 = acc[n][0] + __shfl_xor_sync(0xffffffffu, acc[n][2], 1);
      const float m1 = acc[n][1] + __shfl_xor_sync(0xffffffffu, acc[n][3], 1);
      const float a0 = gate_act2(m0, k_first);                     // i | g
      const float a1 = gate_act2(m1, 1.0f);                        // f | o
      if (tr_now && n == 0) tr[2] = clock_after(a0, a1);
      const float b0 = __shfl_xor_sync(0xffffffffu, a0, 1);
      const float b1 = __shfl_xor_sync(0xffffffffu, a1, 1);
      const float gf = kp ? b1 : a1, go = kp ? a1 : b1;            // (i g = a0 b0 on both lanes)
      const float c_new = fmaf(gf, c_reg[n], a0 * b0);
      const float h_new = go * gate_act2(c_new * (2.f * LOG2E_F), 2.0f);
      if (tr_now && n == 0) tr[3] = clock_after(h_new, 0.f);
      st_shared_if(h_s + (hoff ^ (NB * HP)) + n * HP + jj, h_new, on);
      c_reg[n] = on ? c_new : c_reg[n];
      h_reg[n] = on ? h_new : h_reg[n];
      a0_reg[n] = a0;
      a1_reg[n] = a1;
    }
    roff = (roff + RSLOT) & RMASK;
    hoff ^= NB * HP;
    if (tr_now) tr[4] = clock_after(0.f, 0.f);
    __syncthreads();
  }
  // the last step's values
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const bool on = max_len > 0 && max_len - 1 < len[n], on_sv = on && save;
    st_global_if(op[n], h_reg[n], on);
    if (drop) {
      const bool keep = dropout_keep((uint32_t)(op[n] - a.out), key0, key1, thresh);
      st_global_if(op[n] + y_off, keep ? h_reg[n] * inv_keep : 0.f, on);
    }
    st_global_if(gp[n], a0_reg[n], on_sv);
    st_global_if(gp[n] + H, a1_reg[n], on_sv);
    st_global_if(cp[n], c_reg[n], on_sv);
  }
  cp_async_wait<0>();
  if (TRACE && blockIdx.x == 0 && blockIdx.y == 0 && a.trace)
    for (int i = tid; i < TRACE_NS * 8 * TRACE_PTS; i += NT) a.trace[i] = tr_s[i];

#pragma unroll
  for (int n = 0; n < NB; ++n) {
    if (seq[n] < 0) continue;
    if (live && kp == 0) a.h_n[((size_t)seq[n] * ndir + dir) * H + j] = h_reg[n];
    if (live && kp == 1) a.c_n[((size_t)seq[n] * ndir + dir) * H + j] = c_reg[n];
    // pad_packed_sequence: zeros past the sample's length
    for (int i = tid; i < (L - len[n]) * H; i += NT) {
      const int t = len[n] + i / H, u = i % H;
      a.out[((size_t)seq[n] * L + t) * ndir * H + dir * H + u] = 0.f;
      if (drop) a.y[((size_t)seq[n] * L + t) * ndir * H + dir * H + u] = 0.f;
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------------
// Forward, two CTAs per (sequence, direction): a thread-block CLUSTER of two splits the hidden units.
//
// A step of the kernel above is ISSUE bound, not FMA bound: one CTA runs the whole 4H x H mat-vec of its sequence, 7 warps on 4
// schedulers (2, 2, 2, 1) at ~355 instructions per warp and step -> >= 710 issue slots on the busy schedulers, ~1 300 cycles measured.
// Here each CTA of the pair owns half of the hidden units (same lane-pair layout, same per-thread work: 4 warps, ONE per scheduler)
// and the two halves of h meet in both CTAs' shared memory: every new h value is stored locally and -- st.async with
// mbarrier::complete_tx -- into the partner's buffer, whose threads wait on their own mbarrier for the partner's bytes.  The exchange
// costs one DSMEM latency (~215 cycles) per step, the issue-bound part halves.  The h buffers are double buffered: a CTA can only be
// one step ahead of its partner (it needs the partner's h(t) to run step t), which is exactly what two buffers allow.
// ----------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ unsigned map_to_cta(const void* local_smem, unsigned rank) {
  const unsigned l = static_cast<unsigned>(__cvta_generic_to_shared(local_smem));
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(l), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_f32(unsigned remote_addr, float v, unsigned remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr), "r"(__float_as_uint(v)),
               "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void pair_bar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void pair_bar_expect(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pair_bar_wait(unsigned bar, unsigned parity) {
#pragma unroll 1
  for (unsigned spin = 0; spin < (1u << 26); ++spin) {
    unsigned done;
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
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int KS>
__global__ void __launch_bounds__(threads_for(KS / 2 + 1)) bilstm_fwd_pair_kernel(const LstmArgs a) {
  constexpr int HP = 2 * KS;                       // padded hidden size
  const int H = a.H, L = a.L, ndir = a.ndir;
  const int dir = blockIdx.y;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const unsigned rank = cluster_ctarank();
  const int UH = (H + 1) / 2;                      // units per CTA
  const int jj = tid >> 1, kp = tid & 1;
  const int j = (int)rank * UH + jj;
  const bool live = jj < UH && j < H;

  extern __shared__ __align__(16) float smem[];
  float* h_s = smem;                               // [2][HP]  the full hidden state, both halves
  float* ring = h_s + 2 * HP;                      // [RING][2][nthr]
  __shared__ __align__(8) unsigned long long bars[2];

  const int slot_b = blockIdx.x >> 1;
  const int seq = slot_b < a.B ? (a.order ? a.order[slot_b] : slot_b) : -1;
  const int len = seq >= 0 ? min(max(a.lengths[seq], 0), L) : 0;

  float w[4][KS];
  {
    const float* wd = a.w_hh + (size_t)dir * 4 * H * H;
#pragma unroll
    for (int g = 0; g < 4; ++g)
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        const int k = kp * KS + kk;
        w[g][kk] = (live && k < H) ? wd[(size_t)(g * H + j) * H + k] : 0.f;
      }
  }
  for (int i = tid; i < 2 * HP; i += nthr) h_s[i] = 0.f;
  const unsigned bar0 = static_cast<unsigned>(__cvta_generic_to_shared(&bars[0]));
  if (tid == 0) {
    pair_bar_init(bar0, 1);
    pair_bar_init(bar0 + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // the partner's units and the bytes it sends per step
  const int other_units = max(0, min(UH, H - (int)(rank ^ 1u) * UH));
  const unsigned rbar0 = map_to_cta(&bars[0], rank ^ 1u);
  const unsigned rh0 = map_to_cta(h_s, rank ^ 1u);

  const long sign = dir ? -1 : 1;
  const long g_stride = sign * (long)ndir * 4 * H, o_stride = sign * (long)ndir * H;
  const size_t bt0 = (size_t)max(seq, 0) * L + (dir ? max(len - 1, 0) : 0);
  const int jc = live ? j : 0;
  float* gp = a.gates + (bt0 * ndir + dir) * 4 * H + (2 * kp) * H + jc;
  float* op = a.out + bt0 * ndir * H + dir * H + jc;
  float* cp = a.cell ? a.cell + (bt0 * ndir + dir) * H + jc : nullptr;
  const float* pf = gp;
  float* ring_t = ring + tid;
  auto prefetch = [&](int s, int slot) {
    if (live) {
      if (s < len) {
        cp_async4(ring_t + (slot * 2 + 0) * nthr, pf);
        cp_async4(ring_t + (slot * 2 + 1) * nthr, pf + H);
      }
      pf += g_stride;
    }
    cp_async_commit();
  };
#pragma unroll 1
  for (int s = 0; s < RING - 1; ++s) prefetch(s, s);
  __syncthreads();
  cluster_sync_all();                              // both CTAs' barriers and zeroed buffers exist before any remote store

  float c_reg = 0.f, h_reg = 0.f;
  const float k_first = kp ? 2.0f : 1.0f;          // lane 0: (i, f) both sigmoid; lane 1: (g = tanh, o = sigmoid)
  const bool save = a.save != 0;
  int cur = 0, slot = 0;

#pragma unroll 1
  for (int s = 0; s < len; ++s) {
    const int nxt = cur ^ 1;
    if (tid == 0) pair_bar_expect(bar0 + 8 * nxt, 4u * (unsigned)other_units);   // the partner's half of h(s + 1)
    prefetch(s + RING - 1, (slot + RING - 1) & (RING - 1));
    cp_async_wait<RING - 1>();
    const float* hk = h_s + cur * HP + kp * KS;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k4 = 0; k4 < KS / 4; ++k4) {
      const float4 hv = *reinterpret_cast<const float4*>(hk + k4 * 4);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        acc[g] = fmaf(w[g][k4 * 4 + 0], hv.x, acc[g]);
        acc[g] = fmaf(w[g][k4 * 4 + 1], hv.y, acc[g]);
        acc[g] = fmaf(w[g][k4 * 4 + 2], hv.z, acc[g]);
        acc[g] = fmaf(w[g][k4 * 4 + 3], hv.w, acc[g]);
      }
    }
    // reduce-scatter over the lane pair: lane 0 keeps gates (i, f), lane 1 keeps (g, o)
    float m0 = kp ? acc[2] : acc[0], m1 = kp ? acc[3] : acc[1];
    m0 += __shfl_xor_sync(0xffffffffu, kp ? acc[0] : acc[2], 1);
    m1 += __shfl_xor_sync(0xffffffffu, kp ? acc[1] : acc[3], 1);
    const float* rs = ring_t + slot * 2 * nthr;
    const float a0 = gate_act(m0 + (live ? rs[0] : 0.f), k_first);   // i | g
    const float a1 = gate_act(m1 + (live ? rs[nthr] : 0.f), 1.0f);   // f | o
    const float b0 = __shfl_xor_sync(0xffffffffu, a0, 1);
    const float b1 = __shfl_xor_sync(0xffffffffu, a1, 1);
    const float gi = kp ? b0 : a0, gf = kp ? b1 : a1, gg = kp ? a0 : b0, go = kp ? a1 : b1;
    if (live) {
      c_reg = fmaf(gf, c_reg, gi * gg);
      h_reg = go * tanh_fast(c_reg);
      if (kp == 0) {
        h_s[nxt * HP + j] = h_reg;
        st_async_f32(rh0 + (unsigned)(nxt * HP + j) * 4u, h_reg, rbar0 + 8u * (unsigned)nxt);
        *op = h_reg;
      }
      if (save) {
        gp[0] = a0;
        gp[H] = a1;
        if (kp == 1) *cp = c_reg;
      }
    }
    gp += g_stride;
    op += o_stride;
    if (save) cp += o_stride;
    slot = (slot + 1) & (RING - 1);
    __syncthreads();                                                  // this CTA's half of h(s + 1) is in its buffer
    pair_bar_wait(bar0 + 8 * nxt, (unsigned)(s >> 1) & 1u);           // ... and so is the partner's
    cur = nxt;
  }
  cp_async_wait<0>();
  cluster_sync_all();                              // neither CTA exits while the other may still store into it

  if (seq >= 0) {
    if (live && kp == 0) a.h_n[((size_t)seq * ndir + dir) * H + j] = h_reg;
    if (live && kp == 1) a.c_n[((size_t)seq * ndir + dir) * H + j] = c_reg;
    // pad_packed_sequence: zeros past the sample's length (each CTA of the pair clears its own units)
    const int u0 = (int)rank * UH, nu = max(0, min(UH, H - u0));
    for (int i = tid; i < (L - len) * nu; i += nthr) {
      const int t = len + i / nu, u = u0 + i % nu;
      a.out[((size_t)seq * L + t) * ndir * H + dir * H + u] = 0.f;
    }
  }
}

// Backward through time.  `gates` holds the activated gates on entry and d(pre-activation) on exit
// (zeros past each length), so dW_ih / dx / db / dW_hh are plain GEMMs for the caller.
//
// The recurrent product dh[j] = sum_{g,r} W_hh[g H + r][j] da[g][r] reads FOUR H-vectors from shared memory per step
// (the forward reads one), and a broadcast LDS.128 costs 2.3 cycles per warp (tools/micro/lds_bcast.cu), so the first
// version (two lanes per unit, each reading the 2 x H values of its two gates: 52 LDS.128 per thread) spent ~820 of its
// 1700 cycles per step in the shared-memory pipe.  The second (a thread = TWO units x ONE gate x all r, the gate uniform
// over a warp pair: 26 LDS.128 per thread, 8 FFMAs per load) ran at 0.61, then 0.53 us per step, with a quarter of all
// warp-stall samples on FFMAs waiting for their shared-memory operand (ncu, short scoreboard).  Now a thread = FOUR units
// x ONE gate x HALF of r (the two halves on neighbouring lanes): 13 LDS.128 per thread, 16 FFMAs per load, the same 208
// weights in registers; the halves meet by one shuffle per unit, the four per-gate partial sums of a unit in shared
// memory; the point-wise part of a step is done by one thread per unit (threads 0..H-1), which also owns the cp.async
// ring.  (Packed fma.rn.f32x2 in place of the scalar FMAs halves the instruction count but is not faster: the FMA pipe
// takes an FFMA2 at half rate and the dependent chains get longer.)
constexpr int BWD_NT = 256, BWD_SL = 64;     // 8 warps = 4 gates x 2 halves of 32 unit slots; a slot covers units slot + 32 i, i < 4

// KR: r values per half that are real (H <= 2 KR <= 2 KS): the zero padding of a half costs registers and FFMAs (KS = 52, H = 100: 8 each)
template <int KS, int NB, int KR = KS, bool DROP = false>
__global__ void __launch_bounds__(BWD_NT) bilstm_bwd_kernel(const LstmArgs a) {
  constexpr int HP = 2 * KS;                       // >= H, multiple of 4
  constexpr int KSP = (KS % 32 == 0) ? KS + 4 : KS;   // row half stride of da_s: the two halves of r on different banks
  constexpr int DAS = 2 * KSP;                     // row stride of da_s
  static_assert(HP <= 2 * BWD_SL, "four units per slot cover the hidden size");
  const int H = a.H, L = a.L, ndir = a.ndir;
  const int dir = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp >> 1;                         // the gate whose rows this warp pair multiplies (warp-uniform)
  const int rh = lane & 1;                         // this lane's half of r
  const int slot = (warp & 1) * 16 + (lane >> 1);  // 0..31
  const bool unit = tid < H;                       // point-wise owner of hidden unit j = tid
  const int j = tid;

  extern __shared__ __align__(16) float smem[];
  float* da_s = smem;                              // [NB][4][2][KSP]
  float* part = da_s + NB * 4 * DAS;               // [NB][4][2 * BWD_SL]
  float* ring = part + NB * 4 * 2 * BWD_SL;        // [RING][NB][7][128]

  int seq[NB], len[NB];
  int max_len = 0;
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const int sl = blockIdx.x * NB + n;
    seq[n] = sl < a.B ? (a.order ? a.order[sl] : sl) : -1;
    len[n] = seq[n] >= 0 ? min(max(a.lengths[seq[n]], 0), L) : 0;
    max_len = max(max_len, len[n]);
  }

  float wt[4][KR];                                 // W_hh[q H + rh KR + r][slot + 32 u]
  {
    const float* wd = a.w_hh + (size_t)dir * 4 * H * H;
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int rr = 0; rr < KR; ++rr) {
        const int ju = slot + 32 * u, r = rh * KR + rr;
        wt[u][rr] = (ju < H && r < H) ? wd[(size_t)(q * H + r) * H + ju] : 0.f;
      }
  }
  for (int i = tid; i < NB * 4 * DAS + NB * 4 * 2 * BWD_SL; i += BWD_NT) da_s[i] = 0.f;

  // Backward step s visits the forward steps in reverse: time t = dir ? s : len-1-s.
  const long sign = dir ? 1 : -1;
  const long g_stride = sign * (long)ndir * 4 * H, o_stride = sign * (long)ndir * H;
  float* gp[NB];
  const float *pg[NB], *pc[NB], *pd[NB];           // prefetch pointers: gates, cell, dout (unit threads)
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    const size_t bt0 = (size_t)max(seq[n], 0) * L + (dir ? 0 : max(len[n] - 1, 0));
    gp[n] = a.gates + (bt0 * ndir + dir) * 4 * H + (unit ? j : 0);
    pg[n] = gp[n];
    pc[n] = a.cell + (bt0 * ndir + dir) * H + (unit ? j : 0);
    pd[n] = a.dout + bt0 * ndir * H + dir * H + (unit ? j : 0);
  }
  // Only what depends on the recurrent product of the previous step sits between the two barriers of a step: the point-wise part is
  // split into FACTORS that depend on the saved forward values alone -- computed a step ahead, inside the FMA stream of the previous
  // step's product, together with the global stores of d(pre-activation), the cp.async prefetch and the pointer updates -- and five
  // multiplies that need dh_rec (tools/lstm_trace.py for the forward kernel: a step is issue bound, its serial tail is what is left to cut).
  //   dh = dy + dh_rec;  dct = dh * A + dc;  d_i = dct Ki;  d_f = dct Kf;  d_g = dct Kg;  d_o = dh Ko;  dc = dct Gf
  //   A = go (1 - tanh^2 c),  Ki = gg gi (1 - gi),  Kf = c_prev gf (1 - gf),  Kg = gi (1 - gg^2),  Ko = tanh c  go (1 - go),  Gf = gf
  float* ring_t = ring + (tid & 127);
  const int ju = unit ? j : 0;
  auto prefetch = [&](int s, int sl) {
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const bool p = unit && s < len[n];
      float* dst = ring_t + (sl * NB + n) * 7 * 128;
#pragma unroll
      for (int g = 0; g < 4; ++g) cp_async4_if(dst + g * 128, pg[n] + g * H, p);
      cp_async4_if(dst + 4 * 128, pc[n], p);                                    // c_t
      cp_async4_if(dst + 5 * 128, pc[n] + o_stride, p && s + 1 < len[n]);       // c of the previous forward step
      cp_async4_if(dst + 6 * 128, pd[n], p);                                    // d out
      pg[n] += g_stride;
      pc[n] += o_stride;
      pd[n] += o_stride;
    }
    cp_async_commit();
  };
#pragma unroll 1
  for (int s = 0; s < RING - 1; ++s) prefetch(s, s);

  float dh_rec[NB], dc[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    dh_rec[n] = (unit && seq[n] >= 0 && a.dh_n) ? a.dh_n[((size_t)seq[n] * ndir + dir) * H + j] : 0.f;
    dc[n] = (unit && seq[n] >= 0 && a.dc_n) ? a.dc_n[((size_t)seq[n] * ndir + dir) * H + j] : 0.f;
  }
  // output dropout (see LstmArgs): d out = keep ? d y / keep_prob : 0, the keep bit recomputed from the element index
  constexpr bool drop = DROP;
  const unsigned long long key = drop ? a.rng_key[0] : 0ull;
  const uint32_t key0 = (uint32_t)key, key1 = (uint32_t)(key >> 32), thresh = dropout_thresh(a.keep_prob);
  const float inv_keep = drop ? 1.f / a.keep_prob : 1.f;
  uint32_t eidx[NB];                               // element index of (seq, t of backward step 0, dir H + j) in (B, L, ndir H)
#pragma unroll
  for (int n = 0; n < NB; ++n)
    eidx[n] = (uint32_t)(((size_t)max(seq[n], 0) * L + (dir ? 0 : max(len[n] - 1, 0))) * ndir * H + dir * H + (unit ? j : 0));
  struct Factors { float A, Ki, Kf, Kg, Ko, Gf, Dy; };
  auto factors = [&](int s, int sl, int n) {       // of backward step s, from ring slot sl (all zero past the sequence's end)
    Factors f{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float* rs = ring_t + (sl * NB + n) * 7 * 128;
    const float gi = rs[0], gf = rs[128], gg = rs[2 * 128], go = rs[3 * 128], ct = rs[4 * 128];
    float dy = rs[6 * 128];
    if (drop) dy = dropout_keep(eidx[n] + (uint32_t)(s * (int)o_stride), key0, key1, thresh) ? dy * inv_keep : 0.f;
    const float cprev = s + 1 < len[n] ? rs[5 * 128] : 0.f;
    const float tc = tanh_fast(ct);
    const bool on = s < len[n];
    f.A = on ? go * (1.f - tc * tc) : 0.f;
    f.Ki = on ? gg * gi * (1.f - gi) : 0.f;
    f.Kf = on ? cprev * gf * (1.f - gf) : 0.f;
    f.Kg = on ? gi * (1.f - gg * gg) : 0.f;
    f.Ko = on ? tc * go * (1.f - go) : 0.f;
    f.Gf = on ? gf : 0.f;
    f.Dy = on ? dy : 0.f;
    return f;
  };
  cp_async_wait<RING - 2>();                       // the first step's slot has landed (each thread reads what it copied itself)
  Factors fc[NB];
#pragma unroll
  for (int n = 0; n < NB; ++n) fc[n] = factors(0, 0, n);
  __syncthreads();
  int sl = 0;

#pragma unroll 1
  for (int s = 0; s < max_len; ++s) {
    // ---- between the barriers: what needs dh_rec -----------------------------------------------------------------------
    float dg[NB][4];
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const float dh = fc[n].Dy + dh_rec[n];
      const float dct = fmaf(dh, fc[n].A, dc[n]);
      dg[n][0] = dct * fc[n].Ki;
      dg[n][1] = dct * fc[n].Kf;
      dg[n][2] = dct * fc[n].Kg;
      dg[n][3] = dh * fc[n].Ko;
      dc[n] = dct * fc[n].Gf;
      float* dn = da_s + n * 4 * DAS + (ju / KR) * KSP + (ju % KR);
#pragma unroll
      for (int g = 0; g < 4; ++g) st_shared_if(dn + g * DAS, dg[n][g], unit);
    }
    __syncthreads();
    // ---- dh_rec partials: this warp pair's gate, this thread's two units; and, in the same instruction stream, everything of
    //      this and the next step that does not depend on them ---------------------------------------------------------------
    prefetch(s + RING - 1, (sl + RING - 1) & (RING - 1));
    cp_async_wait<RING - 2>();                                       // slot of step s + 1
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const bool on = unit && s < len[n];
#pragma unroll
      for (int g = 0; g < 4; ++g) st_global_if(gp[n] + g * H, dg[n][g], on);
      gp[n] += g_stride;
      fc[n] = factors(s + 1, (sl + 1) & (RING - 1), n);
    }
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      float pu[4] = {0.f, 0.f, 0.f, 0.f};
      const float* dq = da_s + (n * 4 + q) * DAS + rh * KSP;
#pragma unroll
      for (int r4 = 0; r4 < (KR + 3) / 4; ++r4) {
        const float4 dv = *reinterpret_cast<const float4*>(dq + r4 * 4);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (r4 * 4 + 0 < KR) pu[u] = fmaf(wt[u][r4 * 4 + 0], dv.x, pu[u]);
          if (r4 * 4 + 1 < KR) pu[u] = fmaf(wt[u][r4 * 4 + 1], dv.y, pu[u]);
          if (r4 * 4 + 2 < KR) pu[u] = fmaf(wt[u][r4 * 4 + 2], dv.z, pu[u]);
          if (r4 * 4 + 3 < KR) pu[u] = fmaf(wt[u][r4 * 4 + 3], dv.w, pu[u]);
        }
      }
      // the two halves of r meet: the even lane ends with units 0, 1 of the slot, the odd lane with units 2, 3
      const float s0 = (rh ? pu[2] : pu[0]) + __shfl_xor_sync(0xffffffffu, rh ? pu[0] : pu[2], 1);
      const float s1 = (rh ? pu[3] : pu[1]) + __shfl_xor_sync(0xffffffffu, rh ? pu[1] : pu[3], 1);
      float* pn = part + (n * 4 + q) * 2 * BWD_SL + slot + 64 * rh;
      pn[0] = s0;
      pn[32] = s1;
    }
    __syncthreads();
#pragma unroll
    for (int n = 0; n < NB; ++n) {
      const float* pn = part + n * 4 * 2 * BWD_SL + ju;
      dh_rec[n] = (pn[0] + pn[2 * BWD_SL]) + (pn[4 * BWD_SL] + pn[6 * BWD_SL]);
    }
    sl = (sl + 1) & (RING - 1);
  }
  cp_async_wait<0>();

  // d(pre-activation) is zero past each sample's length
#pragma unroll
  for (int n = 0; n < NB; ++n) {
    if (seq[n] < 0) continue;
    for (int i = tid; i < (L - len[n]) * 4 * H; i += BWD_NT) {
      const int t = len[n] + i / (4 * H), u = i % (4 * H);
      a.gates[(((size_t)seq[n] * L + t) * ndir + dir) * 4 * H + u] = 0.f;
    }
  }
}

template <int KS, int NB>
int launch(const LstmArgs& a, bool backward, cudaStream_t stream) {
  constexpr int HP = 2 * KS;
  const int nthr = max(((2 * a.H + 31) / 32) * 32, 64);
  dim3 grid((a.B + NB - 1) / NB, a.ndir), block(nthr);
  // Opt-in (MMB_LSTM_PAIR=1).  Measured (B = 32, H = 100): 0.62 instead of 0.67 us per step for ONE layer alone -- the step is bound by
  // its dependent chain (LDS -> 52-deep FMA chains -> shuffles -> activations -> barrier), not by issue slots, so halving the warps per
  // scheduler buys 7 % -- but a pair takes 128 SMs per layer and the training step runs three encoders side by side (384 CTAs on 296
  // slots): 5 870 instead of 6 186 videos/s.  Kept as a measured alternative, off by default.  The pair kernel writes neither the
  // dropped output `y` nor trace stamps: a layer with output dropout, or a traced launch, takes the single-CTA kernel below.
  const char* pair_env = getenv("MMB_LSTM_PAIR");
  const bool pair_ok = pair_env && atoi(pair_env) != 0;
  if (!backward && NB == 1 && pair_ok && !a.y && !a.trace && a.H >= 32 && 2 * a.B * a.ndir <= 2 * 148) {
    // two CTAs per (sequence, direction): see bilstm_fwd_pair_kernel
    const int pthr = threads_for(KS / 2 + 1);
    const int UH = (a.H + 1) / 2;
    if (2 * UH <= pthr) {
      const size_t smem = sizeof(float) * (2 * HP + (size_t)RING * 2 * pthr);
      MMB_CUDA(cudaFuncSetAttribute(bilstm_fwd_pair_kernel<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3((unsigned)(2 * a.B), (unsigned)a.ndir);
      cfg.blockDim = dim3((unsigned)pthr);
      cfg.dynamicSmemBytes = smem;
      cfg.stream = stream;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      MMB_CUDA(cudaLaunchKernelEx(&cfg, bilstm_fwd_pair_kernel<KS>, a));
      return check_launch("bilstm_fwd_pair_kernel");
    }
  }
  if (!backward) {
    constexpr int NT = threads_for(KS);
    const size_t smem = sizeof(float) * (2 * NB * HP + (size_t)RING * pow2_ceil(NB * 2 * NT));
    if (NB == 1 && a.trace) {
      MMB_CUDA(cudaFuncSetAttribute(bilstm_fwd_kernel<KS, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      bilstm_fwd_kernel<KS, 1, true><<<grid, NT, smem, stream>>>(a);
      return check_launch("bilstm_fwd_kernel<trace>");
    }
    if (a.y) {
      MMB_CUDA(cudaFuncSetAttribute(bilstm_fwd_kernel<KS, NB, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      bilstm_fwd_kernel<KS, NB, false, true><<<grid, NT, smem, stream>>>(a);
      return check_launch("bilstm_fwd_kernel<dropout>");
    }
    MMB_CUDA(cudaFuncSetAttribute(bilstm_fwd_kernel<KS, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bilstm_fwd_kernel<KS, NB><<<grid, NT, smem, stream>>>(a);
    return check_launch("bilstm_fwd_kernel");
  }
  constexpr int KSP = (KS % 32 == 0) ? KS + 4 : KS;
  const size_t smem = sizeof(float) * (NB * 4 * 2 * KSP + NB * 4 * 2 * BWD_SL + (size_t)RING * NB * 7 * 128);
  constexpr int KR50 = KS == 52 ? 50 : KS;
  if (KS == 52 && a.H <= 100) {                    // the model's hidden size: no padded r values in registers
    if (a.rng_key) {
      MMB_CUDA(cudaFuncSetAttribute(bilstm_bwd_kernel<KS, NB, KR50, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      bilstm_bwd_kernel<KS, NB, KR50, true><<<grid, BWD_NT, smem, stream>>>(a);
      return check_launch("bilstm_bwd_kernel<dropout>");
    }
    MMB_CUDA(cudaFuncSetAttribute(bilstm_bwd_kernel<KS, NB, KR50>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bilstm_bwd_kernel<KS, NB, KR50><<<grid, BWD_NT, smem, stream>>>(a);
    return check_launch("bilstm_bwd_kernel");
  }
  if (a.rng_key) {
    MMB_CUDA(cudaFuncSetAttribute(bilstm_bwd_kernel<KS, NB, KS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bilstm_bwd_kernel<KS, NB, KS, true><<<grid, BWD_NT, smem, stream>>>(a);
    return check_launch("bilstm_bwd_kernel<dropout>");
  }
  MMB_CUDA(cudaFuncSetAttribute(bilstm_bwd_kernel<KS, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bilstm_bwd_kernel<KS, NB><<<grid, BWD_NT, smem, stream>>>(a);
  return check_launch("bilstm_bwd_kernel");
}

int pick_nb(int B, int ndir) {
  // Fewest sequences per CTA that still fits one wave of 148 SMs (latency-bound recurrence).
  return (B * ndir <= 148) ? 1 : 2;
}

int dispatch(const LstmArgs& a, bool backward, cudaStream_t stream) {
  const int nb = pick_nb(a.B, a.ndir);
#define MMB_LSTM_CASE(KS) return nb == 1 ? launch<KS, 1>(a, backward, stream) : launch<KS, 2>(a, backward, stream)
  if (a.H <= 16) { MMB_LSTM_CASE(8); }
  if (a.H <= 64) { MMB_LSTM_CASE(32); }
  if (a.H <= 104) { MMB_LSTM_CASE(52); }
#undef MMB_LSTM_CASE
  set_error("bilstm: hidden size %d > 104 unsupported", a.H);
  return MMB_ERR_UNSUPPORTED;
}

}  // namespace
}  // namespace mmb

static int bilstm_fwd_impl(float* gates, const float* w_hh, const int32_t* lengths, const int32_t* order, float* out, float* y,
                           float* h_n, float* c_n, float* cell, const unsigned long long* rng_key, float keep_prob, int B, int L, int H,
                           int ndir, int save, mmb_stream_t stream, const char* who) {
  MMB_REQUIRE(gates && w_hh && lengths && out && h_n && c_n, MMB_ERR_INVALID, "%s: null pointer", who);
  MMB_REQUIRE(!save || cell, MMB_ERR_INVALID, "%s: save=1 needs a cell buffer", who);
  MMB_REQUIRE(B > 0 && L > 0 && H > 0 && (ndir == 1 || ndir == 2), MMB_ERR_INVALID, "%s: B=%d L=%d H=%d ndir=%d", who, B, L, H, ndir);
  MMB_REQUIRE((y == nullptr) == (rng_key == nullptr), MMB_ERR_INVALID, "%s: y and rng_key go together", who);
  MMB_REQUIRE(!y || (keep_prob > 0.f && keep_prob <= 1.f && (long long)B * L * ndir * H < (1ll << 32)), MMB_ERR_INVALID,
              "%s: keep_prob=%g, or more than 2^32 output elements", who, keep_prob);
  mmb::LstmArgs a{gates, w_hh, lengths, order, out, h_n, c_n, cell, nullptr, nullptr, nullptr, B, L, H, ndir, save, nullptr,
                  y, rng_key, keep_prob};
  static const char* trace_env = getenv("MMB_LSTM_TRACE");                 // debugging aid (tools/lstm_trace.py)
  a.trace = trace_env ? reinterpret_cast<long long*>(strtoull(trace_env, nullptr, 0)) : nullptr;
  return mmb::dispatch(a, false, static_cast<cudaStream_t>(stream));
}

extern "C" int mmb_bilstm_fwd(float* gates, const float* w_hh, const int32_t* lengths, const int32_t* order, float* out,
                              float* h_n, float* c_n, float* cell, int B, int L, int H, int ndir, int save,
                              mmb_stream_t stream) {
  return bilstm_fwd_impl(gates, w_hh, lengths, order, out, nullptr, h_n, c_n, cell, nullptr, 1.f, B, L, H, ndir, save, stream,
                         "mmb_bilstm_fwd");
}

extern "C" int mmb_bilstm_fwd_dropout(float* gates, const float* w_hh, const int32_t* lengths, const int32_t* order, float* out,
                                      float* y, float* h_n, float* c_n, float* cell, const unsigned long long* rng_key,
                                      float keep_prob, int B, int L, int H, int ndir, int save, mmb_stream_t stream) {
  MMB_REQUIRE(y && rng_key, MMB_ERR_INVALID, "mmb_bilstm_fwd_dropout: y / rng_key is null");
  return bilstm_fwd_impl(gates, w_hh, lengths, order, out, y, h_n, c_n, cell, rng_key, keep_prob, B, L, H, ndir, save, stream,
                         "mmb_bilstm_fwd_dropout");
}

static int bilstm_bwd_impl(float* gates, const float* cell, const float* w_hh, const int32_t* lengths, const int32_t* order,
                           const float* dout, const float* dh_n, const float* dc_n, const unsigned long long* rng_key, float keep_prob,
                           int B, int L, int H, int ndir, mmb_stream_t stream, const char* who) {
  MMB_REQUIRE(gates && cell && w_hh && lengths && dout, MMB_ERR_INVALID, "%s: null pointer", who);
  MMB_REQUIRE(B > 0 && L > 0 && H > 0 && (ndir == 1 || ndir == 2), MMB_ERR_INVALID, "%s: B=%d L=%d H=%d ndir=%d", who, B, L, H, ndir);
  MMB_REQUIRE(!rng_key || (keep_prob > 0.f && keep_prob <= 1.f && (long long)B * L * ndir * H < (1ll << 32)), MMB_ERR_INVALID,
              "%s: keep_prob=%g, or more than 2^32 output elements", who, keep_prob);
  mmb::LstmArgs a{gates, w_hh, lengths, order, nullptr, nullptr, nullptr, const_cast<float*>(cell), dout, dh_n, dc_n,
                  B, L, H, ndir, 1, nullptr, nullptr, rng_key, keep_prob};
  return mmb::dispatch(a, true, static_cast<cudaStream_t>(stream));
}

extern "C" int mmb_bilstm_bwd(float* gates, const float* cell, const float* w_hh, const int32_t* lengths,
                              const int32_t* order, const float* dout, const float* dh_n, const float* dc_n, int B, int L,
                              int H, int ndir, mmb_stream_t stream) {
  return bilstm_bwd_impl(gates, cell, w_hh, lengths, order, dout, dh_n, dc_n, nullptr, 1.f, B, L, H, ndir, stream, "mmb_bilstm_bwd");
}

extern "C" int mmb_bilstm_bwd_dropout(float* gates, const float* cell, const float* w_hh, const int32_t* lengths,
                                      const int32_t* order, const float* dy, const float* dh_n, const float* dc_n,
                                      const unsigned long long* rng_key, float keep_prob, int B, int L, int H, int ndir,
                                      mmb_stream_t stream) {
  MMB_REQUIRE(rng_key, MMB_ERR_INVALID, "mmb_bilstm_bwd_dropout: rng_key is null");
  return bilstm_bwd_impl(gates, cell, w_hh, lengths, order, dy, dh_n, dc_n, rng_key, keep_prob, B, L, H, ndir, stream,
                         "mmb_bilstm_bwd_dropout");
}

// ---- the keep mask itself (tests: parity GIVEN the mask) and the key stream ---------------------------------------------------------
namespace mmb {
namespace {
__global__ void dropout_mask_kernel(const unsigned long long* __restrict__ rng_key, float keep_prob, long long n, uint8_t* __restrict__ mask) {
  const unsigned long long key = rng_key[0];
  const uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32), thresh = dropout_thresh(keep_prob);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    mask[i] = dropout_keep((uint32_t)i, k0, k1, thresh) ? 1 : 0;
}
// splitmix64: key_out = mix(state += golden).  One thread; the state lives on the device so that a CUDA-graph replay draws fresh keys.
__global__ void rng_next_kernel(unsigned long long* __restrict__ state, unsigned long long* __restrict__ key_out, int n_keys) {
  unsigned long long s = state[0];
  for (int i = 0; i < n_keys; ++i) {
    s += 0x9E3779B97F4A7C15ull;
    unsigned long long z = s;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    key_out[i] = z ^ (z >> 31);
  }
  state[0] = s;
}
}  // namespace
}  // namespace mmb

extern "C" int mmb_dropout_mask(const unsigned long long* rng_key, float keep_prob, long long n, uint8_t* mask, mmb_stream_t stream) {
  MMB_REQUIRE(rng_key && mask && n > 0 && n < (1ll << 32) && keep_prob > 0.f && keep_prob <= 1.f, MMB_ERR_INVALID,
              "mmb_dropout_mask: bad arguments");
  const long long blocks = (n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184;
  mmb::dropout_mask_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(rng_key, keep_prob, n, mask);
  return mmb::check_launch("dropout_mask_kernel");
}

extern "C" int mmb_rng_next(unsigned long long* state, unsigned long long* key_out, int n_keys, mmb_stream_t stream) {
  MMB_REQUIRE(state && key_out && n_keys > 0, MMB_ERR_INVALID, "mmb_rng_next: bad arguments");
  mmb::rng_next_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(state, key_out, n_keys);
  return mmb::check_launch("rng_next_kernel");
}
