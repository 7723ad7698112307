// Multimodal-attention decoder step (layers/attention.py:145-186), forward, as ONE kernel: north_star (3) -- "the multimodal
// attention and output-layer masked soft-max are fused into one kernel".
//
// The chunk-parallel cut (decoder_step.cu) is five kernels around four library GEMMs: nine dependent launches per step, ~48 us
// of which ~5 us per launch is dependency latency.  Here one thread-block CLUSTER owns one video for the whole step: the CTAs of
// the cluster split the text axis (energies, soft-max partials, contexts, coverage) and the output neurons of the five mat-vecs
// (W2 / W4 / W_beta_2 / W_beta_4 h;  W_beta_1 c1, W_beta_3 c2;  the LSTM gates;  out(h')), and exchange the small vectors in between
// through distributed shared memory (six cluster barriers per step).  Nothing goes through global memory between the stages
// except what the backward pass wants saved.  Videos never interact, so there is no grid-wide synchronisation.
//
//   A  hw = [W2 | W4 | W_beta_2 | W_beta_4] h + folded biases                        (4D outputs, split over the cluster)
//   B  e_k[t] = v_k . tanh(proj_k[t] + hw_k + cov[t] wc_k) + v_k bias; chunk-local soft-max partials and weighted contexts
//      (the un-masked soft-max over the text axis, attention.py:148,154, quirk Q2), merged over the cluster
//   C  pb_k = W_beta_{1,3} c_k (split); beta = soft-max_2; c3 = beta . c; att_cov, coverage', coverage-loss term
//   D  LSTM gates = [W_ih | W_hh] [c3 | sent | h] + b (split by hidden unit), cell update
//   E  logits = out(h') (split), masked soft-max over the M sentences, first-max arg-max, NLL term
//
// fp32 FFMA throughout (warp-per-output mat-vecs with 128-bit loads, warp-shuffle reductions): the step is latency bound, not
// FLOP bound (~0.6 MFLOP per video), and fp32 keeps it inside the 1e-5 tier.
#include <cooperative_groups.h>
#include <stdlib.h>
#include <type_traits>
#include "common.cuh"
#include "tc_common.cuh"     // mbarrier / bulk-copy helpers (mmb::tc)

namespace cg = cooperative_groups;

namespace mmb {
namespace {

constexpr int NT = 512;        // 16 warps: the step is a chain of latency-bound stages, one CTA per SM
constexpr int NW = NT / 32;
constexpr int MAXC = 8;        // cluster sizes 4 and 8
constexpr int SCR = 2048;      // floats of mat-vec scratch in the forward kernel: K slices x outputs of a stage
// hidden units / outputs of a rank: multiples of 4, so that a rank's weight columns start 16-byte aligned (quad form of the mat-vecs)
__host__ __device__ constexpr int split4(int n, int parts) { return ((n + parts - 1) / parts + 3) & ~3; }

__device__ __forceinline__ float rcp_ftz(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Bulk reduction shared -> global (the TMA adds a whole staged block of rows into memory at L2), its group commit / wait
__device__ __forceinline__ void bulk_reduce_add_f32(float* dst, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// Predicated reduction (no branch around it: the sweeps' loop bodies stay one basic block)
__device__ __forceinline__ void red_add_f32_if(float* p, float v, bool on) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %2, 0;\n\t"
      "@q red.global.add.f32 [%0], %1;\n\t"
      "}" ::"l"(p), "f"(v), "r"((int)on)
      : "memory");
}

__device__ long long* g_dec_trace = nullptr;   // debugging aid (MMB_DEC_TRACE): clock64 stamps of block 0 at the stage boundaries
#define DEC_STAMP(i)                                                          \
  do {                                                                        \
    if (g_dec_trace && blockIdx.x == 0 && threadIdx.x == 0) g_dec_trace[i] = clock64(); \
  } while (0)

struct FusedArgs {
  // per sequence
  const float *proj_a, *proj_i, *enc_a, *enc_i;            // (B, Lt, D)
  // weights
  const float *Wh4t, *bh4;                                  // (H, 4D) = Wh4^T, (4D)
  const float *v1, *wc1, *v2, *wc2, *v1b, *v2b;             // (D) x4, (1) x2
  const float *Wb13t;                                       // (2, D, D): [W_beta_1^T; W_beta_3^T]
  const float *vb1, *vb2, *vb1b, *vb2b;
  const float *Wcatt, *bcat;                                // (D+E+H, 4H) = Wcat^T, (4H)
  const float *out_wt, *out_b;                              // (H, M) = out.weight^T, (M)
  // per step inputs
  const float *sent, *h, *cell, *cov;                       // (B,E), (B,H), (B,H), (B,Lt)
  const uint8_t* mask;                                      // (B, M)
  const long long* target;                                  // (B) or null
  // outputs
  float *probs, *h_out, *cell_out, *att_cov, *cov_out;      // (B,M), (B,H), (B,H), (B,Lt), (B,Lt)
  long long* argmax;                                        // (B) or null
  float *nll, *cov_loss;                                    // (B) or null
  // saved for the backward pass (all required)
  float *hw, *alpha, *beta, *ctx12, *pb, *xcat, *gates;     // (B,4D), (B,2,Lt), (B,2), (2,B,D), (2,B,D), (B,D+E+H), (B,4H)
  int B, Lt, D, H, E, M, chunk;
  int stage_off;   // float offset of the row stage in dynamic shared memory ([2 mbarriers][2][chunk * D]), or 0: rows read from L2
  int ctx_vec4;    // 1: the weighted contexts read enc_a / enc_i rows as float4 (D % 4 == 0 and both 16-byte aligned), 0: as floats
};

// y[i] = sum_k Wt[k][col_of(i)] x[k] + bias[col_of(i)] for i < n_out, with the weights TRANSPOSED (Wt (K, ldn): consecutive threads read
// consecutive outputs, no shuffle reductions).  The K axis is split over thread groups whose partial sums meet in shared memory
// (`scratch`, scratch_cap floats).  The stage is a latency problem, not a bandwidth one: every cluster reads the same weights from L2
// (~1 000 cycles per round trip) and what counts is the BYTES IN FLIGHT per SM.
//  * scalar form: one thread per (output, K slice), sixteen 4-byte loads in flight per thread (32 KB per SM);
//  * quad form (`quads`: n_out, ldn and col_of(4 q) are multiples of 4, col_of(4 q + e) = col_of(4 q) + e): one thread per (four outputs,
//    K slice), sixteen 16-byte loads in flight per thread and as many K slices as the scratch holds.  Measured (stamps inside stage D,
//    profiles/r02_decoder_fused.md): a batch of 129 KB per SM takes ~2 900 cycles = 44 B/clk, close to what the L1 / L2 path of one SM
//    delivers -- the stages are bound by the BYTES a CTA pulls (every cluster re-reads the step's weights), not by latency or width.
template <typename ColOf, typename Emit>
__device__ __forceinline__ void block_matvec_t(const float* __restrict__ Wt, const int ldn, const float* __restrict__ bias, const float* x,
                                               const int K, const int n_out, float* scratch, const int scratch_cap, bool quads,
                                               ColOf col_of, Emit emit) {
  const int tid = threadIdx.x;
  if (n_out <= 0) return;
  quads = quads && ((ldn | n_out) & 3) == 0 && (reinterpret_cast<uintptr_t>(Wt) & 15) == 0 && scratch_cap >= 2 * n_out;
  if (quads) {                                                      // (uniform over the block)
    const int nq = n_out >> 2;
    const int S = max(1, min(min(NT / nq, scratch_cap / n_out), K));
    const int q = tid % nq, sl = tid / nq;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (sl < S) {
      const int per = (K + S - 1) / S, k0 = min(K, sl * per), k1 = min(K, k0 + per);
      const float4* w = reinterpret_cast<const float4*>(Wt + (size_t)k0 * ldn + col_of(4 * q));
      const size_t ld4 = (size_t)(ldn >> 2);
      // sixteen independent 16-byte loads in flight per thread, ALL issued before the first FMA: a K slice of up to sixteen rows (the
      // usual case: the slices are as many as the scratch holds) is ONE L2 round trip -- a batch of eight plus a tail was two
      for (int k = k0; k < k1; k += 16) {
        float4 wv[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) wv[u] = k + u < k1 ? __ldcg(w + u * ld4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          const float xv = k + u < k1 ? x[k + u] : 0.f;
          acc.x = fmaf(wv[u].x, xv, acc.x); acc.y = fmaf(wv[u].y, xv, acc.y);
          acc.z = fmaf(wv[u].z, xv, acc.z); acc.w = fmaf(wv[u].w, xv, acc.w);
        }
        w += 16 * ld4;
      }
    }
    __syncthreads();                                                // scratch may still be read from the previous use
    if (sl < S) *reinterpret_cast<float4*>(scratch + sl * n_out + 4 * q) = acc;
    __syncthreads();
    if (tid < n_out) {
      float v = 0.f;
      for (int p = 0; p < S; ++p) v += scratch[p * n_out + tid];
      const int c = col_of(tid);
      emit(tid, v + (bias ? __ldg(bias + c) : 0.f));
    }
    return;
  }
  const int S = max(1, min(min(NT / n_out, scratch_cap / n_out), 32));   // K slices
  const int i = tid % n_out, sl = tid / n_out;
  float acc = 0.f;
  if (sl < S) {
    const int per = (K + S - 1) / S, k0 = min(K, sl * per), k1 = min(K, k0 + per);
    const float* w = Wt + (size_t)k0 * ldn + col_of(i);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int k = k0;
    for (; k + 16 <= k1; k += 16) {                                 // sixteen independent loads in flight per thread
      float wv[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) wv[u] = __ldcg(w + (size_t)u * ldn);
#pragma unroll
      for (int u = 0; u < 16; u += 4) {
        a0 = fmaf(wv[u], x[k + u], a0); a1 = fmaf(wv[u + 1], x[k + u + 1], a1);
        a2 = fmaf(wv[u + 2], x[k + u + 2], a2); a3 = fmaf(wv[u + 3], x[k + u + 3], a3);
      }
      w += (size_t)16 * ldn;
    }
    if (k + 8 <= k1) {
      float wv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) wv[u] = __ldcg(w + (size_t)u * ldn);
#pragma unroll
      for (int u = 0; u < 8; u += 4) {
        a0 = fmaf(wv[u], x[k + u], a0); a1 = fmaf(wv[u + 1], x[k + u + 1], a1);
        a2 = fmaf(wv[u + 2], x[k + u + 2], a2); a3 = fmaf(wv[u + 3], x[k + u + 3], a3);
      }
      w += (size_t)8 * ldn;
      k += 8;
    }
    for (; k < k1; ++k) {
      a0 = fmaf(__ldcg(w), x[k], a0);
      w += ldn;
    }
    acc = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();                                                  // scratch may still be read from the previous use
  if (sl < S && S > 1) scratch[sl * n_out + i] = acc;
  __syncthreads();
  if (tid < n_out) {
    float v = acc;                                                  // slice 0 (sl == 0 for tid < n_out)
    for (int q = 1; q < S; ++q) v += scratch[q * n_out + tid];
    const int c = col_of(tid);
    emit(tid, v + (bias ? __ldg(bias + c) : 0.f));
  }
}

__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = lane < NW ? red[lane] : 0.f;
  return warp_sum(r);
}
__device__ __forceinline__ float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = lane < NW ? red[lane] : -INFINITY;
  return warp_max(r);
}

// The greedy roll-out (mmb_decoder_greedy_fused): the same stages, `steps` times in one launch, in eval mode (models.py:156-199, the
// `else` branches).  The step inputs come from on chip instead of global memory: h = the gathered h' of the previous step (s_hn), the
// cell of a rank's own hidden units (a register of the thread that owns the unit), the coverage of its own text rows (s_cov += att),
// sent = emb_text[b, the previous step's arg-max] (every rank reduces the arg-max candidates itself).  Step 0 starts from h0 and a
// zero cell, coverage and input row (models.py:145-149).  Nothing the backward pass would want is written.
struct GreedyArgs {
  const float *emb_text, *h0;                               // (B, Lt, E), (B, H)
  int steps, T;                                             // roll-out length S; row stride of the target (B, T), T >= S
};

// The beam roll-out (mmb_decoder_beam_fused): the greedy roll-out with K slots per video (include/mmbidaf_b200.h states the rule).  The
// live slots of a step run the stages one after another, each from its own state, so every per-hypothesis value is the step kernel's to
// the bit; what the slots hold between the steps sits in shared memory behind the base arrays (`off`): the table (score, last token,
// status), h / cell / coverage of every slot (this step's inputs and outputs), this rank's share of every slot's distribution and the
// selection exchange.  Each rank ranks its own (slot, sentence) candidates, keeps its best K and publishes them to every rank through
// DSMEM; every rank merges the CL x K entries and the carries of the finished slots in the same order, so all agree on the new table.
constexpr int MAXK = 8;
struct BeamArgs {
  const int* text_len;                                      // (B): the EOS row of video b is text_len[b] - 1
  long long* tokens;                                        // (B, S, K)
  int* parents;                                             // (B, S, K)
  float *scores, *probs;                                    // (B, S, K), (B, S, K, M)
  long long* best;                                          // (B, S): the tokens of slot 0's path after the last step
  int* path;                                                // (B, S): the slot of that path at every step
  int K, off;                                               // width; float offset of the beam region in dynamic shared memory
};
enum : int { kEmpty = 0, kLive = 1, kDone = 2 };

// Constrained roll-outs (mmb_decoder_greedy_constrained_fused / mmb_decoder_beam_constrained_fused; include/mmbidaf_b200.h states the
// rule): the pick of a step -- the greedy arg-max, the beam candidates -- skips sentences that are not eligible.  A hypothesis keeps its
// eligible-sentence bits of this rank's sentences (set for m <= EOS with the mask set; a pick m < EOS clears its own bit under
// no_repeat) and `kept`, its picks below EOS so far.  Greedy: one register per thread, bit j for sentence m0 + tid + j NT (every
// thread learns the pick).  Beam: ceil(ldp / 32) words per slot in shared memory, gathered by parent beside h / cell / coverage.
struct ConstraintArgs {
  const int* text_len;                                      // (B): the EOS row of video b is text_len[b] - 1
  int no_repeat, min_sentences;
};
// the EOS row is eligible once the hypothesis holds min_sentences sentences, or has no other sentence left to add
__device__ __forceinline__ bool eos_allowed(const ConstraintArgs& cn, int eos, int kept) {
  return kept >= cn.min_sentences || eos - (cn.no_repeat ? kept : 0) == 0;
}

// the ranking of the candidates: score descending, then step probability descending, then parent slot, then sentence ascending
__device__ __forceinline__ bool cand_better(float sa, float pa, int ka, int ma, float sb, float pb, int kb, int mb) {
  if (sa != sb) return sa > sb;
  if (pa != pb) return pa > pb;
  if (ka != kb) return ka < kb;
  return ma < mb;
}
// the best candidate of the warp, in every lane
__device__ __forceinline__ void cand_warp_best(float& s, float& p, int& k, int& m) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float s2 = __shfl_xor_sync(0xffffffffu, s, o), p2 = __shfl_xor_sync(0xffffffffu, p, o);
    const int k2 = __shfl_xor_sync(0xffffffffu, k, o), m2 = __shfl_xor_sync(0xffffffffu, m, o);
    if (cand_better(s2, p2, k2, m2, s, p, k, m)) { s = s2; p = p2; k = k2; m = m2; }
  }
}
// Sampled roll-outs (mmb_decoder_sample_fused; include/mmbidaf_b200.h states the rule): the greedy roll-out, or the constrained one,
// with the pick drawn by Gumbel-max over the candidates instead of the arg-max.  Cluster r runs sample r % N of video r / N.  With
// top_k > 0 the candidates are the best top_k by (p descending, m ascending), found after stage E by the beam's selection (each rank's
// best top_k, then the merge of every rank's); the beam region's exchange arrays (`off`) hold them.
struct SampleArgs {
  const unsigned long long* key;                            // (1) on the device
  float T;                                                  // temperature > 0
  int N, top_k, off;                                        // samples per video; 0 or 1..MAXK; float offset of the exchange arrays
};
// The cluster's index in the grid (blockIdx.x / cluster size): in the sampled roll-out, roll-out b N + n.  Read where used (the
// volatile read is not held in a register over the stages).
__device__ __forceinline__ int cluster_row() {
  unsigned r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return (int)r;
}
// z of counter c (common.cuh::sample_score) with the key loaded and 1 / T formed where the pick is drawn (the volatile load keeps the
// compiler from hoisting it into a register held over the step)
__device__ __forceinline__ float sample_z(const SampleArgs& sp, float p, uint32_t c) {
  unsigned long long key;
  asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(key) : "l"(sp.key));
  return sample_score(p, 1.f / sp.T, c, (uint32_t)key, (uint32_t)(key >> 32));
}

// Nucleus roll-outs (mmb_decoder_sample_nucleus_fused; include/mmbidaf_b200.h states the rule): the sampled roll-out with the draw
// limited to the nucleus, the first n candidates in (p descending, m ascending) order whose integer masses q = floor(p 2^24) reach
// need = ceil(P Q / 2^24).  With top_k = 0 every rank writes its candidates' p into every rank's copy of the row (`off`: [M] floats,
// -1 for a non-candidate) and, after one cluster barrier, each rank cuts the same row by itself (nucleus_cut); with top_k > 0 the
// cut is a prefix of the merged top_k entries.
struct NucleusArgs {
  uint32_t P;                                               // rint(top_p 2^24), below 2^24 (top_p = 1 runs dec_sample_kernel)
  int off;                                                  // float offset of the nucleus region (nucleus_floats)
};
constexpr int kNucBuckets = 256;                            // radix digits of 8 bits, four passes over the bits of p

// Stochastic beam roll-outs (mmb_decoder_beam_sample_fused; include/mmbidaf_b200.h states the rule): the beam roll-out with every
// candidate ranked by its key -- its Gumbel-perturbed log-probability under the renormalised, tempered step distribution, truncated
// below its parent's key -- instead of its score.  Per slot the table also keeps phi (the path's log-probability under that
// distribution) and its key.  Before the selection three cluster exchanges per step give every live slot k its normaliser (mu_k, then
// the integer mass Q_k) and the largest perturbed child Z_k; each rank then writes its candidates' keys into `off` and the beam's
// selection runs on them.  The selection keeps K + 1 entries: the (K + 1)-th is the best key pruned at that step, and the threshold
// kappa is the largest of them over the steps (every pruned subtree holds a sequence with exactly its root's key, and no larger one).
struct StochArgs {
  const unsigned long long* key;                            // (1) on the device
  float T;                                                  // temperature > 0
  float *phi, *keys;                                        // (B, S, K)
  long long* paths;                                         // (B, K, S): every final slot's tokens (eos for an empty slot)
  int* path_slots;                                          // (B, K, S): its slot at every step (-1 for an empty slot)
  float* kappa;                                             // (B)
  int off;                                                  // float offset of the stochastic region (stoch_floats)
};
__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  unsigned long long* r = reinterpret_cast<unsigned long long*>(red);   // (NW words: 32 floats)
  __syncthreads();
  if (lane == 0) r[warp] = v;
  __syncthreads();
  unsigned long long t = lane < NW ? r[lane] : 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  return t;
}
// log(1 - e^a) for a <= 0, and the key of a child whose perturbed log-probability is G, under its parent's key kp and the largest
// perturbed child Z (Kool et al. 2019, appendix B.3): at G = Z, v = -inf and the key is kp exactly
__device__ __forceinline__ float log1mexpf(float a) { return a > -0.693147182f ? logf(-expm1f(a)) : log1pf(-expf(a)); }
__device__ __forceinline__ float truncated_key(float kp, float G, float Z) {
  const float v = (kp - G) + log1mexpf(G - Z);
  return (kp - fmaxf(v, 0.f)) - log1pf(expf(-fabsf(v)));
}

// The nucleus of row v[0..M) (v[m] = p, or -1 for a non-candidate), in every thread of the block: its boundary p* (as bits) and m*, so
// that the nucleus is {m : v[m] > p*} + {m : v[m] == p*, m <= m*}.  The masses are integers, so every sum below is exact in any order:
// each rank of the cluster cuts its copy of the row to the same set.
//  * need = 0 (P Q < 2^24, Q = 0 included): the first candidate, the largest p with the smallest m (n = 1).
//  * else p* is radix-selected on the bits of p (monotone for p >= 0), top digit first: a pass histograms the mass q of the candidates
//    under the prefix found so far by digit, and takes the digit where the mass from above reaches what is still needed (`rem`).
//    Candidates with q = 0 are never needed: the mass is reached at a candidate with q* > 0.  Then ceil(rem / q*) ties at p* are
//    needed, and m* is the m of the last of them, found by a block prefix count over contiguous m ranges.
// hist: kNucBuckets u64; red: 32 u64 (warp totals and broadcasts).  Ends behind a block barrier.
struct NucleusCut {
  uint32_t pstar;                                           // bits of p*
  int mstar;                                                // -1: no candidate
};
__device__ __forceinline__ NucleusCut nucleus_cut(const float* __restrict__ v, int M, uint32_t P, unsigned long long* hist,
                                                  unsigned long long* red) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t prefix = 0, pmask = 0;
  unsigned long long rem = 0;
  bool first = false;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    if (tid < kNucBuckets) hist[tid] = 0ull;
    __syncthreads();
    // (flat rows put most candidates under one digit: the lanes of a digit add their masses first, one shared atomic per digit and
    // warp instead of one per candidate -- a warp's masses stay below 2^29)
    for (int m0 = 0; m0 < M; m0 += NT) {
      const int m = m0 + tid;
      const float p = m < M ? v[m] : -1.f;
      const uint32_t bits = __float_as_uint(p);
      uint32_t q = __float2uint_rz(p * 16777216.f);                    // (a non-candidate's -1 gives q = 0)
      const bool in = q != 0u && (bits & pmask) == prefix;
      const uint32_t digit = in ? (bits >> shift) & (kNucBuckets - 1) : kNucBuckets;
      q = in ? q : 0u;
      const uint32_t peers = __match_any_sync(0xffffffffu, digit);
      const uint32_t sum = __reduce_add_sync(peers, q);
      if (in && lane == __ffs(peers) - 1) atomicAdd(hist + digit, (unsigned long long)sum);
    }
    __syncthreads();
    // suffix sums: thread t < 256 holds digit 255 - t, an inclusive scan over the threads
    const unsigned long long h = tid < kNucBuckets ? hist[kNucBuckets - 1 - tid] : 0ull;
    unsigned long long s = h;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += t;
    }
    if (lane == 31 && warp < kNucBuckets / 32) red[warp] = s;
    __syncthreads();
    unsigned long long below = 0, total = 0;
    for (int w = 0; w < kNucBuckets / 32; ++w) {
      below += w < warp ? red[w] : 0ull;
      total += red[w];
    }
    s += below;
    if (pass == 0) {                                         // total = Q, the same in every thread
      const unsigned long long pq = (unsigned long long)P * total;
      rem = (pq >> 24) + ((pq & 0xffffffull) != 0ull);       // need
      if (rem == 0ull) { first = true; break; }
    }
    if (tid < kNucBuckets && s - h < rem && rem <= s) {     // the one digit where the mass from above reaches rem
      red[8] = (unsigned long long)(kNucBuckets - 1 - tid);
      red[9] = rem - (s - h);
    }
    __syncthreads();
    prefix |= (uint32_t)red[8] << shift;
    pmask |= (uint32_t)(kNucBuckets - 1) << shift;
    rem = red[9];
  }
  unsigned long long ties = 1;
  if (first) {                                               // the largest p over the candidates (0 bits also when there is none)
    uint32_t mx = 0;
    for (int m = tid; m < M; m += NT) {
      const float p = v[m];
      if (p >= 0.f) mx = max(mx, __float_as_uint(p));
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    __syncthreads();
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    prefix = 0;
    for (int w = 0; w < NW; ++w) prefix = max(prefix, (uint32_t)red[w]);
  } else {
    const unsigned long long qs = __float2uint_rz(__uint_as_float(prefix) * 16777216.f);
    ties = (rem + qs - 1) / qs;
  }
  // m*: the ties-th m (ascending) with v[m] == p*; thread t counts the ties in its range [t c, t c + c)
  const int c = (M + NT - 1) / NT, lo = min(M, tid * c), hi = min(M, lo + c);
  int cnt = 0;
  for (int m = lo; m < hi; ++m) cnt += __float_as_uint(v[m]) == prefix;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  __syncthreads();                                           // red is read above
  if (lane == 31) red[warp] = (unsigned long long)incl;
  if (tid == 0) red[NW] = ~0ull;                             // m* = -1 when there is no candidate at all
  __syncthreads();
  unsigned long long excl = (unsigned long long)(incl - cnt);
  for (int w = 0; w < warp; ++w) excl += red[w];
  if (excl < ties && ties <= excl + (unsigned long long)cnt) {
    unsigned long long k = excl;
    for (int m = lo; m < hi; ++m)
      if (__float_as_uint(v[m]) == prefix && ++k == ties) red[NW] = (unsigned long long)m;
  }
  __syncthreads();
  const NucleusCut cut{prefix, (int)(long long)red[NW]};
  __syncthreads();                                           // red is free again
  return cut;
}

// kGreedy: the roll-out; kBeam (with kGreedy): the beam roll-out instead of the greedy one; kConstrained (with kGreedy): the pick skips
// the sentences `cn` makes ineligible; kSample (with kGreedy, not kBeam): the pick is drawn (`sp`); kNucleus (with kSample): drawn
// from the nucleus (`nu`); kStoch (with kBeam): the stochastic beam (`st`)
template <bool kGreedy, bool kBeam = false, bool kConstrained = false, bool kSample = false, bool kNucleus = false, bool kStoch = false>
__device__ __forceinline__ void dec_fused_body(const FusedArgs& a, const GreedyArgs& g, const BeamArgs& bm, const ConstraintArgs& cn,
                                               const SampleArgs sp, const NucleusArgs nu = NucleusArgs{}, const StochArgs st = StochArgs{}) {
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = (int)cluster.num_blocks(), R = (int)cluster.block_rank();
  const int ob = blockIdx.x / CL;                         // the output row: the video (sampled: cluster_row(), the roll-out)
  const int b = kSample ? cluster_row() / sp.N : ob;      // the video whose inputs the cluster reads
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = a.D, H = a.H, E = a.E, M = a.M, Lt = a.Lt, K = D + E + H;

  extern __shared__ __align__(16) float smem[];
  auto up4 = [](int v) { return (v + 3) & ~3; };        // every array starts 16-byte aligned
  float* s_hw = smem;                       // [4D]   full, gathered over the cluster
  float* s_x = s_hw + up4(4 * D);           // [K]    xcat = [c3 | sent | h]
  float* s_ctx = s_x + up4(K);              // [2D]   merged contexts
  float* s_pb = s_ctx + up4(2 * D);         // [2D]   gathered
  float* s_hn = s_pb + up4(2 * D);          // [H]    h', gathered
  float* s_part = s_hn + up4(H);            // [MAXC][4 + 2D] soft-max partials of every rank (written remotely)
  float* s_ex = s_part + up4(MAXC * (4 + 2 * D));   // [MAXC][8] small exchanges: coverage loss, soft-max (max, sum), arg-max (p, index)
  float* s_g = s_ex + MAXC * 8;             // [4][ceil(H / CL) + 1] gate pre-activations of this rank's units
  float* s_red = s_g + up4(4 * (split4(H, MAXC / 2) + 1));   // [32]   (sized for the smaller cluster)
  float* s_scr = s_red + 32;                // [SCR]  K-slice partial sums of the mat-vecs
  float* s_vec = s_scr + SCR;               // [4D]   v1 | wc1 | v2 | wc2
  float* s_e = s_vec + up4(4 * D);          // [2][chunk] energies -> p -> alpha of this rank's rows
  float* s_cov = s_e + up4(2 * a.chunk);    // [chunk] coverage input of this rank's rows
  float* s_cpart = s_cov + up4(a.chunk);    // [groups][2][D] context partials inside the block; later this rank's logits

  // Row stage (stage_off != 0): this rank's rows of proj_a / proj_i -- contiguous in memory -- are brought into shared memory by two
  // bulk copies issued NOW, a whole mat-vec stage and a cluster barrier before stage B reads them; when the energies are done the same
  // buffers take the rows of enc_a / enc_i for the weighted contexts (under the chunk-local soft-max).  Without it stage B was two
  // rounds of (issue a warp's loads from L2, wait, compute): 17 k cycles for energies whose MUFU floor is ~5 k (profiles/r02_decoder_fused.md).
  const int t0 = min(Lt, R * a.chunk), t1 = min(Lt, t0 + a.chunk), n = t1 - t0;
  const bool staged = a.stage_off != 0;
  float* const s_st0 = smem + a.stage_off + 4;
  float* const s_st1 = s_st0 + up4(a.chunk * D);
  const uint32_t bar_proj = tc::smem_u32(smem + a.stage_off), bar_enc = bar_proj + 8;
  const uint32_t stage_bytes = (uint32_t)(n * D) * 4u;
  if (staged && tid == 0) {
    tc::mbar_init(bar_proj, 1);
    tc::mbar_init(bar_enc, 1);
    tc::fence_barrier_init();
    if (n > 0) {
      tc::mbar_expect_tx(bar_proj, 2 * stage_bytes, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st0), a.proj_a + ((size_t)b * Lt + t0) * D, stage_bytes, bar_proj, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st1), a.proj_i + ((size_t)b * Lt + t0) * D, stage_bytes, bar_proj, 1);
    }
  }
  DEC_STAMP(0);
  const int S = kGreedy ? g.steps : 1;
  float cell_own = 0.f;                    // greedy: the cell of hidden unit j0 + tid (stage D), carried between the steps
  int pick = 0;                            // greedy: the previous step's arg-max
  // beam: the region behind the base arrays (beam_floats)
  const int KW = kBeam ? bm.K : 1;
  const int ldh = up4(H), ldc = up4(split4(H, CL)), ldv = up4(a.chunk), ldp = up4((M + CL - 1) / CL);
  float* const bs_score = smem + (kSample ? sp.off : bm.off);            // [MAXK] the table: score,
  int* const bs_tok = reinterpret_cast<int*>(bs_score + MAXK);           // [MAXK]   last token,
  int* const bs_stat = bs_tok + MAXK;                                    // [MAXK]   status
  float* const nt_score = bs_score + 3 * MAXK;                           // [MAXK] the next table: score,
  int* const nt_tok = reinterpret_cast<int*>(nt_score + MAXK);           // [MAXK]   token,
  int* const nt_par = nt_tok + MAXK;                                     // [MAXK]   parent slot (-1: empty),
  int* const nt_kind = nt_par + MAXK;                                    // [MAXK]   status
  constexpr int CS = kStoch ? MAXK + 1 : MAXK;  // exchange entries per rank (stochastic: K + 1, the best pruned key)
  float* const s_cand = nt_score + 4 * MAXK;    // [MAXC][CS][4] every rank's best K (score, p, parent, sentence), written remotely
  float* const s_wred = s_cand + MAXC * CS * 4;                          // [NW][4] per-warp bests
  float* const s_loc = s_wred + NW * 4;                                  // [CS][4] this rank's best K
  float* const s_bh = s_loc + CS * 4;                                    // [K][ldh] h of every slot (the step's input)
  float* const s_bhn = s_bh + KW * ldh;                                  // [K][ldh] h' of every slot
  float* const s_bc = s_bhn + KW * ldh;                                  // [K][ldc] cell of this rank's hidden units, in
  float* const s_bcn = s_bc + KW * ldc;                                  //          and out
  float* const s_bcv = s_bcn + KW * ldc;                                 // [K][ldv] coverage of this rank's text rows, in
  float* const s_bcvn = s_bcv + KW * ldv;                                //          and out
  float* const s_bp = s_bcvn + KW * ldv;                                 // [K][ldp] the distribution over this rank's sentences
  const int eos = kBeam ? bm.text_len[b] - 1 : kConstrained ? cn.text_len[b] - 1 : 0;
  int runs = 0;                                                          // beam: slot runs so far (row-stage barrier phases)
  // constrained: this rank's sentences [e_m0, e_m1) of stage E; a sentence is eligible to start with when its mask is set and it
  // is not past EOS
  const int e_per = (M + CL - 1) / CL, e_m0 = min(M, R * e_per), e_m1 = min(M, e_m0 + e_per);
  auto allowed0 = [&](int m) { return m < e_m1 && m <= eos && a.mask[(size_t)b * M + m] != 0; };
  const int ldu = (ldp + 31) / 32;                                       // beam: words of eligible bits per slot
  uint32_t* bu_cur = reinterpret_cast<uint32_t*>(s_bp + KW * ldp);       // [K][ldu] eligible bits of every slot, in
  uint32_t* bu_nxt = bu_cur + KW * ldu;                                  //          and out (swapped after each selection)
  int* bk_cur = reinterpret_cast<int*>(bu_nxt + KW * ldu);               // [MAXK] kept of every slot, in
  int* bk_nxt = bk_cur + MAXK;                                           //        and out
  uint32_t allow = 0;                                                    // greedy: eligible bits of this thread's sentences
  int kept = 0;                                                          // greedy: picks below EOS so far
  // sampled: the key's halves and 1 / T.  The unconstrained roll-out holds them in registers; the constrained one, which also holds
  // its eligible bits and kept count, forms them where a pick is drawn (sample_z): held, they take it past the 128 registers of a
  // 512-thread CTA, and it spills
  uint32_t key0 = 0, key1 = 0;
  float inv_t = 1.f;
  if constexpr (kSample && !kConstrained) {
    const unsigned long long key = *sp.key;
    key0 = (uint32_t)key;
    key1 = (uint32_t)(key >> 32);
    inv_t = 1.f / sp.T;
  }
  if constexpr (kConstrained && !kBeam) {
    for (int m = e_m0 + tid, j = 0; m < e_m1; m += NT, ++j)
      if (allowed0(m)) allow |= 1u << j;
  }
  if constexpr (kConstrained && kBeam) {   // slot 0: every sentence allowed to start with, nothing kept
    for (int w = warp; w < ldu; w += NW) {
      const uint32_t v = __ballot_sync(0xffffffffu, allowed0(e_m0 + 32 * w + lane));
      if (lane == 0) bu_cur[w] = v;
    }
    if (tid == 0) bk_cur[0] = 0;
  }
  if constexpr (kBeam) {                   // before step 0: slot 0 live with score 0, h0 and a zero cell and coverage; the rest empty
    if (tid < MAXK) {
      bs_score[tid] = tid == 0 ? 0.f : -INFINITY;
      bs_tok[tid] = -1;
      bs_stat[tid] = tid == 0 ? kLive : kEmpty;
      if constexpr (kStoch) {              // slot 0: phi 0 and the key G_0 ~ Gumbel(0), of the counter B S K M + b
        float k0 = -INFINITY;
        if (tid == 0) {
          const unsigned long long key = *st.key;
          const uint32_t c = (uint32_t)a.B * (uint32_t)S * (uint32_t)KW * (uint32_t)M + (uint32_t)b;
          const float u = ((float)(hash32(c, (uint32_t)key, (uint32_t)(key >> 32)) >> 9) + 0.5f) * 1.1920928955078125e-7f;
          k0 = -logf(-logf(u));
        }
        smem[st.off + tid] = tid == 0 ? 0.f : -INFINITY;
        smem[st.off + MAXK + tid] = k0;
      }
    }
    for (int i = tid; i < H; i += NT) s_bh[i] = g.h0[(size_t)b * H + i];
    for (int i = tid; i < ldc; i += NT) s_bc[i] = 0.f;
    for (int i = tid; i < n; i += NT) s_bcv[i] = 0.f;
    __syncthreads();
  }
  for (int s = 0; s < S; ++s) {
  for (int slot = 0; slot < KW; ++slot) {  // beam: the live slots one after another; otherwise once
  if (kBeam && bs_stat[slot] != kLive) continue;
  const uint32_t parity = kBeam ? (uint32_t)(runs & 1) : kGreedy ? (uint32_t)(s & 1) : 0u;   // each row-stage barrier completes once per run
  // ---- stage 0: this video's step inputs -----------------------------------------------------------------------------------
  if constexpr (!kGreedy) {
    for (int i = tid; i < n; i += NT) s_cov[i] = a.cov[(size_t)b * Lt + t0 + i];      // (read per row by the energies: not a global load there)
    for (int i = tid; i < H; i += NT) s_x[D + E + i] = a.h[(size_t)b * H + i];
    for (int i = tid; i < E; i += NT) s_x[D + i] = a.sent[(size_t)b * E + i];
  } else if constexpr (kBeam) {
    for (int i = tid; i < n; i += NT) s_cov[i] = s_bcv[slot * ldv + i];
    for (int i = tid; i < H; i += NT) s_x[D + E + i] = s_bh[slot * ldh + i];
    const float* row = g.emb_text + ((size_t)b * Lt + min(max(bs_tok[slot], 0), Lt - 1)) * E;
    for (int i = tid; i < E; i += NT) s_x[D + i] = s == 0 ? 0.f : row[i];
  } else {
    if (s == 0)
      for (int i = tid; i < n; i += NT) s_cov[i] = 0.f;
    for (int i = tid; i < H; i += NT) s_x[D + E + i] = s == 0 ? g.h0[(size_t)b * H + i] : s_hn[i];
    // (the pick is below Lt whenever the mask is the text mask; a mask wider than the text could point past it: its last row is read)
    // (constrained: a pick of EOS = -1, text_len 0, reads row 0)
    const float* row = g.emb_text + ((size_t)b * Lt + min(kConstrained ? max(pick, 0) : pick, Lt - 1)) * E;
    for (int i = tid; i < E; i += NT) s_x[D + i] = s == 0 ? 0.f : row[i];
  }
  if (!kGreedy || s == 0)
    for (int i = tid; i < D; i += NT) {
      s_vec[i] = a.v1[i];
      s_vec[D + i] = a.wc1[i];
      s_vec[2 * D + i] = a.v2[i];
      s_vec[3 * D + i] = a.wc2[i];
    }
  __syncthreads();

  DEC_STAMP(1);
  // ---- stage A: hw = Wh4 h + bh4, outputs split over the ranks, gathered in every rank ------------------------------------
  {
    const int per = (4 * D + CL - 1) / CL, o0 = R * per, o1 = min(4 * D, o0 + per);
    block_matvec_t(a.Wh4t, 4 * D, a.bh4, s_x + D + E, H, o1 - o0, s_scr, SCR, (o0 & 3) == 0, [&](int i) { return o0 + i; }, [&](int i, float v) {
      const int o = o0 + i;
      for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_hw, r)[o] = v;
      if constexpr (!kGreedy) a.hw[(size_t)b * 4 * D + o] = v;
    });
  }
  DEC_STAMP(2);
  cluster.sync();
  DEC_STAMP(3);

  // ---- stage B: energies of this rank's rows, chunk-local soft-max partials and contexts ----------------------------------
  {
    const float v1b = a.v1b[0], v2b = a.v2b[0];
    // pa0 / pi0: row 0 of this rank's chunk (shared-memory stage or global memory: one instantiation per address space).
    // The loop is written for the issue slots (round 2: the first version left the `d < D` test as a divergent branch around every
    // element and re-read its six step constants from shared memory per element -- ~35 instructions and a BSSY / BSYNC pair per two
    // tanh, 16.8 k cycles for a stage whose MUFU floor is 5.2 k): the constants of a lane's NJ columns live in REGISTERS for the whole
    // stage, pre-scaled so that the pre-activation is the ex2 argument directly (tanh x = 1 - 2 / (1 + 2^(2 x log2 e))); columns past D
    // carry v = 0 and a zero row value, so nothing in the body is predicated; ex2 / rcp are the flush-to-zero MUFU forms (no denormal
    // guard instructions; a flushed 2^x is 0 beside the 1 it is added to).
    constexpr float K2 = 2.0f * 1.4426950408889634f;
    auto energies = [&](const float* __restrict__ pa0, const float* __restrict__ pi0, auto nj_tag, auto ru_tag) {
      constexpr int NJ = decltype(nj_tag)::value, RU = decltype(ru_tag)::value;
      float va[NJ], ha[NJ], wa[NJ], vi[NJ], hi[NJ], wi[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const int d = lane + 32 * j;
        const bool in = d < D;
        const int dd = in ? d : 0;
        va[j] = in ? s_vec[dd] : 0.f;
        wa[j] = in ? s_vec[D + dd] * K2 : 0.f;
        ha[j] = in ? s_hw[dd] * K2 : 0.f;
        vi[j] = in ? s_vec[2 * D + dd] : 0.f;
        wi[j] = in ? s_vec[3 * D + dd] * K2 : 0.f;
        hi[j] = in ? s_hw[D + dd] * K2 : 0.f;
      }
      const float* const covp = s_cov;
      for (int i = warp * RU; i < n; i += NW * RU) {
        float s[RU][2];
        float pav[RU][NJ], piv[RU][NJ], cvs[RU];
#pragma unroll
        for (int u = 0; u < RU; ++u) {         // loads first (memory-level parallelism)
          s[u][0] = s[u][1] = 0.f;
          const int r = min(i + u, n - 1);
          const float* pa = pa0 + (size_t)r * D;
          const float* pi = pi0 + (size_t)r * D;
          cvs[u] = covp[r];
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const int d = lane + 32 * j;
            pav[u][j] = d < D ? pa[d] : 0.f;
            piv[u][j] = d < D ? pi[d] : 0.f;
          }
        }
#pragma unroll
        for (int u = 0; u < RU; ++u) {
          const float cv = cvs[u];
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const float x1 = fmaf(cv, wa[j], fmaf(pav[u][j], K2, ha[j]));
            const float x2 = fmaf(cv, wi[j], fmaf(piv[u][j], K2, hi[j]));
            const float r1 = rcp_ftz(1.0f + tc::fast_exp2(x1)), r2 = rcp_ftz(1.0f + tc::fast_exp2(x2));
            s[u][0] = fmaf(va[j], fmaf(-2.0f, r1, 1.0f), s[u][0]);
            s[u][1] = fmaf(vi[j], fmaf(-2.0f, r2, 1.0f), s[u][1]);
          }
        }
#pragma unroll
        for (int u = 0; u < RU; ++u) {
          const float x1 = warp_sum(s[u][0]), x2 = warp_sum(s[u][1]);
          if (lane == 0 && i + u < n) {
            s_e[i + u] = x1 + v1b;
            s_e[a.chunk + i + u] = x2 + v2b;
          }
        }
      }
    };
    const float* const gpa = a.proj_a + ((size_t)b * Lt + t0) * D;
    const float* const gpi = a.proj_i + ((size_t)b * Lt + t0) * D;
    using N7 = std::integral_constant<int, 7>;
    using N8 = std::integral_constant<int, 8>;
    using R2 = std::integral_constant<int, 2>;
    using R4 = std::integral_constant<int, 4>;
    const bool nj7 = D > 192 && D <= 224;      // the model's D = 2 H = 200; any other D <= 256 takes the zero-padded eight
    if (staged) {
      if (n > 0) tc::mbar_wait(bar_proj, parity);
      if (nj7) energies(s_st0, s_st1, N7{}, R2{});
      else energies(s_st0, s_st1, N8{}, R2{});
    } else {
      // (the constrained nucleus roll-out holds more across the step: two rows per warp round keep it at 128 registers without a
      // spill -- four spilled 80 bytes around these loads.  The rows' sums are the same either way)
      using RL = std::conditional_t<kNucleus && kConstrained, R2, R4>;
      if (nj7) energies(gpa, gpi, N7{}, RL{});
      else energies(gpa, gpi, N8{}, RL{});
    }
    __syncthreads();
    if (staged && tid == 0 && n > 0) {       // every read of the proj rows is behind the barrier: the buffers take the enc rows
      tc::fence_proxy_async();
      tc::mbar_expect_tx(bar_enc, 2 * stage_bytes, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st0), a.enc_a + ((size_t)b * Lt + t0) * D, stage_bytes, bar_enc, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st1), a.enc_i + ((size_t)b * Lt + t0) * D, stage_bytes, bar_enc, 1);
    }
    DEC_STAMP(4);
    float m1 = -INFINITY, m2 = -INFINITY;
    for (int i = tid; i < n; i += NT) {
      m1 = fmaxf(m1, s_e[i]);
      m2 = fmaxf(m2, s_e[a.chunk + i]);
    }
    m1 = block_max(m1, s_red);
    m2 = block_max(m2, s_red);
    float l1 = 0.f, l2 = 0.f;
    for (int i = tid; i < n; i += NT) {
      const float p1 = expf(s_e[i] - m1), p2 = expf(s_e[a.chunk + i] - m2);
      s_e[i] = p1;
      s_e[a.chunk + i] = p2;
      l1 += p1;
      l2 += p2;
    }
    l1 = block_sum(l1, s_red);
    l2 = block_sum(l2, s_red);
    __syncthreads();
    DEC_STAMP(5);
    // weighted contexts of this rank's rows
    if (staged && n > 0) tc::mbar_wait(bar_enc, parity);
    const float* ea = staged ? s_st0 : a.enc_a + ((size_t)b * Lt + t0) * D;
    const float* ei = staged ? s_st1 : a.enc_i + ((size_t)b * Lt + t0) * D;
    const bool vec4 = a.ctx_vec4 != 0;       // (staged rows are always aligned; rows read from L2 may not be)
    const int groups = vec4 ? NT / (D >> 2) : NT / D;
    if (vec4) {
      const int dv4 = D >> 2;
      const int g = tid / dv4, c4 = tid - g * dv4;
      if (g < groups) {
        float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
#pragma unroll 8
        for (int i = g; i < n; i += groups) {
          const float w1 = s_e[i], w2 = s_e[a.chunk + i];
          const float4 x1 = *reinterpret_cast<const float4*>(ea + (size_t)i * D + c4 * 4);
          const float4 x2 = *reinterpret_cast<const float4*>(ei + (size_t)i * D + c4 * 4);
          s1.x = fmaf(w1, x1.x, s1.x); s1.y = fmaf(w1, x1.y, s1.y); s1.z = fmaf(w1, x1.z, s1.z); s1.w = fmaf(w1, x1.w, s1.w);
          s2.x = fmaf(w2, x2.x, s2.x); s2.y = fmaf(w2, x2.y, s2.y); s2.z = fmaf(w2, x2.z, s2.z); s2.w = fmaf(w2, x2.w, s2.w);
        }
        *reinterpret_cast<float4*>(s_cpart + (g * 2 + 0) * D + c4 * 4) = s1;
        *reinterpret_cast<float4*>(s_cpart + (g * 2 + 1) * D + c4 * 4) = s2;
      }
    } else {
      const int g = tid / D, d = tid - g * D;
      if (g < groups) {
        float s1 = 0.f, s2 = 0.f;
        for (int i = g; i < n; i += groups) {
          s1 = fmaf(s_e[i], ea[(size_t)i * D + d], s1);
          s2 = fmaf(s_e[a.chunk + i], ei[(size_t)i * D + d], s2);
        }
        s_cpart[(g * 2 + 0) * D + d] = s1;
        s_cpart[(g * 2 + 1) * D + d] = s2;
      }
    }
    __syncthreads();
    if constexpr (kGreedy) {
      // every read of the enc rows is behind the barrier: the buffers take the NEXT step's proj rows, which then arrive while
      // stages C - E and the next stage A run
      // (beam: whether another run follows is known only after the selection -- the last copy is waited for before the exit)
      if (staged && tid == 0 && n > 0 && (kBeam || s + 1 < S)) {
        tc::fence_proxy_async();
        tc::mbar_expect_tx(bar_proj, 2 * stage_bytes, 1);
        tc::tma_bulk_g2s(tc::smem_u32(s_st0), a.proj_a + ((size_t)b * Lt + t0) * D, stage_bytes, bar_proj, 1);
        tc::tma_bulk_g2s(tc::smem_u32(s_st1), a.proj_i + ((size_t)b * Lt + t0) * D, stage_bytes, bar_proj, 1);
      }
    }
    // this rank's partials -> slot R of every rank
    for (int d = tid; d < 2 * D; d += NT) {
      const int k = d / D, dd = d - k * D;
      float s = 0.f;
      for (int g = 0; g < groups; ++g) s += s_cpart[(g * 2 + k) * D + dd];
      for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_part, r)[R * (4 + 2 * D) + 4 + d] = s;
    }
    if (tid < CL) {
      float* dst = cluster.map_shared_rank(s_part, tid) + R * (4 + 2 * D);
      dst[0] = m1; dst[1] = l1; dst[2] = m2; dst[3] = l2;
    }
  }
  DEC_STAMP(6);
  cluster.sync();
  DEC_STAMP(7);

  // merge (every rank, redundantly): contexts c1, c2; the scale that turns this rank's p into alpha
  float scale_own[2];
  {
    float* s_w = s_scr;                                           // [2][MAXC] merge weights w_r / l, then [2 MAXC .. ] own scales
    if (tid < 2) {
      const int k = tid;
      float m = -INFINITY;
      for (int r = 0; r < CL; ++r)
        if (min(Lt, r * a.chunk) < Lt) m = fmaxf(m, s_part[r * (4 + 2 * D) + 2 * k]);     // (a rank without rows: m = -inf, l = 0)
      float l = 0.f, w[MAXC];
#pragma unroll
      for (int r = 0; r < MAXC; ++r) {
        w[r] = (r < CL && min(Lt, r * a.chunk) < Lt) ? expf(s_part[r * (4 + 2 * D) + 2 * k] - m) : 0.f;
        l = fmaf(w[r], r < CL ? s_part[r * (4 + 2 * D) + 2 * k + 1] : 0.f, l);
      }
      const float inv = 1.f / l;
#pragma unroll
      for (int r = 0; r < MAXC; ++r) s_w[k * MAXC + r] = w[r] * inv;
    }
    __syncthreads();
    scale_own[0] = s_w[R];
    scale_own[1] = s_w[MAXC + R];
    for (int i = tid; i < 2 * D; i += NT) {
      const int k = i / D;
      float sum = 0.f;
      for (int r = 0; r < CL; ++r) sum = fmaf(s_w[k * MAXC + r], s_part[r * (4 + 2 * D) + 4 + i], sum);
      s_ctx[i] = sum;
      if (!kGreedy && R == 0) a.ctx12[((size_t)k * a.B + b) * D + (i - k * D)] = sum;
    }
  }
  __syncthreads();
  DEC_STAMP(8);

  // ---- stage C: pb_k = W_beta_{1,3} c_k (split), gathered; beta; c3; attention / coverage outputs of this rank's rows ------
  {
    const int per = (2 * D + CL - 1) / CL, o0 = R * per, o1 = min(2 * D, o0 + per);
    // outputs below D take c1 (W_beta_1), the others c2 (W_beta_3); a rank's range may straddle the two
    for (int k = 0; k < 2; ++k) {
      const int lo = max(o0, k * D), hi = min(o1, (k + 1) * D);
      block_matvec_t(a.Wb13t + (size_t)k * D * D, D, nullptr, s_ctx + k * D, D, hi - lo, s_scr, SCR, ((lo - k * D) & 3) == 0,
                     [&](int i) { return lo - k * D + i; },
                     [&](int i, float v) {
                       const int o = lo + i;
                       for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_pb, r)[o] = v;
                       if constexpr (!kGreedy) a.pb[((size_t)k * a.B + b) * D + (o - k * D)] = v;
                     });
    }
  }
  DEC_STAMP(9);
  cluster.sync();
  DEC_STAMP(10);
  float beta1, beta2;
  {
    float eb1 = 0.f, eb2 = 0.f;
    for (int d = tid; d < D; d += NT) {
      eb1 = fmaf(a.vb1[d], tanh_fast(s_pb[d] + s_hw[2 * D + d]), eb1);
      eb2 = fmaf(a.vb2[d], tanh_fast(s_pb[D + d] + s_hw[3 * D + d]), eb2);
    }
    eb1 = block_sum(eb1, s_red) + a.vb1b[0];
    eb2 = block_sum(eb2, s_red) + a.vb2b[0];
    const float mb = fmaxf(eb1, eb2);
    const float x1 = expf(eb1 - mb), x2 = expf(eb2 - mb);
    beta1 = x1 / (x1 + x2);
    beta2 = x2 / (x1 + x2);
    for (int d = tid; d < D; d += NT) s_x[d] = s_ctx[d] * beta1 + s_ctx[D + d] * beta2;
    float closs = 0.f;
    for (int i = tid; i < n; i += NT) {
      const int t = t0 + i;
      const float a1 = s_e[i] * scale_own[0], a2 = s_e[a.chunk + i] * scale_own[1];
      if constexpr (!kGreedy) {
        a.alpha[((size_t)b * 2 + 0) * Lt + t] = a1;
        a.alpha[((size_t)b * 2 + 1) * Lt + t] = a2;
      }
      const float att = a1 * beta1 + a2 * beta2;                 // bmm([a1 a2], beta), attention.py:167
      if constexpr (kBeam) {
        const float cnew = s_cov[i] + att;
        s_bcvn[slot * ldv + i] = cnew;
        closs += fminf(att, cnew);
      } else if constexpr (kGreedy) {
        const float cnew = s_cov[i] + att;                       // (the energies of this step have read s_cov: barriers since)
        s_cov[i] = cnew;
        closs += fminf(att, cnew);
      } else {
        const float cnew = a.cov[(size_t)b * Lt + t] + att;
        a.att_cov[(size_t)b * Lt + t] = att;
        a.cov_out[(size_t)b * Lt + t] = cnew;
        closs += fminf(att, cnew);
      }
    }
    closs = block_sum(closs, s_red);
    if (tid == 0) cluster.map_shared_rank(s_ex, 0)[R * 8 + 0] = closs;      // summed by rank 0 after the next cluster barrier
    if (!kGreedy && R == 0 && tid == 0) {
      a.beta[b * 2 + 0] = beta1;
      a.beta[b * 2 + 1] = beta2;
    }
  }
  __syncthreads();
  if (!kGreedy && R == 0)
    for (int i = tid; i < K; i += NT) a.xcat[(size_t)b * K + i] = s_x[i];

  DEC_STAMP(11);
  // ---- stage D: LSTM gates of this rank's hidden units, cell update; h' gathered -------------------------------------------
  {
    // (units per rank: a multiple of 4 -- the four gate segments of a rank start 16-byte aligned and hold whole quads)
    const int per = split4(H, CL), j0 = R * per, j1 = min(H, j0 + per), nj = max(0, j1 - j0);
    block_matvec_t(a.Wcatt, 4 * H, a.bcat, s_x, K, 4 * nj, s_scr, SCR, ((H | nj) & 3) == 0, [&](int i) { return (i / nj) * H + j0 + (i % nj); },
                   [&](int i, float v) { s_g[(i / nj) * (per + 1) + (i % nj)] = v; });
    __syncthreads();
    if (tid < nj) {
      const int j = j0 + tid;
      const float gi = gate_act(s_g[tid], 1.f), gf = gate_act(s_g[(per + 1) + tid], 1.f), gg = tanh_fast(s_g[2 * (per + 1) + tid]),
                  go = gate_act(s_g[3 * (per + 1) + tid], 1.f);
      const float c = fmaf(gf, kBeam ? s_bc[slot * ldc + tid] : kGreedy ? cell_own : a.cell[(size_t)b * H + j], gi * gg);
      const float hn = go * tanh_fast(c);
      if constexpr (kBeam) {
        s_bcn[slot * ldc + tid] = c;
      } else if constexpr (kGreedy) {
        cell_own = c;
      } else {
        a.cell_out[(size_t)b * H + j] = c;
        a.h_out[(size_t)b * H + j] = hn;
        float* gs = a.gates + (size_t)b * 4 * H;                // activated gates, kept for the backward pass
        gs[j] = gi; gs[H + j] = gf; gs[2 * H + j] = gg; gs[3 * H + j] = go;
      }
      for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_hn, r)[j] = hn;
    }
  }
  DEC_STAMP(12);
  cluster.sync();
  DEC_STAMP(13);
  if constexpr (kBeam)                     // (s_hn is written again only behind the cluster barriers of the next run)
    for (int i = tid; i < H; i += NT) s_bhn[slot * ldh + i] = s_hn[i];
  // greedy: the probabilities / arg-max of step s go to row (b, s) of (B, S, M) / (B, S); the loss terms (S, 2, B) to row s
  // (sampled: row (b N + n, s) of (B N, S, M) / (B N, S))
  const size_t prow = kGreedy ? (size_t)(kSample ? cluster_row() : ob) * S + s : (size_t)b;
  const int lrow = kGreedy ? s * 2 * a.B + b : b;
  if (R == 0 && tid == 0 && a.cov_loss) {
    float cs = 0.f;
    for (int r = 0; r < CL; ++r) cs += s_ex[r * 8 + 0];
    a.cov_loss[lrow] = cs;
  }

  // ---- stage E: logits of this rank's sentences, masked soft-max over M, arg-max, NLL ---------------------------------------
  {
    const int per = (M + CL - 1) / CL, m0 = min(M, R * per), m1 = min(M, m0 + per);
    float* const lg = s_cpart;                                   // this rank's logits (the context partials are dead)
    block_matvec_t(a.out_wt, M, a.out_b, s_hn, H, m1 - m0, s_scr, SCR, (m0 & 3) == 0, [&](int i) { return m0 + i; }, [&](int i, float v) { lg[i] = v; });
    __syncthreads();
    for (int m = m0 + tid; m < m1; m += NT)
      if (!a.mask[(size_t)b * M + m]) lg[m - m0] = kNegFill;     // attention.py:184 (masked_softmax)
    __syncthreads();
    float mx = -INFINITY;
    for (int m = m0 + tid; m < m1; m += NT) mx = fmaxf(mx, lg[m - m0]);
    mx = block_max(mx, s_red);
    float sum = 0.f;
    for (int m = m0 + tid; m < m1; m += NT) sum += expf(lg[m - m0] - mx);
    sum = block_sum(sum, s_red);
    if (tid < CL) {
      float* dst = cluster.map_shared_rank(s_ex, tid) + R * 8;
      dst[1] = mx;
      dst[2] = sum;
    }
    DEC_STAMP(14);
    cluster.sync();
    DEC_STAMP(15);
    float gmx = -INFINITY;
    for (int r = 0; r < CL; ++r)
      if (min(M, r * per) < M) gmx = fmaxf(gmx, s_ex[r * 8 + 1]);
    float gsum = 0.f;
    for (int r = 0; r < CL; ++r)
      if (min(M, r * per) < M) gsum = fmaf(s_ex[r * 8 + 2], expf(s_ex[r * 8 + 1] - gmx), gsum);
    const float inv = 1.f / gsum;
    float best = -INFINITY;
    int best_i = M;
    const int tg = a.target ? (int)a.target[kGreedy ? b * g.T + s : b] : -1;
    const bool eos_ok = kConstrained && !kBeam && eos_allowed(cn, eos, kept);
    const uint32_t cbase = ((uint32_t)(kSample ? cluster_row() : 0) * (uint32_t)S + (uint32_t)s) * (uint32_t)M;   // sampled: the counter of sentence 0
    for (int m = m0 + tid; m < m1; m += NT) {
      const float p = expf(lg[m - m0] - gmx) * inv;
      if constexpr (kBeam) s_bp[slot * ldp + m - m0] = p;
      else a.probs[prow * M + m] = p;
      if constexpr (kSample) {
        // top_k = 0: the first maximum of z over the candidates (the first candidate stands even at z = -inf);
        // top_k > 0: this rank's p for the selection below
        const bool cand = !kConstrained || (((allow >> ((unsigned)(m - m0) / NT)) & 1u) && (m != eos || eos_ok));
        if (sp.top_k > 0) {
          lg[m - m0] = p;
        } else if constexpr (kNucleus) {                         // nucleus: the row of every rank (the draw follows the cut)
          for (int r = 0; r < CL; ++r) cluster.map_shared_rank(smem + nu.off, r)[m] = cand ? p : -1.f;
        } else if (cand) {
          const float z = kConstrained ? sample_z(sp, p, cbase + (uint32_t)m) : sample_score(p, inv_t, cbase + (uint32_t)m, key0, key1);
          if (z > best || best_i == M) { best = z; best_i = m; }
        }
      } else if constexpr (kConstrained && !kBeam) {             // the first maximum over the eligible sentences
        if (((allow >> ((unsigned)(m - m0) / NT)) & 1u) && (m != eos || eos_ok) && p > best) { best = p; best_i = m; }
      } else if (p > best) { best = p; best_i = m; }
      if (m == tg && a.nll) a.nll[lrow] = -logf(p + 1e-12f);      // models.py:168-170
    }
    if constexpr (kNucleus) {
      if (sp.top_k == 0) {                                       // (uniform) the cut of the whole row, then the draw over this rank's members
        cluster.sync();
        const float* const nv = smem + nu.off;
        const NucleusCut cut = nucleus_cut(nv, M, nu.P, reinterpret_cast<unsigned long long*>(smem + nu.off + up4(M)),
                                           reinterpret_cast<unsigned long long*>(smem + nu.off + up4(M) + 2 * kNucBuckets));
        for (int m = m0 + tid; m < m1; m += NT) {
          const float p = nv[m];
          const uint32_t bits = __float_as_uint(p);
          if (p >= 0.f && (bits > cut.pstar || (bits == cut.pstar && m <= cut.mstar))) {
            const float z = kConstrained ? sample_z(sp, p, cbase + (uint32_t)m) : sample_score(p, inv_t, cbase + (uint32_t)m, key0, key1);
            if (z > best || best_i == M) { best = z; best_i = m; }
          }
        }
      }
    }
    // (sampled with top_k > 0: the pick is made after the step, by the selection)
    if (!kBeam && (kGreedy || a.argmax) && !(kSample && sp.top_k > 0)) {     // first maximal index, as torch.max(dim) documents
      const float bbest = block_max(best, s_red);
      int cand = best == bbest ? best_i : M;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
      __shared__ int redi[NW];
      __syncthreads();
      if (lane == 0) redi[warp] = cand;
      __syncthreads();
      if (tid == 0) {
        int r = M;
        for (int w = 0; w < NW; ++w) r = min(r, redi[w]);
        // (greedy: to every rank, each of which needs the pick for its next step's input row)
        for (int q = 0; q < (kGreedy ? CL : 1); ++q) {
          float* dst = cluster.map_shared_rank(s_ex, q) + R * 8;
          dst[3] = bbest;
          dst[4] = __int_as_float(r);
        }
      }
      cluster.sync();
      // (the step kernel: rank 0 alone; the roll-out: every thread of every rank, for the next step's input row)
      if (kGreedy || (R == 0 && tid == 0)) {
        float gb = -INFINITY;
        int gi = M;
        for (int r = 0; r < CL; ++r) {
          if (min(M, r * per) >= M) continue;
          const float pb_ = s_ex[r * 8 + 3];
          const int ib = __float_as_int(s_ex[r * 8 + 4]);
          if (pb_ > gb || (pb_ == gb && ib < gi)) { gb = pb_; gi = ib; }
        }
        if constexpr (kGreedy) {
          if constexpr (kConstrained) {
            if (gi == M) gi = eos;                                 // no eligible sentence (the caller's mask hides rows below EOS)
            if (gi < eos) {
              ++kept;
              const int j = gi - m0;                               // under no_repeat the pick is no longer eligible
              if (cn.no_repeat && j >= 0 && gi < m1 && j % NT == tid) allow &= ~(1u << (j / NT));
            }
          }
          if (R == 0 && tid == 0) a.argmax[prow] = gi;
          pick = gi;
        } else {
          a.argmax[b] = gi;
        }
      }
    }
  }
  if constexpr (kBeam) ++runs;
  }  // slots
  if constexpr (kBeam || kSample) {
    // ---- selection: the new table from the live slots' candidates and the finished slots' carries ---------------------------------
    // (sampled, top_k > 0: the best top_k of this step's (p, sentence) candidates, and the draw among them)
    constexpr int kNone = 0x7fffffff;
    const int per = (M + CL - 1) / CL, m0 = min(M, R * per), m1 = min(M, m0 + per), nm = m1 - m0;
    // the selection's width (stochastic: one more, the best pruned key)
    const int KS = kSample ? sp.top_k : kStoch ? KW + 1 : KW;
    // the exchange arrays (sampled: formed here from the parameter, so that nothing of them is held over the step's other stages)
    float* const q_cand = kSample ? smem + sp.off + 7 * MAXK : s_cand;
    float* const q_wred = kSample ? q_cand + MAXC * MAXK * 4 : s_wred;
    float* const q_loc = kSample ? q_wred + NW * 4 : s_loc;
    bool any_live = false;
    if constexpr (kSample) any_live = sp.top_k > 0;             // (uniform)
    else for (int k = 0; k < KW; ++k) any_live = any_live || bs_stat[k] == kLive;
    __syncthreads();                                             // s_bp of the last run (sampled: this rank's p in s_cpart)
    const bool eos_ok = kSample && kConstrained && eos_allowed(cn, eos, kept);
    // stochastic: the stochastic region (see StochArgs), formed here like the sampled exchange arrays
    float* const x_phi = smem + st.off;                          // [MAXK] phi of every slot,
    float* const x_key = x_phi + MAXK;                           // [MAXK]   key,
    float* const x_nphi = x_key + MAXK;                          // [MAXK]   of the next table,
    float* const x_nkey = x_nphi + MAXK;                         // [MAXK]
    float* const x_lam = x_nkey + MAXK;                          // [MAXK] lam of every slot this step
    unsigned long long* const x_q = reinterpret_cast<unsigned long long*>(x_lam + MAXK);   // [MAXC][MAXK] every rank's mass, remote
    float* const x_mu = reinterpret_cast<float*>(x_q + MAXC * MAXK);                     // [MAXC][MAXK] every rank's max l, remote
    float* const x_z = x_mu + MAXC * MAXK;                                               // [MAXC][MAXK] every rank's max G, remote
    float* const s_key = x_z + MAXC * MAXK;                      // [K][ldp] the key of every (slot, sentence) of this rank
    if constexpr (kStoch) {
      if (any_live) {                                            // (uniform) the keys of every live slot's candidates
        unsigned long long key;
        asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(key) : "l"(st.key));
        const float it = 1.f / st.T;                             // (l = logf(p) it is rounded before it is used: never an FMA)
        auto cand = [&](int k, int m, float p) {                 // the beam's candidates (p > 0, eligible)
          if (!(p > 0.f)) return false;
          if constexpr (kConstrained) {
            if (!((bu_cur[k * ldu + ((m - m0) >> 5)] >> ((m - m0) & 31)) & 1u)) return false;
            if (m == eos && !eos_allowed(cn, eos, bk_cur[k])) return false;
          }
          return true;
        };
        auto rank_max = [&](const float* x, int k) {             // over the ranks (a rank without candidates gives -inf)
          float v = -INFINITY;
          for (int r = 0; r < CL; ++r) v = fmaxf(v, x[r * MAXK + k]);
          return v;
        };
        // mu: the largest l = logf(p) / T of the candidates
        for (int k = 0; k < KW; ++k) {
          if (bs_stat[k] != kLive) continue;
          float mx = -INFINITY;
          for (int m = m0 + tid; m < m1; m += NT) {
            const float p = s_bp[k * ldp + m - m0];
            if (cand(k, m, p)) mx = fmaxf(mx, __fmul_rn(logf(p), it));
          }
          mx = block_max(mx, s_red);
          if (tid < CL) cluster.map_shared_rank(x_mu, tid)[R * MAXK + k] = mx;
        }
        cluster.sync();
        // Q: the integer masses floor(e^(l - mu) 2^24), summed exactly
        for (int k = 0; k < KW; ++k) {
          if (bs_stat[k] != kLive) continue;
          const float mu = rank_max(x_mu, k);
          unsigned long long q = 0;
          for (int m = m0 + tid; m < m1; m += NT) {
            const float p = s_bp[k * ldp + m - m0];
            if (cand(k, m, p)) q += __float2ull_rz(expf(__fmul_rn(logf(p), it) - mu) * 16777216.f);
          }
          q = block_sum_u64(q, s_red);
          if (tid < CL) cluster.map_shared_rank(x_q, tid)[R * MAXK + k] = q;
        }
        cluster.sync();
        // lam, the perturbed log-probabilities G of the children and their largest, Z
        for (int k = 0; k < KW; ++k) {
          if (bs_stat[k] != kLive) continue;
          unsigned long long Q = 0;
          for (int r = 0; r < CL; ++r) Q += x_q[r * MAXK + k];
          const float lam = rank_max(x_mu, k) + logf((float)Q * 5.9604644775390625e-8f);
          if (tid == 0) x_lam[k] = lam;
          const float phk = x_phi[k];
          const uint32_t cb = (((uint32_t)b * (uint32_t)S + (uint32_t)s) * (uint32_t)KW + (uint32_t)k) * (uint32_t)M;
          float mx = -INFINITY;
          for (int m = m0 + tid; m < m1; m += NT) {
            const float p = s_bp[k * ldp + m - m0];
            float G = -INFINITY;
            if (cand(k, m, p)) {
              const float u = ((float)(hash32(cb + (uint32_t)m, (uint32_t)key, (uint32_t)(key >> 32)) >> 9) + 0.5f) * 1.1920928955078125e-7f;
              G = (phk + (__fmul_rn(logf(p), it) - lam)) + -logf(-logf(u));
              mx = fmaxf(mx, G);
            }
            s_key[k * ldp + m - m0] = G;
          }
          mx = block_max(mx, s_red);
          if (tid < CL) cluster.map_shared_rank(x_z, tid)[R * MAXK + k] = mx;
        }
        cluster.sync();
        // the keys: G truncated below the parent's key at Z
        for (int k = 0; k < KW; ++k) {
          if (bs_stat[k] != kLive) continue;
          const float Z = rank_max(x_z, k), kp = x_key[k];
          for (int m = m0 + tid; m < m1; m += NT) {
            const float G = s_key[k * ldp + m - m0];
            if (G != -INFINITY) s_key[k * ldp + m - m0] = truncated_key(kp, G, Z);
          }
        }
        __syncthreads();
      }
    }
    if (any_live) {
      // this rank's best K of its (live slot, sentence) candidates, one block-wide pick per round; each pick ranks below the last
      float ps = INFINITY, pp = INFINITY;
      int pk = -1, pm = -1;
      for (int r = 0; r < KS; ++r) {
        float cs = -INFINITY, cp = -1.f;
        int ck = kNone, cm = kNone;
        for (int c = tid; c < (kSample ? nm : KW * nm); c += NT) {
          if constexpr (kSample) {                               // ranked by p (as score and p), then sentence; k = 0
            const int m = m0 + c;
            if (kConstrained && (!((allow >> ((unsigned)c / NT)) & 1u) || (m == eos && !eos_ok))) continue;
            const float p = s_cpart[c];
            if (cand_better(ps, pp, pk, pm, p, p, 0, m) && cand_better(p, p, 0, m, cs, cp, ck, cm)) { cs = p; cp = p; ck = 0; cm = m; }
            continue;
          }
          const int k = c / nm, m = m0 + (c - k * nm);
          if (bs_stat[k] != kLive) continue;
          const float p = s_bp[k * ldp + m - m0];
          if (!(p > 0.f)) continue;                              // masked sentences: exactly 0
          if constexpr (kConstrained) {                          // ineligible sentences offer nothing
            if (!((bu_cur[k * ldu + ((m - m0) >> 5)] >> ((m - m0) & 31)) & 1u)) continue;
            if (m == eos && !eos_allowed(cn, eos, bk_cur[k])) continue;
          }
          const float sc = kStoch ? s_key[k * ldp + m - m0] : bs_score[k] + logf(p);      // (stochastic: ranked by key)
          if (cand_better(ps, pp, pk, pm, sc, p, k, m) && cand_better(sc, p, k, m, cs, cp, ck, cm)) { cs = sc; cp = p; ck = k; cm = m; }
        }
        cand_warp_best(cs, cp, ck, cm);
        if (lane == 0) {
          q_wred[warp * 4 + 0] = cs; q_wred[warp * 4 + 1] = cp;
          q_wred[warp * 4 + 2] = __int_as_float(ck); q_wred[warp * 4 + 3] = __int_as_float(cm);
        }
        __syncthreads();
        if (warp == 0) {
          float ws = -INFINITY, wp = -1.f;
          int wk = kNone, wm = kNone;
          if (lane < NW) {
            ws = q_wred[lane * 4 + 0]; wp = q_wred[lane * 4 + 1];
            wk = __float_as_int(q_wred[lane * 4 + 2]); wm = __float_as_int(q_wred[lane * 4 + 3]);
          }
          cand_warp_best(ws, wp, wk, wm);
          if (lane == 0) {
            q_loc[r * 4 + 0] = ws; q_loc[r * 4 + 1] = wp;
            q_loc[r * 4 + 2] = __int_as_float(wk); q_loc[r * 4 + 3] = __int_as_float(wm);
          }
        }
        __syncthreads();
        ps = q_loc[r * 4 + 0]; pp = q_loc[r * 4 + 1];
        pk = __float_as_int(q_loc[r * 4 + 2]); pm = __float_as_int(q_loc[r * 4 + 3]);
      }
      for (int i = tid; i < CL * KS * 4; i += NT) {              // -> slot R of every rank
        const int q = i / (KS * 4), e = i - q * KS * 4;
        cluster.map_shared_rank(q_cand, q)[R * CS * 4 + e] = q_loc[e];
      }
      cluster.sync();
    }
    // every rank merges the same entries in the same order: the ranks' best K (none when no slot is live), then the carries
    // (sampled: every warp, no carries; each of the best top_k is drawn for -- the largest z, ties to the smaller sentence)
    float bz = -INFINITY;
    int drawn = M;
    if (kSample ? any_live : warp == 0) {
      const int npub = any_live ? CL * KS : 0, tot = npub + (kSample ? 0 : KW);
      float ps = INFINITY, pp = INFINITY;
      int pk = -1, pm = -1;
      float nuc_p = 0.f;                                         // nucleus: lane j keeps the j-th entry (nuc_m = M: none)
      int nuc_m = M;
      for (int j = 0; j < KS; ++j) {
        float cs = -INFINITY, cp = -1.f;
        int ck = kNone, cm = kNone;
        for (int i = lane; i < tot; i += 32) {
          float es, ep;
          int ek, em;
          if (i < npub) {
            const float* e = q_cand + ((i / KS) * CS + i % KS) * 4;
            es = e[0]; ep = e[1]; ek = __float_as_int(e[2]); em = __float_as_int(e[3]);
          } else {
            const int k = i - npub;
            if (bs_stat[k] != kDone) continue;
            // a finished slot carries its hypothesis with probability 1 (stochastic: its key)
            es = kStoch ? x_key[k] : bs_score[k]; ep = 1.f; ek = k; em = eos;
          }
          if (ek == kNone) continue;
          if (cand_better(ps, pp, pk, pm, es, ep, ek, em) && cand_better(es, ep, ek, em, cs, cp, ck, cm)) { cs = es; cp = ep; ck = ek; cm = em; }
        }
        cand_warp_best(cs, cp, ck, cm);
        if constexpr (kNucleus) {
          if (ck != kNone && lane == j) { nuc_p = cp; nuc_m = cm; }
        } else if constexpr (kSample) {
          if (ck != kNone) {
            const uint32_t c = ((uint32_t)cluster_row() * (uint32_t)S + (uint32_t)s) * (uint32_t)M + (uint32_t)cm;
            const float z = kConstrained ? sample_z(sp, cp, c) : sample_score(cp, inv_t, c, key0, key1);
            if (drawn == M || z > bz || (z == bz && cm < drawn)) { bz = z; drawn = cm; }
          }
        } else if constexpr (kStoch) {
          if (lane == 0) {
            // the table as the beam's, with the score, phi and key of the new slot; the (K + 1)-th entry is the best pruned key,
            // and the threshold the largest of them so far
            const bool none = ck == kNone, carry = !none && bs_stat[ck] == kDone;
            if (j == KW) {
              if (R == 0) st.kappa[b] = fmaxf(s == 0 ? -INFINITY : st.kappa[b], none ? -INFINITY : cs);
            } else {
              nt_score[j] = none ? -INFINITY : carry ? bs_score[ck] : bs_score[ck] + logf(cp);
              x_nphi[j] = none ? -INFINITY : carry ? x_phi[ck] : x_phi[ck] + (__fmul_rn(logf(cp), 1.f / st.T) - x_lam[ck]);
              x_nkey[j] = none ? -INFINITY : cs;
              nt_tok[j] = none ? -1 : cm;
              nt_par[j] = none ? -1 : ck;
              nt_kind[j] = none ? 0 : carry ? 3 : cm == eos ? 2 : 1;
            }
          }
        } else if (lane == 0) {
          // kind: 0 empty, 1 live, 2 finished by this step's EOS pick, 3 carried
          const bool none = ck == kNone;
          nt_score[j] = none ? -INFINITY : cs;
          nt_tok[j] = none ? -1 : cm;
          nt_par[j] = none ? -1 : ck;
          nt_kind[j] = none ? 0 : bs_stat[ck] == kDone ? 3 : cm == eos ? 2 : 1;
        }
        ps = cs; pp = cp; pk = ck; pm = cm;
      }
      if constexpr (kNucleus) {
        // the nucleus is the first n entries: lane j is in when the mass before it is below need (lane 0 always).  At most 8
        // masses of at most 2^24: the sums fit 32 bits
        const uint32_t q = nuc_m < M ? __float2uint_rz(nuc_p * 16777216.f) : 0u;
        uint32_t incl = q;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += t;
        }
        const unsigned long long pq = (unsigned long long)nu.P * __shfl_sync(0xffffffffu, incl, 31);
        const unsigned long long need = (pq >> 24) + ((pq & 0xffffffull) != 0ull);
        if (nuc_m < M && (lane == 0 || (unsigned long long)(incl - q) < need)) {
          const uint32_t c = ((uint32_t)cluster_row() * (uint32_t)S + (uint32_t)s) * (uint32_t)M + (uint32_t)nuc_m;
          bz = kConstrained ? sample_z(sp, nuc_p, c) : sample_score(nuc_p, inv_t, c, key0, key1);
          drawn = nuc_m;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {                       // the largest z, ties to the smaller sentence
          const float z2 = __shfl_xor_sync(0xffffffffu, bz, o);
          const int d2 = __shfl_xor_sync(0xffffffffu, drawn, o);
          if (d2 != M && (drawn == M || z2 > bz || (z2 == bz && d2 < drawn))) { bz = z2; drawn = d2; }
        }
      }
    }
    if constexpr (kSample) {
      if (any_live) {                                            // the pick, as stage E takes it without top_k
        int gi = drawn;
        if constexpr (kConstrained) {
          if (gi == M) gi = eos;                                 // no eligible sentence (the caller's mask hides rows below EOS)
          if (gi < eos) {
            ++kept;
            const int j = gi - m0;                               // under no_repeat the pick is no longer eligible
            if (cn.no_repeat && j >= 0 && gi < m1 && j % NT == tid) allow &= ~(1u << (j / NT));
          }
        }
        if (R == 0 && tid == 0) a.argmax[(size_t)cluster_row() * S + s] = gi;
        pick = gi;
      }
    } else {
    __syncthreads();
    // outputs of step s; the state of the new live slots gathered from their parents' step outputs; the new table
    const size_t row = ((size_t)b * S + s) * KW;
    if (R == 0 && tid == 0)
      for (int j = 0; j < KW; ++j) {
        bm.tokens[row + j] = nt_tok[j];
        bm.parents[row + j] = nt_par[j];
        bm.scores[row + j] = nt_score[j];
        if constexpr (kStoch) {
          st.phi[row + j] = x_nphi[j];
          st.keys[row + j] = x_nkey[j];
        }
      }
    for (int i = tid; i < KW * nm; i += NT) {                    // the row the parent produced (zero for carries and empty slots)
      const int j = i / nm, m = m0 + (i - j * nm), kd = nt_kind[j];
      bm.probs[(row + j) * M + m] = (kd == 1 || kd == 2) ? s_bp[nt_par[j] * ldp + m - m0] : 0.f;
    }
    for (int j = 0; j < KW; ++j) {
      if (nt_kind[j] != 1) continue;                             // (uniform) only live slots run again
      const int q = nt_par[j];
      for (int i = tid; i < H; i += NT) s_bh[j * ldh + i] = s_bhn[q * ldh + i];
      for (int i = tid; i < ldc; i += NT) s_bc[j * ldc + i] = s_bcn[q * ldc + i];
      for (int i = tid; i < n; i += NT) s_bcv[j * ldv + i] = s_bcvn[q * ldv + i];
      if constexpr (kConstrained) {          // the parent's eligible bits and kept, then the new slot's own token
        const int tk = nt_tok[j], rel = tk - m0;
        const bool clear = cn.no_repeat && tk < eos && rel >= 0 && tk < m1;
        for (int w = tid; w < ldu; w += NT)
          bu_nxt[j * ldu + w] = bu_cur[q * ldu + w] & ~(clear && (rel >> 5) == w ? 1u << (rel & 31) : 0u);
        if (tid == 0) bk_nxt[j] = bk_cur[q] + (tk < eos ? 1 : 0);
      }
    }
    if (tid < KW) {
      const int kd = nt_kind[tid];
      bs_score[tid] = nt_score[tid];
      bs_tok[tid] = nt_tok[tid];
      bs_stat[tid] = kd == 1 ? kLive : kd == 0 ? kEmpty : kDone;
      if constexpr (kStoch) {
        x_phi[tid] = x_nphi[tid];
        x_key[tid] = x_nkey[tid];
      }
    }
    __syncthreads();
    if constexpr (kConstrained) {            // (uniform) the gathered bits are the next step's input
      uint32_t* const t = bu_cur; bu_cur = bu_nxt; bu_nxt = t;
      int* const u = bk_cur; bk_cur = bk_nxt; bk_nxt = u;
    }
    }  // (beam)
  }
  }  // steps (the loop body keeps the step kernel's indentation)
  if constexpr (kBeam) {
    if (staged && tid == 0 && n > 0) tc::mbar_wait(bar_proj, (uint32_t)(runs & 1));   // the proj rows copied after the last run
    if constexpr (kStoch) {
      if (R == 0 && tid < KW) {                                  // backtrack every final slot (an empty one: eos, slot -1)
        const size_t o = ((size_t)b * KW + tid) * S;
        int j = bm.parents[((size_t)b * S + S - 1) * KW + tid] < 0 ? -1 : tid;
        for (int s = S - 1; s >= 0; --s) {
          const size_t row = ((size_t)b * S + s) * KW;
          st.path_slots[o + s] = j;
          st.paths[o + s] = j >= 0 ? bm.tokens[row + j] : eos;
          j = j >= 0 ? bm.parents[row + j] : -1;
        }
      }
    } else if (R == 0 && tid == 0) {                             // backtrack the best hypothesis: slot 0 after the last step
      int j = 0;
      for (int s = S - 1; s >= 0; --s) {
        const size_t row = ((size_t)b * S + s) * KW;
        bm.path[(size_t)b * S + s] = j;
        bm.best[(size_t)b * S + s] = j >= 0 ? bm.tokens[row + j] : -1;
        j = j >= 0 ? bm.parents[row + j] : -1;
      }
    }
  }
  DEC_STAMP(16);
  // (No barrier before the exit: every rank's LAST store into another rank's shared memory -- the soft-max statistics or the arg-max
  // candidates -- lies before a cluster barrier it has passed, so nothing can still be written into a rank that leaves here.  In the
  // greedy loop the same holds between the steps: a store of step s + 1 into another rank lies behind at least one cluster barrier
  // that the other rank reaches only after its last read of what step s stored there.)
  DEC_STAMP(17);
}

__global__ void __launch_bounds__(NT) dec_step_fused_kernel(const FusedArgs a) {
  dec_fused_body<false>(a, GreedyArgs{}, BeamArgs{}, ConstraintArgs{}, SampleArgs{});
}

__global__ void __launch_bounds__(NT) dec_greedy_fused_kernel(const FusedArgs a, const GreedyArgs g) {
  dec_fused_body<true>(a, g, BeamArgs{}, ConstraintArgs{}, SampleArgs{});
}

__global__ void __launch_bounds__(NT) dec_beam_fused_kernel(const FusedArgs a, const GreedyArgs g, const BeamArgs bm) {
  dec_fused_body<true, true>(a, g, bm, ConstraintArgs{}, SampleArgs{});
}

__global__ void __launch_bounds__(NT) dec_greedy_constrained_kernel(const FusedArgs a, const GreedyArgs g, const ConstraintArgs cn) {
  dec_fused_body<true, false, true>(a, g, BeamArgs{}, cn, SampleArgs{});
}

__global__ void __launch_bounds__(NT) dec_beam_constrained_kernel(const FusedArgs a, const GreedyArgs g, const BeamArgs bm,
                                                                  const ConstraintArgs cn) {
  dec_fused_body<true, true, true>(a, g, bm, cn, SampleArgs{});
}

__global__ void __launch_bounds__(NT) dec_sample_kernel(const FusedArgs a, const GreedyArgs g, const SampleArgs sp) {
  dec_fused_body<true, false, false, true>(a, g, BeamArgs{}, ConstraintArgs{}, sp);
}

__global__ void __launch_bounds__(NT) dec_sample_constrained_kernel(const FusedArgs a, const GreedyArgs g, const ConstraintArgs cn,
                                                                    const SampleArgs sp) {
  dec_fused_body<true, false, true, true>(a, g, BeamArgs{}, cn, sp);
}

__global__ void __launch_bounds__(NT) dec_sample_nucleus_kernel(const FusedArgs a, const GreedyArgs g, const SampleArgs sp,
                                                                const NucleusArgs nu) {
  dec_fused_body<true, false, false, true, true>(a, g, BeamArgs{}, ConstraintArgs{}, sp, nu);
}

__global__ void __launch_bounds__(NT) dec_sample_nucleus_constrained_kernel(const FusedArgs a, const GreedyArgs g,
                                                                            const ConstraintArgs cn, const SampleArgs sp,
                                                                            const NucleusArgs nu) {
  dec_fused_body<true, false, true, true, true>(a, g, BeamArgs{}, cn, sp, nu);
}

__global__ void __launch_bounds__(NT) dec_beam_sample_kernel(const FusedArgs a, const GreedyArgs g, const BeamArgs bm,
                                                             const StochArgs st) {
  dec_fused_body<true, true, false, false, false, true>(a, g, bm, ConstraintArgs{}, SampleArgs{}, NucleusArgs{}, st);
}

__global__ void __launch_bounds__(NT) dec_beam_sample_constrained_kernel(const FusedArgs a, const GreedyArgs g, const BeamArgs bm,
                                                                         const ConstraintArgs cn, const StochArgs st) {
  dec_fused_body<true, true, true, false, false, true>(a, g, bm, cn, SampleArgs{}, NucleusArgs{}, st);
}

}  // namespace

// ----------------------------------------------------------------------------------------------------------------------------------
// Backward, the "head" of a step: everything between the previous step's text sweeps and this step's -- the masked soft-max backward,
// d h = d_logits out.weight, the LSTM cell backward, d c3 = d_gates W_ih[:, :D], the modality soft-max / W_beta tanh backward and
// d c_k += W_beta_k^T d_pre_k -- as ONE cluster kernel per step instead of three kernels and three library GEMMs (25 us of the 63 us of a
// backward step inside a CUDA graph: each of the six is a 2 - 5 us launch on a few CTAs).  Same cut as the forward: a cluster per video,
// mat-vecs split over the ranks with the weights read so that consecutive threads read consecutive outputs, small vectors through DSMEM.
// The two sweeps over the text axis (decoder_step.cu: dec_attn_sweep1 / sweep2) and the final d h GEMM keep their kernels.
// ----------------------------------------------------------------------------------------------------------------------------------
struct HeadArgs {
  const float *probs, *d_probs;                             // (B,M); d_probs may be null
  const long long* target;                                  // (B) or null
  const float *g_nll, *g_cov;                               // (B) or null: d loss / d [nll | coverage term]
  const float* out_w;                                       // (M, H) row-major (rows past M are never read)
  const float *gates, *cell_in, *cell_out;                  // (B,4H) activated gates, (B,H), (B,H)
  const float *d_h_out, *d_cell_out;                        // (B,H) or null
  const float* Wcat_ctx;                                    // (4H, D) = lstm.weight_ih[:, :D]
  const float *d_att_cov, *d_cov_out;                       // (B,Lt) or null
  const float *alpha, *beta, *ctx12, *pb, *hw;              // (B,2,Lt), (B,2), (2,B,D), (2,B,D), (B,4D)
  const float *vb1, *vb2;                                   // (D)
  const float *att, *cov_out;                               // (B,Lt): the step's att_cov / coverage' (fused coverage loss) or null
  const float* Wb13;                                        // (2, D, D) row-major
  float* d_logits;                                          // (B, ldd), columns M..ldd-1 zeroed
  float* d_gates;                                           // (B, ldg): first 4H columns
  float *d_cell, *datt, *dcov_tot, *d_pre_b, *d_ctx12;      // (B,H), (B,Lt), (B,Lt), (2,B,D), (2,B,D)
  float *vec_acc, *scal_acc;                                // (B,6,D), (B,4): accumulated in place (rows 4, 5; columns 2, 3)
  int B, Lt, D, H, M, ldd, ldg, chunk;
  // the whole step (mmb_decoder_step_fused_bwd): the two sweeps over the text axis and d h follow in the same launch
  int sweeps;
  const float *proj_a, *proj_i, *enc_a, *enc_i, *cov;       // (B,Lt,D) x4, (B,Lt) the step's coverage input
  const float *v1, *wc1, *v2, *wc2;                         // (D)
  float *d_proj_a, *d_proj_i, *d_cov;                       // (B,Lt,D) accumulated, (B,Lt) written
  const float* Wh_stack;                                    // (4H + 4D, H): [W_hh; W2; W4; W_beta_2; W_beta_4]
  float* d_h;                                               // (B,H)
  int stage_off;   // whole step: float offset of the row stage ([2 mbarriers][2][chunk * D]) in dynamic shared memory, or 0
};

__global__ void __launch_bounds__(NT) dec_bwd_head_kernel(const HeadArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = (int)cluster.num_blocks(), R = (int)cluster.block_rank();
  const int b = blockIdx.x / CL;
  const int tid = threadIdx.x;
  const int D = a.D, H = a.H, M = a.M, Lt = a.Lt;

  extern __shared__ __align__(16) float smem[];
  auto up4 = [](int v) { return (v + 3) & ~3; };
  float* s_dl = smem;                                   // [per_m]  this rank's slice of d_logits (first: p dp)
  const int per_m = (M + CL - 1) / CL;
  float* s_dhp = s_dl + up4(per_m);                     // [MAXC][H]  partial d h of every rank (written remotely)
  float* s_dg = s_dhp + up4(MAXC * H);                  // [4H]     d_gates
  float* s_dctx = s_dg + up4(4 * H);                    // [D]      d c3, gathered
  float* s_dpre = s_dctx + up4(D);                      // [2D]     d_pre_b
  float* s_ex = s_dpre + up4(2 * D);                    // [MAXC][4] scalar exchanges
  float* s_red = s_ex + MAXC * 4;                       // [32]
  float* s_scr = s_red + 32;                            // [NT]
  // mat-vec scratch: the whole-step launch lends the (then dead) column-partial buffer of sweep 8 -- room for the quad form's K slices
  const int mv_cap = a.sweeps ? (a.stage_off != 0 ? NW / 2 : NW) * 3 * D : NT;
  float* const mv_scr = a.sweeps ? s_scr + NT + up4(2 * D) + up4(2 * a.chunk) + up4(4 * a.chunk) + up4(6 * D) : s_scr;
  const bool mv_quads = a.sweeps != 0;

  // Row stage of the whole-step launch (see dec_step_fused_kernel): this rank's rows of enc_a / enc_i come in by two bulk copies issued
  // NOW, six head stages before sweep 7 reads them; when sweep 7 is done the same buffers take the rows of proj_a / proj_i for sweep 8
  // (under the block sums and the cluster barrier between the sweeps).  Without it every warp iteration of a sweep began with an L2
  // round trip (tools/decoder_bwd_trace.py: 11.3 k + 30.5 k cycles for the two sweeps).
  const int t0 = min(Lt, R * a.chunk), t1 = min(Lt, t0 + a.chunk), n = t1 - t0;
  const bool staged = a.stage_off != 0;
  float* const s_st0 = smem + a.stage_off + 4;
  float* const s_st1 = s_st0 + up4(a.chunk * D);
  const uint32_t bar_enc = tc::smem_u32(smem + a.stage_off), bar_proj = bar_enc + 8;
  const uint32_t stage_bytes = (uint32_t)(n * D) * 4u;
  if (staged && tid == 0) {
    tc::mbar_init(bar_enc, 1);
    tc::mbar_init(bar_proj, 1);
    tc::fence_barrier_init();
    if (n > 0) {
      tc::mbar_expect_tx(bar_enc, 2 * stage_bytes, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st0), a.enc_a + ((size_t)b * Lt + t0) * D, stage_bytes, bar_enc, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st1), a.enc_i + ((size_t)b * Lt + t0) * D, stage_bytes, bar_enc, 1);
    }
  }
  DEC_STAMP(18);
  // ---- 1: masked soft-max backward: d_logit = p (dp - sum p dp); masked entries have p = 0 ---------------------------------
  const int m0 = min(M, R * per_m), m1 = min(M, m0 + per_m);
  const int tg = a.target ? (int)a.target[b] : -1;
  const float dp_t = a.target ? -a.g_nll[b] / (a.probs[(size_t)b * M + tg] + 1e-12f) : 0.f;   // d(-log(p_tgt + eps)) at the target column
  if (a.d_probs) {      // (uniform over the cluster.  With the fused loss terms alone -- a training step -- sum p dp has the target's term
                        // only, which every rank forms by itself: no exchange, no cluster barrier)
    float dot = 0.f;
    for (int m = m0 + tid; m < m1; m += NT) dot = fmaf(a.probs[(size_t)b * M + m], a.d_probs[(size_t)b * M + m], dot);
    dot = block_sum(dot, s_red);
    if (tid < CL) cluster.map_shared_rank(s_ex, tid)[R * 4 + 0] = dot;
    cluster.sync();
  }
  {
    float dot = 0.f;
    if (a.d_probs)
      for (int r = 0; r < CL; ++r) dot += s_ex[r * 4 + 0];
    if (a.target) dot = fmaf(a.probs[(size_t)b * M + tg], dp_t, dot);
    for (int m = m0 + tid; m < m1; m += NT) {
      const float dp = (a.d_probs ? a.d_probs[(size_t)b * M + m] : 0.f) + (m == tg ? dp_t : 0.f);
      const float v = a.probs[(size_t)b * M + m] * (dp - dot);
      s_dl[m - m0] = v;
      a.d_logits[(size_t)b * a.ldd + m] = v;
    }
    if (R == 0)
      for (int m = M + tid; m < a.ldd; m += NT) a.d_logits[(size_t)b * a.ldd + m] = 0.f;   // row padding (keeps the weight-gradient GEMM aligned)
  }
  __syncthreads();
  DEC_STAMP(19);
  // ---- 2: d h (from the logits) = d_logits out.weight: this rank's rows of out.weight, all H outputs; partials summed over the ranks
  block_matvec_t(a.out_w + (size_t)m0 * H, H, nullptr, s_dl, m1 - m0, H, mv_scr, mv_cap, mv_quads, [](int i) { return i; }, [&](int i, float v) {
    for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_dhp, r)[R * H + i] = v;
  });
  if (m1 - m0 <= 0 && tid < H)
    for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_dhp, r)[R * H + tid] = 0.f;
  cluster.sync();
  DEC_STAMP(20);
  // ---- 3: LSTM cell backward (every rank, redundantly: H elements) ------------------------------------------------------------
  if (tid < H) {
    const int j = tid;
    float dh = 0.f;
    for (int r = 0; r < CL; ++r) dh += s_dhp[r * H + j];
    if (a.d_h_out) dh += a.d_h_out[(size_t)b * H + j];
    const float* g = a.gates + (size_t)b * 4 * H;
    const float gi = g[j], gf = g[H + j], gg = g[2 * H + j], go = g[3 * H + j];
    const float tc = tanh_fast(a.cell_out[(size_t)b * H + j]);
    const float dc = fmaf(dh * go, 1.f - tc * tc, a.d_cell_out ? a.d_cell_out[(size_t)b * H + j] : 0.f);
    const float di = dc * gg * gi * (1.f - gi), df = dc * a.cell_in[(size_t)b * H + j] * gf * (1.f - gf);
    const float dg = dc * gi * (1.f - gg * gg), dO = dh * tc * go * (1.f - go);
    s_dg[j] = di; s_dg[H + j] = df; s_dg[2 * H + j] = dg; s_dg[3 * H + j] = dO;
    if (R == 0) {
      float* o = a.d_gates + (size_t)b * a.ldg;
      o[j] = di; o[H + j] = df; o[2 * H + j] = dg; o[3 * H + j] = dO;
      a.d_cell[(size_t)b * H + j] = dc * gf;
    }
  }
  __syncthreads();
  DEC_STAMP(21);
  // ---- 4: d c3 = d_gates W_ih[:, :D]: outputs split over the ranks, gathered -----------------------------------------------------
  {
    const int per = split4(D, CL), d0 = min(D, R * per), d1 = min(D, d0 + per);
    block_matvec_t(a.Wcat_ctx, D, nullptr, s_dg, 4 * H, d1 - d0, mv_scr, mv_cap, mv_quads, [&](int i) { return d0 + i; }, [&](int i, float v) {
      for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_dctx, r)[d0 + i] = v;
    });
  }
  cluster.sync();
  DEC_STAMP(22);
  // ---- 5: modality soft-max + W_beta tanh backward; datt / dcov_tot of this rank's text rows ---------------------------------------
  const float beta1 = a.beta[b * 2 + 0], beta2 = a.beta[b * 2 + 1];
  {
    float db1 = 0.f, db2 = 0.f;
    if (R == 0)
      for (int d = tid; d < D; d += NT) {
        db1 = fmaf(a.ctx12[(size_t)b * D + d], s_dctx[d], db1);
        db2 = fmaf(a.ctx12[((size_t)a.B + b) * D + d], s_dctx[d], db2);
      }
    const float gc = a.g_cov ? a.g_cov[b] : 0.f;
    const int t0 = min(Lt, R * a.chunk), t1 = min(Lt, t0 + a.chunk);
    for (int t = t0 + tid; t < t1; t += NT) {
      float dcv = a.d_cov_out ? a.d_cov_out[(size_t)b * Lt + t] : 0.f;
      float g = a.d_att_cov ? a.d_att_cov[(size_t)b * Lt + t] : 0.f;
      if (a.g_cov) {                                              // d sum min(att, cov'): ties split evenly (torch.minimum)
        const float av = a.att[(size_t)b * Lt + t], cv = a.cov_out[(size_t)b * Lt + t];
        const float tie = av == cv ? 0.5f * gc : 0.f;
        g += av < cv ? gc : tie;
        dcv += cv < av ? gc : tie;
      }
      a.dcov_tot[(size_t)b * Lt + t] = dcv;
      g += dcv;                                                   // coverage' = coverage + att
      a.datt[(size_t)b * Lt + t] = g;
      db1 = fmaf(a.alpha[((size_t)b * 2 + 0) * Lt + t], g, db1);
      db2 = fmaf(a.alpha[((size_t)b * 2 + 1) * Lt + t], g, db2);
    }
    db1 = block_sum(db1, s_red);
    db2 = block_sum(db2, s_red);
    if (tid < CL) {
      float* dst = cluster.map_shared_rank(s_ex, tid) + R * 4;
      dst[1] = db1;
      dst[2] = db2;
    }
  }
  cluster.sync();
  {
    float db1 = 0.f, db2 = 0.f;
    for (int r = 0; r < CL; ++r) {
      db1 += s_ex[r * 4 + 1];
      db2 += s_ex[r * 4 + 2];
    }
    const float mix = beta1 * db1 + beta2 * db2;
    const float deb1 = beta1 * (db1 - mix), deb2 = beta2 * (db2 - mix);
    for (int d = tid; d < D; d += NT) {
      const float t1 = tanh_fast(a.pb[(size_t)b * D + d] + a.hw[(size_t)b * 4 * D + 2 * D + d]);
      const float t2 = tanh_fast(a.pb[((size_t)a.B + b) * D + d] + a.hw[(size_t)b * 4 * D + 3 * D + d]);
      const float p1 = deb1 * a.vb1[d] * (1.f - t1 * t1), p2 = deb2 * a.vb2[d] * (1.f - t2 * t2);
      s_dpre[d] = p1;
      s_dpre[D + d] = p2;
      if (R == 0) {
        a.d_pre_b[(size_t)b * D + d] = p1;
        a.d_pre_b[((size_t)a.B + b) * D + d] = p2;
        a.vec_acc[((size_t)b * 6 + 4) * D + d] += deb1 * t1;        // d v_beta_1 weight
        a.vec_acc[((size_t)b * 6 + 5) * D + d] += deb2 * t2;
      }
    }
    if (R == 0 && tid == 0) {
      a.scal_acc[b * 4 + 2] += deb1;
      a.scal_acc[b * 4 + 3] += deb2;
    }
  }
  __syncthreads();
  DEC_STAMP(23);
  // ---- 6: d c_k = beta_k d c3 + W_beta_k^T d_pre_k: the 2D outputs split over the ranks --------------------------------------------
  float* s_dc = s_scr + NT;                             // [2D]  d c_1 | d c_2, gathered (whole-step launch)
  {
    const int per = (2 * D + CL - 1) / CL, o0 = min(2 * D, R * per), o1 = min(2 * D, o0 + per);
    for (int k = 0; k < 2; ++k) {
      const int lo = max(o0, k * D), hi = min(o1, (k + 1) * D);
      const float bk = k == 0 ? beta1 : beta2;
      block_matvec_t(a.Wb13 + (size_t)k * D * D, D, nullptr, s_dpre + k * D, D, hi - lo, mv_scr, mv_cap, mv_quads && ((lo - k * D) & 3) == 0,
                     [&](int i) { return lo - k * D + i; },
                     [&](int i, float v) {
                       const int dd = lo - k * D + i;
                       const float x = fmaf(bk, s_dctx[dd], v);
                       a.d_ctx12[((size_t)k * a.B + b) * D + dd] = x;
                       if (a.sweeps)
                         for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_dc, r)[k * D + dd] = x;
                     });
    }
  }
  cluster.sync();      // no rank exits while another may still write into its shared memory; s_dc is complete
  if (!a.sweeps) return;

  // ==== the text sweeps of the step (decoder_step.cu: dec_attn_sweep1 / sweep2 / reduce_video), this rank's rows [t0, t1) ============
  const int lane = tid & 31, warp = tid >> 5;
  auto up4s = [](int v) { return (v + 3) & ~3; };
  float* s_da = s_dc + up4s(2 * D);                     // [2][chunk]  d alpha_k of this rank's rows, then alpha_k (d alpha_k - sum)
  float* s_rowc = s_da + up4s(2 * a.chunk);             // [4][chunk]  per-row scalars of this rank's rows: alpha_1 | alpha_2 | datt | cov
  float* s_vec = s_rowc + up4s(4 * a.chunk);            // [6][D]  v1 | wc1 | hw1 | v2 | wc2 | hw2
  const int PW = staged ? NW / 2 : NW;                  // warps per pass of the column-partial reduction (staged: half the buffer, two passes)
  float* s_part = s_vec + up4s(6 * D);                  // [PW][3][D]
  float* s_row = s_part + up4s(PW * 3 * D);             // [chunk]  d cov accumulation
  float* s_colp = s_row + up4s(a.chunk);                // [CL][2][3][D]  column partials of every rank (written remotely)
  float* s_in = s_colp + up4s(CL * 6 * D);              // [4H + 4D]  d_gates | d (W2 h) | d (W4 h) | d_pre_b
  // Both sweeps are written like stage B of the forward kernel (see there): a lane's per-column constants live in registers for the
  // whole sweep (zero past D, so the arithmetic is unpredicated), NJ = 7 for the model's D = 200 and the zero-padded 8 for any other D.
  using N7 = std::integral_constant<int, 7>;
  using N8 = std::integral_constant<int, 8>;
  const bool nj7 = D > 192 && D <= 224;
  DEC_STAMP(24);
  // ---- 7: d alpha_k[t] = beta_k datt[t] + d c_k . enc_k[t];  sum_t alpha d alpha over the cluster ----------------------------------
  for (int i = tid; i < D; i += NT) {
    s_vec[i] = a.v1[i];
    s_vec[D + i] = a.wc1[i];
    s_vec[2 * D + i] = a.hw[(size_t)b * 4 * D + i];
    s_vec[3 * D + i] = a.v2[i];
    s_vec[4 * D + i] = a.wc2[i];
    s_vec[5 * D + i] = a.hw[(size_t)b * 4 * D + D + i];
  }
  // the per-row scalars of both sweeps come in ONCE, here: read inside the sweeps they were dependent global loads at the end (sweep
  // 7) or in the middle (sweep 8) of every warp iteration -- ~800 exposed cycles each (tools/decoder_bwd_trace.py)
  for (int i = tid; i < n; i += NT) {
    s_row[i] = a.dcov_tot[(size_t)b * Lt + t0 + i];
    s_rowc[i] = a.alpha[((size_t)b * 2 + 0) * Lt + t0 + i];
    s_rowc[a.chunk + i] = a.alpha[((size_t)b * 2 + 1) * Lt + t0 + i];
    s_rowc[2 * a.chunk + i] = a.datt[(size_t)b * Lt + t0 + i];      // (written by this rank in stage 5)
    s_rowc[3 * a.chunk + i] = a.cov[(size_t)b * Lt + t0 + i];
  }
  __syncthreads();
  float s1 = 0.f, s2 = 0.f;
  auto sweep7 = [&](const float* __restrict__ ea0, const float* __restrict__ ei0, auto nj_tag) {
    constexpr int NJ = decltype(nj_tag)::value;
    float dca[NJ], dci[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int d = lane + 32 * j;
      dca[j] = d < D ? s_dc[d] : 0.f;
      dci[j] = d < D ? s_dc[D + d] : 0.f;
    }
    for (int i = warp * 2; i < n; i += NW * 2) {
      float d1[2] = {0.f, 0.f}, d2[2] = {0.f, 0.f};
      float eav[2][NJ], eiv[2][NJ];
#pragma unroll
      for (int u = 0; u < 2; ++u) {                     // loads first (memory-level parallelism)
        const float* ea = ea0 + (size_t)min(i + u, n - 1) * D;
        const float* ei = ei0 + (size_t)min(i + u, n - 1) * D;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int d = lane + 32 * j;
          eav[u][j] = d < D ? ea[d] : 0.f;
          eiv[u][j] = d < D ? ei[d] : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          d1[u] = fmaf(dca[j], eav[u][j], d1[u]);
          d2[u] = fmaf(dci[j], eiv[u][j], d2[u]);
        }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float x1 = warp_sum(d1[u]), x2 = warp_sum(d2[u]);
        if (lane == 0 && i + u < n) {
          const float g = s_rowc[2 * a.chunk + i + u];
          const float da1 = x1 + beta1 * g, da2 = x2 + beta2 * g;
          s_da[i + u] = da1;
          s_da[a.chunk + i + u] = da2;
          s1 = fmaf(s_rowc[i + u], da1, s1);
          s2 = fmaf(s_rowc[a.chunk + i + u], da2, s2);
        }
      }
    }
  };
  if (staged) {
    if (n > 0) tc::mbar_wait(bar_enc, 0);
    if (nj7) sweep7(s_st0, s_st1, N7{}); else sweep7(s_st0, s_st1, N8{});
  } else {
    const float* const gea = a.enc_a + ((size_t)b * Lt + t0) * D;
    const float* const gei = a.enc_i + ((size_t)b * Lt + t0) * D;
    if (nj7) sweep7(gea, gei, N7{}); else sweep7(gea, gei, N8{});
  }
  {
    s1 = block_sum(s1, s_red);
    if (staged && tid == 0 && n > 0) {       // every read of the enc rows is behind block_sum's barriers: the buffers take the proj rows
      tc::fence_proxy_async();
      tc::mbar_expect_tx(bar_proj, 2 * stage_bytes, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st0), a.proj_a + ((size_t)b * Lt + t0) * D, stage_bytes, bar_proj, 1);
      tc::tma_bulk_g2s(tc::smem_u32(s_st1), a.proj_i + ((size_t)b * Lt + t0) * D, stage_bytes, bar_proj, 1);
    }
    s2 = block_sum(s2, s_red);
    if (tid < CL) {
      float* dst = cluster.map_shared_rank(s_ex, tid) + R * 4;
      dst[0] = s1;
      dst[1] = s2;
    }
  }
  cluster.sync();
  float stot0 = 0.f, stot1 = 0.f;
  for (int r = 0; r < CL; ++r) {
    stot0 += s_ex[r * 4 + 0];
    stot1 += s_ex[r * 4 + 1];
  }
  DEC_STAMP(25);
  for (int i = tid; i < n; i += NT) {                   // d e_k[t] = alpha_k (d alpha_k - sum_t alpha_k d alpha_k), in place
    s_da[i] = s_rowc[i] * (s_da[i] - stot0);
    s_da[a.chunk + i] = s_rowc[a.chunk + i] * (s_da[a.chunk + i] - stot1);
  }
  __syncthreads();
  // ---- 8: soft-max backward, tanh backward, d proj (+=), d cov, column partials ------------------------------------------------------
  constexpr float K2 = 2.0f * 1.4426950408889634f;      // tanh x = 1 - 2 / (1 + 2^(K2 x)), flush-to-zero MUFU forms (no guard instructions)
  float se_m0 = 0.f, se_m1 = 0.f;
  // proj: row 0 of this rank's chunk.  STAGED: the rows sit in a stage buffer; d z overwrites them in place and the whole block is added
  // into d proj by ONE bulk reduction (d proj accumulates over the steps of the sequence: one writer per element and step, steps in
  // stream order -- deterministic); else d z goes out as predicated L2 reductions (a warp-wide RED per 128 bytes: ~as slow as the load -
  // add - store round trip it replaced).
  auto sweep8 = [&](const int m, float* proj, auto nj_tag, auto staged_tag) {
    constexpr int NJ = decltype(nj_tag)::value;
    constexpr bool STAGED = decltype(staged_tag)::value;
    float* dproj = (m == 0 ? a.d_proj_a : a.d_proj_i) + ((size_t)b * Lt + t0) * D;
    float vvr[NJ], wcr[NJ], hwk[NJ];                    // v, Wc, K2 (W h) of this lane's columns
    float c_dz[NJ], c_cov[NJ], c_v[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int d = lane + 32 * j;
      const float* vv = s_vec + 3 * m * D;
      vvr[j] = d < D ? vv[d] : 0.f;
      wcr[j] = d < D ? vv[D + d] : 0.f;
      hwk[j] = d < D ? vv[2 * D + d] * K2 : 0.f;
      c_dz[j] = c_cov[j] = c_v[j] = 0.f;
    }
    float se = 0.f;
    for (int i0 = warp * 2; i0 < n; i0 += NW * 2) {     // two sentences per warp iteration: every load in flight before the first tanh
      float cvs[2], dets[2], pv[2][NJ];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int i = min(i0 + u, n - 1);
        cvs[u] = s_rowc[3 * a.chunk + i];
        dets[u] = i0 + u < n ? s_da[m * a.chunk + i] : 0.f;          // a row past the end: all zero
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int d = lane + 32 * j;
          pv[u][j] = d < D ? proj[(size_t)i * D + d] : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int i = i0 + u;
        const bool valid = i < n;
        const float cv = cvs[u], det = dets[u], cvk = cv * K2;
        float row = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int d = lane + 32 * j;
          const float tz = fmaf(-2.0f, rcp_ftz(1.0f + tc::fast_exp2(fmaf(cvk, wcr[j], fmaf(pv[u][j], K2, hwk[j])))), 1.0f);
          const float dz = det * vvr[j] * (1.f - tz * tz);
          if (STAGED) {
            if (valid && d < D) proj[(size_t)i * D + d] = dz;
          } else {
            red_add_f32_if(dproj + (size_t)i * D + d, dz, valid && d < D);
          }
          c_dz[j] += dz;
          c_cov[j] = fmaf(dz, cv, c_cov[j]);
          c_v[j] = fmaf(det, tz, c_v[j]);
          row = fmaf(dz, wcr[j], row);
        }
        row = warp_sum(row);
        if (lane == 0 && valid) {
          s_row[i] += row;
          se += det;
        }
      }
    }
    if (STAGED) tc::fence_proxy_async();                // this thread's d z stores, before the bulk reduction reads them
    se = block_sum(se, s_red);                          // (its barriers: every warp is done with its rows)
    if (m == 0) se_m0 = se; else se_m1 = se;
    if (STAGED && tid == 0 && n > 0) {
      bulk_reduce_add_f32(dproj, tc::smem_u32(proj), stage_bytes);
      bulk_commit();
    }
    // column partials: per-warp rows -> fixed-order sum over the warps (PW warps per pass) -> slot R of every rank
    float xacc[2] = {0.f, 0.f};                         // outputs tid and tid + NT of the 3 D (D <= 256)
    for (int w0 = 0; w0 < NW; w0 += PW) {
      if (warp >= w0 && warp < w0 + PW) {
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int d = lane + 32 * j;
          if (d < D) {
            s_part[((warp - w0) * 3 + 0) * D + d] = c_dz[j];
            s_part[((warp - w0) * 3 + 1) * D + d] = c_cov[j];
            s_part[((warp - w0) * 3 + 2) * D + d] = c_v[j];
          }
        }
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int i = tid + q * NT;
        if (i < 3 * D)
          for (int w = 0; w < PW; ++w) xacc[q] += s_part[w * 3 * D + i];
      }
      __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int i = tid + q * NT;
      if (i < 3 * D)
        for (int r = 0; r < CL; ++r) cluster.map_shared_rank(s_colp, r)[(R * 2 + m) * 3 * D + i] = xacc[q];
    }
  };
  if (staged && n > 0) tc::mbar_wait(bar_proj, 0);
  for (int m = 0; m < 2; ++m) {
    if (staged) {
      float* const sp = m == 0 ? s_st0 : s_st1;
      if (nj7) sweep8(m, sp, N7{}, std::true_type{}); else sweep8(m, sp, N8{}, std::true_type{});
    } else {
      float* const gp = const_cast<float*>(m == 0 ? a.proj_a : a.proj_i) + ((size_t)b * Lt + t0) * D;      // (read only on this path)
      if (nj7) sweep8(m, gp, N7{}, std::false_type{}); else sweep8(m, gp, N8{}, std::false_type{});
    }
  }
  for (int i = tid; i < n; i += NT) a.d_cov[(size_t)b * Lt + t0 + i] = s_row[i];
  if (tid < CL) {
    float* dst = cluster.map_shared_rank(s_ex, tid) + R * 4;
    dst[2] = se_m0;
    dst[3] = se_m1;
  }
  cluster.sync();
  DEC_STAMP(26);
  // ---- 9: the column sums over the cluster (fixed order) -> d (W2 h) | d (W4 h), parameter-gradient accumulators; d h -----------------
  for (int i = tid; i < 2 * D; i += NT) {
    const int m = i / D, d = i - m * D;
    float x = 0.f, y = 0.f, z = 0.f;
    for (int r = 0; r < CL; ++r) {
      const float* q = s_colp + (r * 2 + m) * 3 * D;
      x += q[d];
      y += q[D + d];
      z += q[2 * D + d];
    }
    s_in[4 * H + m * D + d] = x;
    s_in[4 * H + (2 + m) * D + d] = s_dpre[m * D + d];
    if (R == 0) {
      float* o = a.d_gates + (size_t)b * a.ldg + 4 * H;                   // d_hw4 sits beside d_gates
      o[m * D + d] = x;
      o[(2 + m) * D + d] = s_dpre[m * D + d];
      a.vec_acc[((size_t)b * 6 + m) * D + d] += y;                         // d Wc weight
      a.vec_acc[((size_t)b * 6 + 2 + m) * D + d] += z;                     // d v weight
    }
  }
  for (int i = tid; i < 4 * H; i += NT) s_in[i] = s_dg[i];
  if (R == 0 && tid < 2) {
    float sv = 0.f;
    for (int r = 0; r < CL; ++r) sv += s_ex[r * 4 + 2 + tid];
    a.scal_acc[b * 4 + tid] += sv;                                         // d v bias (identically 0 up to rounding)
  }
  __syncthreads();
  {
    const int per = split4(H, CL), j0 = min(H, R * per), j1 = min(H, j0 + per);
    block_matvec_t(a.Wh_stack, H, nullptr, s_in, 4 * H + 4 * D, j1 - j0, mv_scr, mv_cap, mv_quads, [&](int i) { return j0 + i; },
                   [&](int i, float v) { a.d_h[(size_t)b * H + j0 + i] = v; });
  }
  if (staged && tid == 0) bulk_wait_all();              // the stage buffers are read by the bulk reductions until here
  DEC_STAMP(27);
  // (No barrier before the exit: the last stores into another rank's shared memory -- the column partials of sweep 8 -- lie before
  // the cluster barrier in front of stage 9.)
}

static size_t g_head_smem_set = 0;   // dynamic shared memory the kernel attribute of dec_bwd_head_kernel allows (both launchers share it)

static size_t head_smem_bytes(int D, int H, int M, int CL, int chunk = 0, bool sweeps = false, int PW = NW) {
  auto up4 = [](size_t v) { return (v + 3) & ~(size_t)3; };
  const size_t per_m = (M + CL - 1) / CL;
  size_t floats = up4(per_m) + up4((size_t)MAXC * H) + up4(4 * H) + up4(D) + up4(2 * D) + MAXC * 4 + 32 + NT;
  if (sweeps)
    floats += up4(2 * D) + up4(2 * (size_t)chunk) + up4(4 * (size_t)chunk) + up4(6 * D) + up4((size_t)PW * 3 * D) + up4(chunk) + up4((size_t)CL * 6 * D) +
              up4(4 * H + 4 * D);
  return floats * sizeof(float) + 64;
}

// bytes of dynamic shared memory for the launch below
static size_t fused_smem_bytes(int Lt, int D, int H, int E, int M, int CL, int* chunk_out) {
  const int chunk = (Lt + CL - 1) / CL;
  const int K = D + E + H;
  const int groups = (D & 3) == 0 ? NT / (D >> 2) : NT / D;
  const int per_m = (M + CL - 1) / CL;
  int cpart = groups * 2 * D;
  if (cpart < per_m) cpart = per_m;
  auto up4 = [](size_t v) { return (v + 3) & ~(size_t)3; };
  const size_t floats = up4(4 * D) + up4(K) + 2 * up4(2 * D) + up4(H) + up4((size_t)MAXC * (4 + 2 * D)) + MAXC * 8 +
                        up4(4 * (split4(H, MAXC / 2) + 1)) + 32 + SCR + up4(4 * D) + up4(2 * (size_t)chunk) + up4(chunk) + up4(cpart);
  if (chunk_out) *chunk_out = chunk;
  return floats * sizeof(float) + 64;
}

// floats of the beam region (see dec_fused_body): the tables, the selection exchange and K slots of state; constrained, also every
// slot's eligible bits and kept count, in and out
static size_t beam_floats(int K, int CL, int chunk, int H, int M, bool constrained = false) {
  auto up4 = [](size_t v) { return (v + 3) & ~(size_t)3; };
  const size_t ldp = up4((M + CL - 1) / CL);
  const size_t per_slot = 2 * (up4(H) + up4(split4(H, CL)) + up4(chunk)) + ldp;
  const size_t cons = constrained ? 2 * (size_t)K * ((ldp + 31) / 32) + 2 * MAXK : 0;
  return 7 * MAXK + MAXC * MAXK * 4 + NW * 4 + MAXK * 4 + (size_t)K * per_slot + cons;
}

// floats of the nucleus region (see nucleus_cut): every rank's copy of the row, the histogram (u64) and the block exchanges (u64)
static size_t nucleus_floats(int M) { return (((size_t)M + 3) & ~(size_t)3) + 2 * kNucBuckets + 2 * 32; }

// floats the stochastic beam adds: the ninth exchange entry of every rank and of this rank's list (they lengthen the beam region),
// then the stochastic region (phi / key tables, lam, the three exchanges of the normaliser and Z, every candidate's key)
constexpr size_t kStochBeamExtra = MAXC * 4 + 4;
static size_t stoch_floats(int K, int CL, int M) {
  const size_t ldp = (((size_t)M + CL - 1) / CL + 3) & ~(size_t)3;
  return 5 * MAXK + 2 * MAXC * MAXK + 2 * MAXC * MAXK + (size_t)K * ldp;
}

// Shape checks, cluster size, shared memory and row stage of the forward cluster kernels, then the launch: `g` null launches one step
// (dec_step_fused_kernel), else the greedy roll-out (dec_greedy_fused_kernel), or with `bm` the beam roll-out (dec_beam_fused_kernel);
// with `cn` the constrained roll-out of either (dec_greedy_constrained_kernel, dec_beam_constrained_kernel); with `sp` (not `bm`) the
// sampled roll-out (dec_sample_kernel, with `cn` dec_sample_constrained_kernel), one cluster per (video, sample); with `sp` and `nu`
// the nucleus roll-out (dec_sample_nucleus_kernel, with `cn` dec_sample_nucleus_constrained_kernel); with `bm` and `sb` the
// stochastic beam (dec_beam_sample_kernel, with `cn` dec_beam_sample_constrained_kernel).
static int launch_fused(FusedArgs a, const GreedyArgs* g, const char* who, mmb_stream_t stream, BeamArgs* bm = nullptr,
                        const ConstraintArgs* cn = nullptr, SampleArgs* sp = nullptr, NucleusArgs* nu = nullptr,
                        StochArgs* sb = nullptr) {
  const int B = a.B, Lt = a.Lt, D = a.D, H = a.H, E = a.E, M = a.M;
  MMB_REQUIRE(B > 0 && Lt > 0 && D > 0 && H > 0 && E >= 0 && M > 0, MMB_ERR_INVALID,
              "%s: B=%d Lt=%d D=%d H=%d E=%d M=%d", who, B, Lt, D, H, E, M);
  MMB_REQUIRE(D <= 256, MMB_ERR_UNSUPPORTED, "%s: D=%d > 256", who, D);
  const int rows = sp ? B * sp->N : B;     // clusters: one per video, or per (video, sample)
  // few videos: eight CTAs per video keep more of the chip busy on the text sweep
  const int CL = (long long)rows * 4 * 2 <= 160 ? 8 : 4;
  size_t smem = fused_smem_bytes(Lt, D, H, E, M, CL, &a.chunk);
  MMB_REQUIRE(smem <= 200 * 1024, MMB_ERR_UNSUPPORTED, "%s: %zu B of shared memory (Lt=%d)", who, smem, Lt);
  // constrained greedy: a thread keeps the eligible bits of its sentences in one 32-bit register
  MMB_REQUIRE(!cn || bm || (M + CL - 1) / CL <= 32 * NT, MMB_ERR_UNSUPPORTED, "%s: M=%d > %d sentences per CTA", who, M, 32 * NT);
  if (bm) {                                // the beam region behind the base arrays; the row stage follows if it still fits
    bm->off = (int)((smem + 15) / 16 * 4);
    smem = ((size_t)bm->off + beam_floats(bm->K, CL, a.chunk, H, M, cn != nullptr)) * 4 + 64;
    if (sb) {                              // stochastic: the longer exchange, then its region
      sb->off = (int)(((size_t)bm->off + beam_floats(bm->K, CL, a.chunk, H, M, cn != nullptr) + kStochBeamExtra + 3) & ~(size_t)3);
      smem = ((size_t)sb->off + stoch_floats(bm->K, CL, M)) * 4 + 64;
    }
    MMB_REQUIRE(smem <= 227 * 1024, MMB_ERR_UNSUPPORTED, "%s: width %d needs %zu B of shared memory per CTA, more than 232448 (B=%d Lt=%d M=%d)",
                who, bm->K, smem, B, Lt, M);
  } else if (sp) {                         // sampled: the beam region's tables and exchange arrays, no slots
    sp->off = (int)((smem + 15) / 16 * 4);
    smem = ((size_t)sp->off + beam_floats(0, CL, a.chunk, H, M)) * 4 + 64;
    if (nu) {                              // nucleus: its region behind the exchange arrays
      nu->off = (int)((smem + 15) / 16 * 4);
      smem = ((size_t)nu->off + nucleus_floats(M)) * 4 + 64;
      MMB_REQUIRE(smem <= 227 * 1024, MMB_ERR_UNSUPPORTED, "%s: the nucleus row of M=%d needs %zu B of shared memory per CTA, more than "
                  "232448 (Lt=%d)", who, M, smem, Lt);
    }
  }
  {
    // the row stage (see the kernel): two buffers of chunk x D floats behind two mbarriers, when they fit and bulk copies apply
    // (16-byte row granularity).  MMB_DEC_STAGE=0 turns it off (A/B measurements; read once per process, on the first launch: the
    // cross-check in tests/test_decoder_paths_gpu.py sets it in a child process).
    static const char* stage_env = getenv("MMB_DEC_STAGE");
    const size_t base_floats = (smem + 15) / 16 * 4;
    const size_t stage_floats = 4 + 2 * (((size_t)a.chunk * D + 3) & ~(size_t)3);
    const bool enc_aligned = ((reinterpret_cast<uintptr_t>(a.enc_a) | reinterpret_cast<uintptr_t>(a.enc_i)) & 15) == 0;
    const bool aligned = enc_aligned && ((reinterpret_cast<uintptr_t>(a.proj_a) | reinterpret_cast<uintptr_t>(a.proj_i)) & 15) == 0;
    // with D % 4 == 0 every row start keeps the base pointer's alignment: float4 context loads when the bases are 16-byte aligned
    a.ctx_vec4 = (D & 3) == 0 && enc_aligned;
    if ((D & 3) == 0 && aligned && (base_floats + stage_floats) * 4 <= 227 * 1024 && !(stage_env && atoi(stage_env) == 0)) {
      a.stage_off = (int)base_floats;
      smem = (base_floats + stage_floats) * 4;
    }
  }
  static size_t smem_set[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  const int which = sb ? (cn ? 10 : 9) : nu ? (cn ? 8 : 7) : sp ? (cn ? 6 : 5) : bm ? (cn ? 4 : 2) : g ? (cn ? 3 : 1) : 0;
  if (smem > smem_set[which]) {
    const void* fn = which == 10 ? (const void*)dec_beam_sample_constrained_kernel : which == 9 ? (const void*)dec_beam_sample_kernel
                   : which == 8 ? (const void*)dec_sample_nucleus_constrained_kernel : which == 7 ? (const void*)dec_sample_nucleus_kernel
                   : which == 6 ? (const void*)dec_sample_constrained_kernel : which == 5 ? (const void*)dec_sample_kernel
                   : which == 4 ? (const void*)dec_beam_constrained_kernel : which == 3 ? (const void*)dec_greedy_constrained_kernel
                   : which == 2 ? (const void*)dec_beam_fused_kernel : which == 1 ? (const void*)dec_greedy_fused_kernel
                                : (const void*)dec_step_fused_kernel;
    MMB_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set[which] = smem;
  }
  static const char* trace_env = getenv("MMB_DEC_TRACE");
  static bool trace_set = false;
  if (trace_env && !trace_set) {
    long long* ptr = reinterpret_cast<long long*>(strtoull(trace_env, nullptr, 0));
    MMB_CUDA(cudaMemcpyToSymbol(g_dec_trace, &ptr, sizeof(ptr)));
    trace_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(rows * CL));
  cfg.blockDim = dim3(NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (sb && cn) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_beam_sample_constrained_kernel, a, *g, *bm, *cn, *sb));
    return check_launch("dec_beam_sample_constrained_kernel");
  }
  if (sb) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_beam_sample_kernel, a, *g, *bm, *sb));
    return check_launch("dec_beam_sample_kernel");
  }
  if (nu && cn) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_sample_nucleus_constrained_kernel, a, *g, *cn, *sp, *nu));
    return check_launch("dec_sample_nucleus_constrained_kernel");
  }
  if (nu) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_sample_nucleus_kernel, a, *g, *sp, *nu));
    return check_launch("dec_sample_nucleus_kernel");
  }
  if (sp && cn) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_sample_constrained_kernel, a, *g, *cn, *sp));
    return check_launch("dec_sample_constrained_kernel");
  }
  if (sp) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_sample_kernel, a, *g, *sp));
    return check_launch("dec_sample_kernel");
  }
  if (cn && bm) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_beam_constrained_kernel, a, *g, *bm, *cn));
    return check_launch("dec_beam_constrained_kernel");
  }
  if (cn) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_greedy_constrained_kernel, a, *g, *cn));
    return check_launch("dec_greedy_constrained_kernel");
  }
  if (bm) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_beam_fused_kernel, a, *g, *bm));
    return check_launch("dec_beam_fused_kernel");
  }
  if (g) {
    MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_greedy_fused_kernel, a, *g));
    return check_launch("dec_greedy_fused_kernel");
  }
  MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_step_fused_kernel, a));
  return check_launch("dec_step_fused_kernel");
}

}  // namespace mmb

extern "C" int mmb_decoder_step_fused_fwd(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                          const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                          const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                          const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt,
                                          const float* bcat, const float* out_wt, const float* out_b, const float* sent,
                                          const float* h, const float* cell, const float* cov, const uint8_t* mask,
                                          const long long* target, float* probs, float* h_out, float* cell_out, float* att_cov,
                                          float* cov_out, long long* argmax, float* nll, float* cov_loss, float* hw, float* alpha,
                                          float* beta, float* ctx12, float* pb, float* xcat, float* gates, int B, int Lt, int D,
                                          int H, int E, int M, mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && sent && h && cell && cov && mask && probs && h_out &&
                  cell_out && att_cov && cov_out && hw && alpha && beta && ctx12 && pb && xcat && gates,
              MMB_ERR_INVALID, "mmb_decoder_step_fused_fwd: null pointer");
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              sent, h, cell, cov, mask, target, probs, h_out, cell_out, att_cov, cov_out, argmax, nll, cov_loss, hw, alpha, beta,
              ctx12, pb, xcat, gates, B, Lt, D, H, E, M, 0, 0};
  return launch_fused(a, nullptr, "mmb_decoder_step_fused_fwd", stream);
}

extern "C" int mmb_decoder_greedy_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                        const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                        const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                        const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                        const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                        const uint8_t* mask, const long long* target, float* probs, long long* argmax,
                                        float* loss_terms, int B, int Lt, int D, int H, int E, int M, int S, int T,
                                        mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && emb_text && h0 && mask && probs && argmax,
              MMB_ERR_INVALID, "mmb_decoder_greedy_fused: null pointer");
  MMB_REQUIRE(S > 0 && (!target || (loss_terms && T >= S)), MMB_ERR_INVALID, "mmb_decoder_greedy_fused: S=%d T=%d, target %s, loss_terms %s",
              S, T, target ? "set" : "null", loss_terms ? "set" : "null");
  // (the per-step inputs and the saved arrays of the step kernel stay null: the roll-out keeps its state on chip)
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              nullptr, nullptr, nullptr, nullptr, mask, target, probs, nullptr, nullptr, nullptr, nullptr, argmax,
              target ? loss_terms : nullptr, target ? loss_terms + B : nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
              nullptr, B, Lt, D, H, E, M, 0, 0};
  const GreedyArgs g{emb_text, h0, S, target ? T : 0};
  return launch_fused(a, &g, "mmb_decoder_greedy_fused", stream);
}

extern "C" int mmb_decoder_beam_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                      const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                      const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                      const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                      const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                      const uint8_t* mask, const int* text_len, long long* tokens, int* parents, float* scores,
                                      float* probs, long long* best, int* path, int B, int Lt, int D, int H, int E, int M, int K,
                                      int S, mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && emb_text && h0 && mask && text_len && tokens && parents &&
                  scores && probs && best && path,
              MMB_ERR_INVALID, "mmb_decoder_beam_fused: null pointer");
  MMB_REQUIRE(K >= 1 && K <= MAXK && S > 0, MMB_ERR_INVALID, "mmb_decoder_beam_fused: width K=%d (1..%d), S=%d", K, MAXK, S);
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              nullptr, nullptr, nullptr, nullptr, mask, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
              nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, B, Lt, D, H, E, M, 0, 0};
  const GreedyArgs g{emb_text, h0, S, 0};
  BeamArgs bm{text_len, tokens, parents, scores, probs, best, path, K, 0};
  return launch_fused(a, &g, "mmb_decoder_beam_fused", stream, &bm);
}

extern "C" int mmb_decoder_greedy_constrained_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                                    const float* Wh4t, const float* bh4, const float* v1, const float* wc1,
                                                    const float* v2, const float* wc2, const float* v1b, const float* v2b,
                                                    const float* Wb13t, const float* vb1, const float* vb2, const float* vb1b,
                                                    const float* vb2b, const float* Wcatt, const float* bcat, const float* out_wt,
                                                    const float* out_b, const float* emb_text, const float* h0, const uint8_t* mask,
                                                    const int* text_len, float* probs, long long* argmax, int B, int Lt, int D,
                                                    int H, int E, int M, int S, int no_repeat, int min_sentences,
                                                    mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && emb_text && h0 && mask && text_len && probs && argmax,
              MMB_ERR_INVALID, "mmb_decoder_greedy_constrained_fused: null pointer");
  MMB_REQUIRE(S > 0 && (no_repeat == 0 || no_repeat == 1) && min_sentences >= 0, MMB_ERR_INVALID,
              "mmb_decoder_greedy_constrained_fused: S=%d no_repeat=%d (0 or 1) min_sentences=%d (>= 0)", S, no_repeat, min_sentences);
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              nullptr, nullptr, nullptr, nullptr, mask, nullptr, probs, nullptr, nullptr, nullptr, nullptr, argmax,
              nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, B, Lt, D, H, E, M, 0, 0};
  const GreedyArgs g{emb_text, h0, S, 0};
  const ConstraintArgs cn{text_len, no_repeat, min_sentences};
  return launch_fused(a, &g, "mmb_decoder_greedy_constrained_fused", stream, nullptr, &cn);
}

extern "C" int mmb_decoder_beam_constrained_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                                  const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                                  const float* wc2, const float* v1b, const float* v2b, const float* Wb13t,
                                                  const float* vb1, const float* vb2, const float* vb1b, const float* vb2b,
                                                  const float* Wcatt, const float* bcat, const float* out_wt, const float* out_b,
                                                  const float* emb_text, const float* h0, const uint8_t* mask, const int* text_len,
                                                  long long* tokens, int* parents, float* scores, float* probs, long long* best,
                                                  int* path, int B, int Lt, int D, int H, int E, int M, int K, int S, int no_repeat,
                                                  int min_sentences, mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && emb_text && h0 && mask && text_len && tokens && parents &&
                  scores && probs && best && path,
              MMB_ERR_INVALID, "mmb_decoder_beam_constrained_fused: null pointer");
  MMB_REQUIRE(K >= 1 && K <= MAXK && S > 0 && (no_repeat == 0 || no_repeat == 1) && min_sentences >= 0, MMB_ERR_INVALID,
              "mmb_decoder_beam_constrained_fused: width K=%d (1..%d), S=%d, no_repeat=%d (0 or 1), min_sentences=%d (>= 0)", K, MAXK,
              S, no_repeat, min_sentences);
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              nullptr, nullptr, nullptr, nullptr, mask, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
              nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, B, Lt, D, H, E, M, 0, 0};
  const GreedyArgs g{emb_text, h0, S, 0};
  BeamArgs bm{text_len, tokens, parents, scores, probs, best, path, K, 0};
  const ConstraintArgs cn{text_len, no_repeat, min_sentences};
  return launch_fused(a, &g, "mmb_decoder_beam_constrained_fused", stream, &bm, &cn);
}

extern "C" int mmb_decoder_beam_sample_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                             const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                             const float* wc2, const float* v1b, const float* v2b, const float* Wb13t,
                                             const float* vb1, const float* vb2, const float* vb1b, const float* vb2b,
                                             const float* Wcatt, const float* bcat, const float* out_wt, const float* out_b,
                                             const float* emb_text, const float* h0, const uint8_t* mask, const int* text_len,
                                             const unsigned long long* key, long long* tokens, int* parents, float* scores,
                                             float* probs, float* phi, float* keys, long long* paths, int* path_slots, float* kappa,
                                             int B, int Lt, int D, int H, int E, int M, int K, int S, float T, int no_repeat,
                                             int min_sentences, mmb_stream_t stream) {
  using namespace mmb;
  const char* who = "mmb_decoder_beam_sample_fused";
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && emb_text && h0 && mask && text_len && key && tokens &&
                  parents && scores && probs && phi && keys && paths && path_slots && kappa,
              MMB_ERR_INVALID, "%s: null pointer", who);
  MMB_REQUIRE(K >= 1 && K <= MAXK && S > 0 && T > 0.f && isfinite(T) && (no_repeat == 0 || no_repeat == 1) && min_sentences >= 0,
              MMB_ERR_INVALID, "%s: width K=%d (1..%d), S=%d, T=%g (finite, > 0), no_repeat=%d (0 or 1), min_sentences=%d (>= 0)", who,
              K, MAXK, S, (double)T, no_repeat, min_sentences);
  MMB_REQUIRE(B > 0 && M > 0, MMB_ERR_INVALID, "%s: B=%d M=%d", who, B, M);
  MMB_REQUIRE((unsigned long long)B * S * K * M + B <= (1ull << 32), MMB_ERR_UNSUPPORTED,
              "%s: B S K M + B = %d x %d x %d x %d + %d exceeds the 2^32 counters of a key", who, B, S, K, M, B);
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              nullptr, nullptr, nullptr, nullptr, mask, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
              nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, B, Lt, D, H, E, M, 0, 0};
  const GreedyArgs g{emb_text, h0, S, 0};
  BeamArgs bm{text_len, tokens, parents, scores, probs, nullptr, nullptr, K, 0};
  const ConstraintArgs cn{text_len, no_repeat, min_sentences};
  StochArgs sb{key, T, phi, keys, paths, path_slots, kappa, 0};
  return launch_fused(a, &g, who, stream, &bm, no_repeat != 0 || min_sentences != 0 ? &cn : nullptr, nullptr, nullptr, &sb);
}

namespace mmb {
// the sampled roll-out (nu null) or the nucleus roll-out: argument checks, then launch_fused
static int sample_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                        const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                        const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                        const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                        const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                        const uint8_t* mask, const int* text_len, const unsigned long long* key, float* probs,
                        long long* tokens, int B, int Lt, int D, int H, int E, int M, int S, int N, float T,
                        int top_k, int no_repeat, int min_sentences, mmb_stream_t stream, NucleusArgs* nu, const char* who) {
  const bool constrained = no_repeat != 0 || min_sentences != 0;
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && Wh4t && bh4 && v1 && wc1 && v2 && wc2 && v1b && v2b && Wb13t && vb1 && vb2 &&
                  vb1b && vb2b && Wcatt && bcat && out_wt && out_b && emb_text && h0 && mask && key && probs && tokens &&
                  (text_len || !constrained),
              MMB_ERR_INVALID, "%s: null pointer", who);
  MMB_REQUIRE(S > 0 && N >= 1 && N <= 64 && T > 0.f && isfinite(T) && top_k >= 0 && top_k <= MAXK && (no_repeat == 0 || no_repeat == 1) &&
                  min_sentences >= 0,
              MMB_ERR_INVALID,
              "%s: S=%d, N=%d (1..64), T=%g (finite, > 0), top_k=%d (0..%d), no_repeat=%d (0 or 1), "
              "min_sentences=%d (>= 0)", who, S, N, (double)T, top_k, MAXK, no_repeat, min_sentences);
  MMB_REQUIRE(B > 0 && M > 0, MMB_ERR_INVALID, "%s: B=%d M=%d", who, B, M);
  MMB_REQUIRE((unsigned long long)B * N * S * M <= (1ull << 32), MMB_ERR_UNSUPPORTED,
              "%s: B N S M = %d x %d x %d x %d exceeds the 2^32 counters of a key", who, B, N, S, M);
  FusedArgs a{proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat, out_wt, out_b,
              nullptr, nullptr, nullptr, nullptr, mask, nullptr, probs, nullptr, nullptr, nullptr, nullptr, tokens,
              nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, B, Lt, D, H, E, M, 0, 0};
  const GreedyArgs g{emb_text, h0, S, 0};
  const ConstraintArgs cn{text_len, no_repeat, min_sentences};
  SampleArgs sp{key, T, N, top_k, 0};
  return launch_fused(a, &g, who, stream, nullptr, constrained ? &cn : nullptr, &sp, nu);
}
}  // namespace mmb

extern "C" int mmb_decoder_sample_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                        const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                        const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                        const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                        const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                        const uint8_t* mask, const int* text_len, const unsigned long long* key, float* probs,
                                        long long* tokens, int B, int Lt, int D, int H, int E, int M, int S, int N, float T,
                                        int top_k, int no_repeat, int min_sentences, mmb_stream_t stream) {
  return mmb::sample_fused(proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt,
                           bcat, out_wt, out_b, emb_text, h0, mask, text_len, key, probs, tokens, B, Lt, D, H, E, M, S, N, T, top_k,
                           no_repeat, min_sentences, stream, nullptr, "mmb_decoder_sample_fused");
}

extern "C" int mmb_decoder_sample_nucleus_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                                const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                                const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                                const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                                const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                                const uint8_t* mask, const int* text_len, const unsigned long long* key, float* probs,
                                                long long* tokens, int B, int Lt, int D, int H, int E, int M, int S, int N, float T,
                                                int top_k, int no_repeat, int min_sentences, float top_p,
                                                mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(top_p > 0.f && top_p <= 1.f, MMB_ERR_INVALID, "mmb_decoder_sample_nucleus_fused: top_p=%g (in (0, 1])", (double)top_p);
  // the integer masses of the rule: P Q < 2^24 2^24 M fits 64 bits
  MMB_REQUIRE(top_p == 1.f || M < 65536, MMB_ERR_UNSUPPORTED, "mmb_decoder_sample_nucleus_fused: M=%d (below 65536 with top_p < 1)", M);
  NucleusArgs nu{(uint32_t)rintf(top_p * 16777216.f), 0};
  return sample_fused(proj_a, proj_i, enc_a, enc_i, Wh4t, bh4, v1, wc1, v2, wc2, v1b, v2b, Wb13t, vb1, vb2, vb1b, vb2b, Wcatt, bcat,
                      out_wt, out_b, emb_text, h0, mask, text_len, key, probs, tokens, B, Lt, D, H, E, M, S, N, T, top_k, no_repeat,
                      min_sentences, stream, top_p == 1.f ? nullptr : &nu, "mmb_decoder_sample_nucleus_fused");   // (1: no cut, the sampled roll-out)
}

extern "C" int mmb_decoder_bwd_head(const float* probs, const float* d_probs, const long long* target, const float* g_nll,
                                    const float* g_cov, const float* out_w, const float* gates, const float* cell_in,
                                    const float* cell_out, const float* d_h_out, const float* d_cell_out, const float* Wcat_ctx,
                                    const float* d_att_cov, const float* d_cov_out, const float* alpha, const float* beta,
                                    const float* ctx12, const float* pb, const float* hw, const float* vb1, const float* vb2,
                                    const float* att, const float* cov_out, const float* Wb13, float* d_logits, int ldd, float* d_gates,
                                    int ldg, float* d_cell, float* datt, float* dcov_tot, float* d_pre_b, float* d_ctx12, float* vec_acc,
                                    float* scal_acc, int B, int Lt, int D, int H, int M, mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(probs && out_w && gates && cell_in && cell_out && Wcat_ctx && alpha && beta && ctx12 && pb && hw && vb1 && vb2 && Wb13 &&
                  d_logits && d_gates && d_cell && datt && dcov_tot && d_pre_b && d_ctx12 && vec_acc && scal_acc,
              MMB_ERR_INVALID, "mmb_decoder_bwd_head: null pointer");
  MMB_REQUIRE((!target || g_nll) && (!g_cov || (att && cov_out)), MMB_ERR_INVALID, "mmb_decoder_bwd_head: loss-term pointers");
  MMB_REQUIRE(B > 0 && Lt > 0 && D > 0 && H > 0 && M > 0 && ldd >= M && ldg >= 4 * H && H <= NT, MMB_ERR_INVALID,
              "mmb_decoder_bwd_head: B=%d Lt=%d D=%d H=%d M=%d ldd=%d ldg=%d", B, Lt, D, H, M, ldd, ldg);
  const int CL = (long long)B * 4 * 2 <= 160 ? 8 : 4;
  HeadArgs a{probs, d_probs, target, g_nll, g_cov, out_w, gates, cell_in, cell_out, d_h_out, d_cell_out, Wcat_ctx, d_att_cov, d_cov_out,
             alpha, beta, ctx12, pb, hw, vb1, vb2, att, cov_out, Wb13, d_logits, d_gates, d_cell, datt, dcov_tot, d_pre_b, d_ctx12,
             vec_acc, scal_acc, B, Lt, D, H, M, ldd, ldg, (Lt + CL - 1) / CL,
             0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0};
  const size_t smem = head_smem_bytes(D, H, M, CL);
  MMB_REQUIRE(smem <= 200 * 1024, MMB_ERR_UNSUPPORTED, "mmb_decoder_bwd_head: %zu B of shared memory", smem);
  if (smem > g_head_smem_set) {
    MMB_CUDA(cudaFuncSetAttribute(dec_bwd_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    g_head_smem_set = smem;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(B * CL));
  cfg.blockDim = dim3(NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_bwd_head_kernel, a));
  return check_launch("dec_bwd_head_kernel");
}

// The WHOLE backward step as one cluster kernel: mmb_decoder_bwd_head + the two text sweeps of mmb_decoder_attn_bwd + d h =
// [d_gates | d_hw4] Wh_stack (a library GEMM before).  d_gates points at a (B, ldg) buffer with ldg >= 4H + 4D: d_hw4 is written beside
// d_gates.  One launch per backward step instead of four.
extern "C" int mmb_decoder_step_fused_bwd(const float* probs, const float* d_probs, const long long* target, const float* g_nll,
                                          const float* g_cov, const float* out_w, const float* gates, const float* cell_in,
                                          const float* cell_out, const float* d_h_out, const float* d_cell_out, const float* Wcat_ctx,
                                          const float* d_att_cov, const float* d_cov_out, const float* alpha, const float* beta,
                                          const float* ctx12, const float* pb, const float* hw, const float* vb1, const float* vb2,
                                          const float* att, const float* cov_out, const float* Wb13, float* d_logits, int ldd,
                                          float* d_gates, int ldg, float* d_cell, float* datt, float* dcov_tot, float* d_pre_b,
                                          float* d_ctx12, float* vec_acc, float* scal_acc, const float* proj_a, const float* proj_i,
                                          const float* enc_a, const float* enc_i, const float* coverage, const float* v1, const float* wc1,
                                          const float* v2, const float* wc2, float* d_proj_a, float* d_proj_i, float* d_cov,
                                          const float* Wh_stack, float* d_h, int B, int Lt, int D, int H, int M, mmb_stream_t stream) {
  using namespace mmb;
  MMB_REQUIRE(probs && out_w && gates && cell_in && cell_out && Wcat_ctx && alpha && beta && ctx12 && pb && hw && vb1 && vb2 && Wb13 &&
                  d_logits && d_gates && d_cell && datt && dcov_tot && d_pre_b && d_ctx12 && vec_acc && scal_acc && proj_a && proj_i &&
                  enc_a && enc_i && coverage && v1 && wc1 && v2 && wc2 && d_proj_a && d_proj_i && d_cov && Wh_stack && d_h,
              MMB_ERR_INVALID, "mmb_decoder_step_fused_bwd: null pointer");
  MMB_REQUIRE((!target || g_nll) && (!g_cov || (att && cov_out)), MMB_ERR_INVALID, "mmb_decoder_step_fused_bwd: loss-term pointers");
  MMB_REQUIRE(B > 0 && Lt > 0 && D > 0 && D <= 256 && H > 0 && M > 0 && ldd >= M && ldg >= 4 * H + 4 * D && H <= NT, MMB_ERR_INVALID,
              "mmb_decoder_step_fused_bwd: B=%d Lt=%d D=%d H=%d M=%d ldd=%d ldg=%d", B, Lt, D, H, M, ldd, ldg);
  const int CL = (long long)B * 4 * 2 <= 160 ? 8 : 4;
  const int chunk = (Lt + CL - 1) / CL;
  HeadArgs a{probs, d_probs, target, g_nll, g_cov, out_w, gates, cell_in, cell_out, d_h_out, d_cell_out, Wcat_ctx, d_att_cov, d_cov_out,
             alpha, beta, ctx12, pb, hw, vb1, vb2, att, cov_out, Wb13, d_logits, d_gates, d_cell, datt, dcov_tot, d_pre_b, d_ctx12,
             vec_acc, scal_acc, B, Lt, D, H, M, ldd, ldg, chunk,
             1, proj_a, proj_i, enc_a, enc_i, coverage, v1, wc1, v2, wc2, d_proj_a, d_proj_i, d_cov, Wh_stack, d_h, 0};
  size_t smem = head_smem_bytes(D, H, M, CL, chunk, true);
  MMB_REQUIRE(smem <= 200 * 1024, MMB_ERR_UNSUPPORTED, "mmb_decoder_step_fused_bwd: %zu B of shared memory (Lt=%d)", smem, Lt);
  {
    // the row stage (see the kernel): two buffers of chunk x D floats behind two mbarriers; the column-partial reduction then runs in two
    // passes over half the buffer.  MMB_DEC_STAGE=0 turns it off (read once per process, as in launch_fused).
    static const char* stage_env = getenv("MMB_DEC_STAGE");
    const size_t base_floats = (head_smem_bytes(D, H, M, CL, chunk, true, NW / 2) - 64) / 4;
    const size_t stage_floats = 4 + 2 * (((size_t)chunk * D + 3) & ~(size_t)3);
    const bool aligned = ((reinterpret_cast<uintptr_t>(proj_a) | reinterpret_cast<uintptr_t>(proj_i) | reinterpret_cast<uintptr_t>(enc_a) |
                           reinterpret_cast<uintptr_t>(enc_i) | reinterpret_cast<uintptr_t>(d_proj_a) |
                           reinterpret_cast<uintptr_t>(d_proj_i)) & 15) == 0;
    if ((D & 3) == 0 && aligned && (base_floats + stage_floats) * 4 + 64 <= 227 * 1024 && !(stage_env && atoi(stage_env) == 0)) {
      a.stage_off = (int)base_floats;
      smem = (base_floats + stage_floats) * 4 + 64;
    }
  }
  if (smem > g_head_smem_set) {
    MMB_CUDA(cudaFuncSetAttribute(dec_bwd_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    g_head_smem_set = smem;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(B * CL));
  cfg.blockDim = dim3(NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MMB_CUDA(cudaLaunchKernelEx(&cfg, dec_bwd_head_kernel, a));
  return check_launch("dec_bwd_head_kernel (whole step)");
}
