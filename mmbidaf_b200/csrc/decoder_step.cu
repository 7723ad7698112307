// Multimodal-attention decoder step (layers/attention.py:145-186), forward and backward, as chunk-parallel
// kernels around small batched GEMMs.
//
// A decode step touches, per video, two (Lt x 2H) tensors twice (projected encodings for the energies,
// encodings for the contexts) plus a handful of (2H x H), (2H x 2H), (4H x (2H+E+H)) and (M x H) mat-vecs.
// With one CTA per video the step is latency bound (B = 32 CTAs on 148 SMs, long serial loops), so:
//   * every mat-vec becomes a (B x K) x (K x N) GEMM over the whole batch -- plain library GEMMs issued by the
//     caller (functional.py) between the kernels below;
//   * the per-(video, sentence) sweeps run on a (chunks x B) grid; the un-masked soft-max over the text axis
//     (attention.py:148,154, quirk Q2) is computed "flash" style: chunk-local max / sum / weighted context,
//     merged by a tiny combine kernel.
// Forward:  attn_partial -> attn_combine -> [GEMM W_beta] -> attn_finish -> [GEMM LSTM] -> cell_pointwise
//           -> [GEMM out] -> out_softmax
// Backward: out_softmax_bwd -> [GEMM] -> cell_bwd -> [GEMM] -> attn_finish_bwd -> [GEMM] -> sweep1 -> sweep2
//           -> attn_reduce -> [GEMM]
// W1.enc / W3.enc are step invariant and arrive pre-multiplied (proj_a / proj_i).
#include <type_traits>
#include "common.cuh"

namespace mmb {
namespace {

constexpr int NT = 256;
constexpr int NW = NT / 32;
// flush-to-zero MUFU forms (no denormal guard instructions around them)
__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_ftz(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
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

// ----------------------------------------------------------------------------------------------------------
// forward 1: energies of one chunk of sentences + chunk-local soft-max partials
//   e_k[t] = v_k . tanh(proj_k[t] + hw_k + cov[t] wc_k) + v_k bias                       (attention.py:147,153)
//   p[b,k,t] = exp(e_k[t] - m_c),  stats[b,c,k] = (m_c, sum_t p),  ctxp[b,c,k,:] = sum_t p enc_k[t]
// ----------------------------------------------------------------------------------------------------------
// forward 2: merge the chunk partials -> contexts c1, c2 (2,B,D) and per-chunk scales (B,2,nch).  Run by the LAST chunk
// block of a video to finish (see last_block_of_video), so the step needs no separate launch for it.
__device__ __forceinline__ void combine_video(const float* stats, const float* ctxp,   /* other blocks' partials: no read-only path */
                                              float* ctx12, float* scale, int b, int B, int D, int nch) {
  const int tid = threadIdx.x;
  __shared__ float w[2][64];
  __shared__ float inv_l[2];
  if (tid < 2) {
    const int k = tid;
    float m = -INFINITY;
    for (int c = 0; c < nch; ++c) m = fmaxf(m, stats[((size_t)b * nch + c) * 4 + 2 * k]);
    float l = 0.f;
    for (int c = 0; c < nch; ++c) {
      const float wc = expf(stats[((size_t)b * nch + c) * 4 + 2 * k] - m);
      w[k][c] = wc;
      l = fmaf(wc, stats[((size_t)b * nch + c) * 4 + 2 * k + 1], l);
    }
    inv_l[k] = 1.f / l;
    for (int c = 0; c < nch; ++c) scale[((size_t)b * 2 + k) * nch + c] = w[k][c] / l;
  }
  __syncthreads();
  for (int i = tid; i < 2 * D; i += NT) {
    const int k = i / D, d = i - k * D;
    float s = 0.f;
    for (int c = 0; c < nch; ++c) s = fmaf(w[k][c], ctxp[(((size_t)b * nch + c) * 2 + k) * D + d], s);
    ctx12[((size_t)k * B + b) * D + d] = s * inv_l[k];
  }
}

// True in exactly one of the `nblk` blocks that call it for video b: the last one to arrive, after whose fence the global
// writes of all the others are visible.  `counter` (one int per video, zero on entry) is left at zero again.
__device__ __forceinline__ bool last_block_of_video(int* counter, int nblk) {
  __shared__ int last;
  __threadfence();                                   // this block's partials, device-wide
  __syncthreads();
  if (threadIdx.x == 0) {
    const int prev = atomicAdd(counter, 1);
    last = prev == nblk - 1;
    if (last) *counter = 0;
  }
  __syncthreads();
  const bool is_last = last != 0;
  if (is_last) __threadfence();
  return is_last;
}

struct PartialArgs {
  const float *proj_a, *proj_i, *enc_a, *enc_i, *hw, *cov;   // hw (B,4D): [W2 h+b | W4 h+b | ...]
  const float *v1, *wc1, *v2, *wc2, *v1b, *v2b;
  float *p, *stats, *ctxp;
  float *ctx12, *scale;      // written by the last chunk block of each video (combine_video)
  int* counters;             // (B) zero on entry, zero on exit
  int B, Lt, D, chunk, nch;
  int vec4;                  // 1: the weighted contexts read enc_a / enc_i rows as float4 (D % 4 == 0 and both 16-byte aligned)
};

__global__ void __launch_bounds__(NT) dec_attn_partial_kernel(const PartialArgs a) {
  const int D = a.D, Lt = a.Lt;
  const int c = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t0 = c * a.chunk, t1 = min(Lt, t0 + a.chunk), n = t1 - t0;
  extern __shared__ __align__(16) float smem[];
  float* part = smem;                    // [groups][2][D]  (16-byte aligned, float4 path)
  const bool vec4 = a.vec4 != 0;
  const int groups = vec4 ? NT / (D >> 2) : NT / D;
  float* vec = part + groups * 2 * D;    // [6][D]: v1 | wc1 | hw1 | v2 | wc2 | hw2
  float* red = vec + 6 * D;              // [32]
  float* e = red + 32;                   // [2][chunk]
  for (int i = tid; i < D; i += NT) {
    vec[i] = a.v1[i];
    vec[D + i] = a.wc1[i];
    vec[2 * D + i] = a.hw[(size_t)b * 4 * D + i];
    vec[3 * D + i] = a.v2[i];
    vec[4 * D + i] = a.wc2[i];
    vec[5 * D + i] = a.hw[(size_t)b * 4 * D + D + i];
  }
  __syncthreads();
  const float v1b = a.v1b[0], v2b = a.v2b[0];
  // Two sentences per warp iteration: all loads of both rows are in flight before the first tanh.  Written for the issue slots like
  // stage B of the one-kernel step (decoder_fused.cu): a lane's per-column constants live in registers for the whole chunk, pre-scaled
  // so that the pre-activation is the ex2 argument (tanh x = 1 - 2 / (1 + 2^(2 x log2 e))); columns past D carry v = 0, so nothing in
  // the body is predicated (the first version branched around every element and re-read six constants from shared memory per element).
  constexpr float K2 = 2.0f * 1.4426950408889634f;
  auto energies = [&](auto nj_tag) {
    constexpr int NJ = decltype(nj_tag)::value;
    float va[NJ], ha[NJ], wa[NJ], vi[NJ], hi[NJ], wi[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int d = lane + 32 * j;
      const bool in = d < D;
      const int dd = in ? d : 0;
      va[j] = in ? vec[dd] : 0.f;
      wa[j] = in ? vec[D + dd] * K2 : 0.f;
      ha[j] = in ? vec[2 * D + dd] * K2 : 0.f;
      vi[j] = in ? vec[3 * D + dd] : 0.f;
      wi[j] = in ? vec[4 * D + dd] * K2 : 0.f;
      hi[j] = in ? vec[5 * D + dd] * K2 : 0.f;
    }
    for (int i = warp * 2; i < n; i += NW * 2) {
      float s[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
      float pav[2][NJ], piv[2][NJ], cvs[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {          // loads first (memory-level parallelism)
        const int t = t0 + min(i + u, n - 1);
        const float* pa = a.proj_a + ((size_t)b * Lt + t) * D;
        const float* pi = a.proj_i + ((size_t)b * Lt + t) * D;
        cvs[u] = a.cov[(size_t)b * Lt + t];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int d = lane + 32 * j;
          pav[u][j] = d < D ? pa[d] : 0.f;
          piv[u][j] = d < D ? pi[d] : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float cv = cvs[u];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const float x1 = fmaf(cv, wa[j], fmaf(pav[u][j], K2, ha[j]));
          const float x2 = fmaf(cv, wi[j], fmaf(piv[u][j], K2, hi[j]));
          const float r1 = rcp_ftz(1.0f + ex2_ftz(x1)), r2 = rcp_ftz(1.0f + ex2_ftz(x2));
          s[u][0] = fmaf(va[j], fmaf(-2.0f, r1, 1.0f), s[u][0]);
          s[u][1] = fmaf(vi[j], fmaf(-2.0f, r2, 1.0f), s[u][1]);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float x1 = warp_sum(s[u][0]), x2 = warp_sum(s[u][1]);
        if (lane == 0 && i + u < n) {
          e[i + u] = x1 + v1b;
          e[a.chunk + i + u] = x2 + v2b;
        }
      }
    }
  };
  if (D > 192 && D <= 224) energies(std::integral_constant<int, 7>{});      // the model's D = 2 H = 200
  else energies(std::integral_constant<int, 8>{});                          // any other D <= 256: zero padded
  __syncthreads();
  float m1 = -INFINITY, m2 = -INFINITY;
  for (int i = tid; i < n; i += NT) {
    m1 = fmaxf(m1, e[i]);
    m2 = fmaxf(m2, e[a.chunk + i]);
  }
  m1 = block_max(m1, red);
  m2 = block_max(m2, red);
  float l1 = 0.f, l2 = 0.f;
  for (int i = tid; i < n; i += NT) {
    const float p1 = expf(e[i] - m1), p2 = expf(e[a.chunk + i] - m2);
    e[i] = p1;
    e[a.chunk + i] = p2;
    a.p[((size_t)b * 2 + 0) * Lt + t0 + i] = p1;
    a.p[((size_t)b * 2 + 1) * Lt + t0 + i] = p2;
    l1 += p1;
    l2 += p2;
  }
  l1 = block_sum(l1, red);
  l2 = block_sum(l2, red);
  if (tid == 0) {
    float* st = a.stats + ((size_t)b * a.nch + c) * 4;
    st[0] = m1; st[1] = l1; st[2] = m2; st[3] = l2;
  }
  __syncthreads();
  const float* ea = a.enc_a + ((size_t)b * Lt + t0) * D;
  const float* ei = a.enc_i + ((size_t)b * Lt + t0) * D;
  if (vec4) {
    const int dv4 = D >> 2;
    const int g = tid / dv4, c4 = tid - g * dv4;
    if (g < groups) {
      float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
#pragma unroll 4
      for (int i = g; i < n; i += groups) {
        const float w1 = e[i], w2 = e[a.chunk + i];
        const float4 x1 = *reinterpret_cast<const float4*>(ea + (size_t)i * D + c4 * 4);
        const float4 x2 = *reinterpret_cast<const float4*>(ei + (size_t)i * D + c4 * 4);
        s1.x = fmaf(w1, x1.x, s1.x); s1.y = fmaf(w1, x1.y, s1.y); s1.z = fmaf(w1, x1.z, s1.z); s1.w = fmaf(w1, x1.w, s1.w);
        s2.x = fmaf(w2, x2.x, s2.x); s2.y = fmaf(w2, x2.y, s2.y); s2.z = fmaf(w2, x2.z, s2.z); s2.w = fmaf(w2, x2.w, s2.w);
      }
      *reinterpret_cast<float4*>(part + (g * 2 + 0) * D + c4 * 4) = s1;
      *reinterpret_cast<float4*>(part + (g * 2 + 1) * D + c4 * 4) = s2;
    }
  } else {
    const int g = tid / D, d = tid - g * D;
    if (g < groups) {
      float s1 = 0.f, s2 = 0.f;
      for (int i = g; i < n; i += groups) {
        s1 = fmaf(e[i], ea[(size_t)i * D + d], s1);
        s2 = fmaf(e[a.chunk + i], ei[(size_t)i * D + d], s2);
      }
      part[(g * 2 + 0) * D + d] = s1;
      part[(g * 2 + 1) * D + d] = s2;
    }
  }
  __syncthreads();
  for (int d = tid; d < 2 * D; d += NT) {
    const int k = d / D, dd = d - k * D;
    float s = 0.f;
    for (int g = 0; g < groups; ++g) s += part[(g * 2 + k) * D + dd];
    a.ctxp[(((size_t)b * a.nch + c) * 2 + k) * D + dd] = s;
  }
  if (last_block_of_video(a.counters + b, a.nch)) combine_video(a.stats, a.ctxp, a.ctx12, a.scale, b, a.B, D, a.nch);
}

// forward 3: modality soft-max, attended context, attention / coverage outputs         (attention.py:161-177)
struct FinishArgs {
  const float *pb, *hw, *ctx12, *scale, *cov, *sent, *h;      // pb (2,B,D) = W_beta_{1,3} c_k + bias
  const float *vb1, *vb2, *vb1b, *vb2b;
  float *p_alpha;                                             // in: p (B,2,Lt)  out: alpha
  float *xcat, *att_cov, *cov_out, *beta;                     // xcat (B, D+E+H) = [ctx | sent | h]
  float* cov_loss;                                            // (B) sum_t min(att_cov, coverage') (models.py:177) or null
  int B, Lt, D, E, H, chunk, nch;
};

__global__ void __launch_bounds__(NT) dec_attn_finish_kernel(const FinishArgs a) {
  const int D = a.D, Lt = a.Lt, b = blockIdx.x, tid = threadIdx.x;
  __shared__ float red[32];
  float eb1 = 0.f, eb2 = 0.f;
  for (int d = tid; d < D; d += NT) {
    eb1 = fmaf(a.vb1[d], tanh_fast(a.pb[(size_t)b * D + d] + a.hw[(size_t)b * 4 * D + 2 * D + d]), eb1);
    eb2 = fmaf(a.vb2[d], tanh_fast(a.pb[((size_t)a.B + b) * D + d] + a.hw[(size_t)b * 4 * D + 3 * D + d]), eb2);
  }
  eb1 = block_sum(eb1, red) + a.vb1b[0];
  eb2 = block_sum(eb2, red) + a.vb2b[0];
  const float mb = fmaxf(eb1, eb2);
  const float x1 = expf(eb1 - mb), x2 = expf(eb2 - mb);
  const float beta1 = x1 / (x1 + x2), beta2 = x2 / (x1 + x2);
  const int K = D + a.E + a.H;
  float* xr = a.xcat + (size_t)b * K;
  for (int d = tid; d < D; d += NT) xr[d] = a.ctx12[(size_t)b * D + d] * beta1 + a.ctx12[((size_t)a.B + b) * D + d] * beta2;
  for (int i = tid; i < a.E; i += NT) xr[D + i] = a.sent[(size_t)b * a.E + i];
  for (int i = tid; i < a.H; i += NT) xr[D + a.E + i] = a.h[(size_t)b * a.H + i];
  float* p1 = a.p_alpha + ((size_t)b * 2 + 0) * Lt;
  float* p2 = a.p_alpha + ((size_t)b * 2 + 1) * Lt;
  const float* sc = a.scale + (size_t)b * 2 * a.nch;
  float closs = 0.f;
  for (int t = tid; t < Lt; t += NT) {
    const int c = t / a.chunk;
    const float a1 = p1[t] * sc[c], a2 = p2[t] * sc[a.nch + c];
    p1[t] = a1;
    p2[t] = a2;
    const float att = a1 * beta1 + a2 * beta2;                 // bmm([a1 a2], beta), attention.py:167
    const float cnew = a.cov[(size_t)b * Lt + t] + att;
    a.att_cov[(size_t)b * Lt + t] = att;
    a.cov_out[(size_t)b * Lt + t] = cnew;
    closs += fminf(att, cnew);
  }
  if (a.cov_loss) {
    closs = block_sum(closs, red);
    if (tid == 0) a.cov_loss[b] = closs;
  }
  if (tid == 0) {
    a.beta[b * 2 + 0] = beta1;
    a.beta[b * 2 + 1] = beta2;
  }
}

// forward 4: LSTM cell point-wise part on pre-activations (B,4H) = [ctx|sent|h] [W_ih|W_hh]^T + b   (attention.py:181)
__global__ void __launch_bounds__(NT) dec_cell_pointwise_kernel(float* __restrict__ gates, const float* __restrict__ cell,
                                                                float* __restrict__ h_out, float* __restrict__ cell_out, int B,
                                                                int H) {
  const int i = blockIdx.x * NT + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, j = i - b * H;
  float* g = gates + (size_t)b * 4 * H;
  const float gi = gate_act(g[j], 1.f), gf = gate_act(g[H + j], 1.f), gg = tanh_fast(g[2 * H + j]), go = gate_act(g[3 * H + j], 1.f);
  const float c = fmaf(gf, cell[i], gi * gg);
  cell_out[i] = c;
  h_out[i] = go * tanh_fast(c);
  g[j] = gi; g[H + j] = gf; g[2 * H + j] = gg; g[3 * H + j] = go;        // activated gates, kept for the backward pass
}

// forward 5: masked soft-max over the M outputs (attention.py:184) + first-max arg-max; logits -> probs in place
__global__ void __launch_bounds__(NT) dec_out_softmax_kernel(float* __restrict__ logits, const uint8_t* __restrict__ mask,
                                                             long long* __restrict__ argmax, const long long* __restrict__ tgt,
                                                             float* __restrict__ nll, int M) {
  __shared__ float red[32];
  __shared__ int redi[NW];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* lg = logits + (size_t)b * M;
  const uint8_t* mk = mask + (size_t)b * M;
  float mx = -INFINITY;
  for (int m = tid; m < M; m += NT) mx = fmaxf(mx, mk[m] ? lg[m] : kNegFill);
  mx = block_max(mx, red);
  float sum = 0.f;
  for (int m = tid; m < M; m += NT) sum += expf((mk[m] ? lg[m] : kNegFill) - mx);
  sum = block_sum(sum, red);
  const float inv = 1.f / sum;
  float best = -INFINITY;
  int best_i = M;
  for (int m = tid; m < M; m += NT) {
    const float p = expf((mk[m] ? lg[m] : kNegFill) - mx) * inv;
    lg[m] = p;
    if (p > best) { best = p; best_i = m; }
    if (tgt && m == (int)tgt[b]) nll[b] = -logf(p + 1e-12f);     // models.py:168-170
  }
  if (argmax) {                                                 // first maximal index, as torch.max(dim) documents
    const float gbest = block_max(best, red);
    int cand = best == gbest ? best_i : M;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
    __syncthreads();
    if (lane == 0) redi[warp] = cand;
    __syncthreads();
    if (tid == 0) {
      int r = M;
      for (int w = 0; w < NW; ++w) r = min(r, redi[w]);
      argmax[b] = r;
    }
  }
}

// ----------------------------------------------------------------------------------------------------------
// backward
// ----------------------------------------------------------------------------------------------------------
// 1: masked soft-max backward: dlogit = p (dp - sum p dp); masked entries have p = 0
__global__ void __launch_bounds__(NT) dec_out_softmax_bwd_kernel(const float* __restrict__ probs, const float* __restrict__ d_probs,
                                                                 const long long* __restrict__ tgt, const float* __restrict__ g_nll,
                                                                 float* __restrict__ d_logits, int ldd, int M) {
  __shared__ float red[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  // optional sparse part: d(-log(p_tgt + eps)) = -g / (p_tgt + eps) at the target column only
  const int tg = tgt ? (int)tgt[b] : -1;
  const float dp_t = tgt ? -g_nll[b] / (probs[(size_t)b * M + tg] + 1e-12f) : 0.f;
  float dot = 0.f;
  if (d_probs)
    for (int m = tid; m < M; m += NT) dot = fmaf(probs[(size_t)b * M + m], d_probs[(size_t)b * M + m], dot);
  dot = block_sum(dot, red);
  if (tgt) dot = fmaf(probs[(size_t)b * M + tg], dp_t, dot);
  for (int m = tid; m < M; m += NT) {
    const float dp = (d_probs ? d_probs[(size_t)b * M + m] : 0.f) + (m == tg ? dp_t : 0.f);
    d_logits[(size_t)b * ldd + m] = probs[(size_t)b * M + m] * (dp - dot);
  }
  for (int m = M + tid; m < ldd; m += NT) d_logits[(size_t)b * ldd + m] = 0.f;   // row padding (keeps the next GEMM's K aligned)
}

// 2: LSTM cell backward (point-wise): activated gates -> d pre-activations (in place), d cell
__global__ void __launch_bounds__(NT) dec_cell_bwd_kernel(float* __restrict__ gates, const float* __restrict__ cell_in,
                                                          const float* __restrict__ cell_out, const float* __restrict__ d_h,
                                                          const float* __restrict__ d_h2, const float* __restrict__ d_cell_out,
                                                          float* __restrict__ d_gates, int ldg, float* __restrict__ d_cell, int B,
                                                          int H) {
  const int i = blockIdx.x * NT + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, j = i - b * H;
  const float* g = gates + (size_t)b * 4 * H;
  const float gi = g[j], gf = g[H + j], gg = g[2 * H + j], go = g[3 * H + j];
  const float tc = tanh_fast(cell_out[i]);
  const float dh = d_h[i] + (d_h2 ? d_h2[i] : 0.f);      // e.g. d logits out.weight + the next step's d h
  const float dc = fmaf(dh * go, 1.f - tc * tc, d_cell_out ? d_cell_out[i] : 0.f);
  float* o = d_gates + (size_t)b * ldg;
  o[j] = dc * gg * gi * (1.f - gi);
  o[H + j] = dc * cell_in[i] * gf * (1.f - gf);
  o[2 * H + j] = dc * gi * (1.f - gg * gg);
  o[3 * H + j] = dh * tc * go * (1.f - go);
  d_cell[i] = dc * gf;
}

// 3: modality soft-max + W_beta tanh backward.  d_ctx arrives as the first D columns of d xcat (row stride ldx).
struct FinishBwdArgs {
  const float *d_xcat, *d_att_cov, *d_cov_out, *alpha, *beta, *ctx12, *pb, *hw, *vb1, *vb2;
  float *datt, *d_pre_b, *d_ctx12, *vec_acc, *scal_acc;       // datt (B,Lt); d_pre_b, d_ctx12 (2,B,D)
  const float *att, *cov_out, *g_cov;                         // fused coverage loss (g_cov (B) or null)
  float* dcov_tot;                                            // (B,Lt) d coverage' incl. the loss term
  int B, Lt, D, ldx;
};

__global__ void __launch_bounds__(NT) dec_attn_finish_bwd_kernel(const FinishBwdArgs a) {
  const int D = a.D, Lt = a.Lt, b = blockIdx.x, tid = threadIdx.x;
  __shared__ float red[32];
  const float beta1 = a.beta[b * 2 + 0], beta2 = a.beta[b * 2 + 1];
  const float* dctx = a.d_xcat + (size_t)b * a.ldx;
  float db1 = 0.f, db2 = 0.f;
  for (int d = tid; d < D; d += NT) {
    const float g = dctx[d];
    db1 = fmaf(a.ctx12[(size_t)b * D + d], g, db1);
    db2 = fmaf(a.ctx12[((size_t)a.B + b) * D + d], g, db2);
  }
  const float gc = a.g_cov ? a.g_cov[b] : 0.f;
  for (int t = tid; t < Lt; t += NT) {
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
  db1 = block_sum(db1, red);
  db2 = block_sum(db2, red);
  const float mix = beta1 * db1 + beta2 * db2;
  const float deb1 = beta1 * (db1 - mix), deb2 = beta2 * (db2 - mix);
  for (int d = tid; d < D; d += NT) {
    const float t1 = tanh_fast(a.pb[(size_t)b * D + d] + a.hw[(size_t)b * 4 * D + 2 * D + d]);
    const float t2 = tanh_fast(a.pb[((size_t)a.B + b) * D + d] + a.hw[(size_t)b * 4 * D + 3 * D + d]);
    a.d_pre_b[(size_t)b * D + d] = deb1 * a.vb1[d] * (1.f - t1 * t1);
    a.d_pre_b[((size_t)a.B + b) * D + d] = deb2 * a.vb2[d] * (1.f - t2 * t2);
    a.vec_acc[((size_t)b * 6 + 4) * D + d] += deb1 * t1;        // d v_beta_1 weight
    a.vec_acc[((size_t)b * 6 + 5) * D + d] += deb2 * t2;
    a.d_ctx12[(size_t)b * D + d] = beta1 * dctx[d];             // the W_beta^T d_pre part is added by a GEMM
    a.d_ctx12[((size_t)a.B + b) * D + d] = beta2 * dctx[d];
  }
  if (tid == 0) {
    a.scal_acc[b * 4 + 2] += deb1;
    a.scal_acc[b * 4 + 3] += deb2;
  }
}

// 4: sweep 1 over the encodings of a chunk: d alpha_k[t] = beta_k datt[t] + d c_k . enc_k[t]
struct SweepArgs {
  const float *proj_a, *proj_i, *enc_a, *enc_i, *hw, *cov, *alpha, *beta, *datt, *d_ctx12, *d_cov_out;
  const float *v1, *wc1, *v2, *wc2;
  float *d_alpha, *spart;                                     // (B,2,Lt), (B,nch,2)
  float *d_proj_a, *d_proj_i, *d_cov, *colp, *separt;         // colp (B,nch,2,3,D), separt (B,nch,2)
  const float* d_pre_b;                                       // reduce_video
  float *d_hw4, *vec_acc, *scal_acc;
  int* counters;                                              // (B) zero on entry, zero on exit
  int ldhw;                                                   // row stride of d_hw4 (>= 4D)
  int B, Lt, D, chunk, nch;
};

__global__ void __launch_bounds__(NT) dec_attn_sweep1_kernel(const SweepArgs a) {
  const int D = a.D, Lt = a.Lt;
  const int c = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t0 = c * a.chunk, t1 = min(Lt, t0 + a.chunk), n = t1 - t0;
  extern __shared__ __align__(16) float smem[];
  float* dc = smem;                      // [2][D]
  float* red = dc + 2 * D;               // [32]
  for (int i = tid; i < 2 * D; i += NT) dc[i] = a.d_ctx12[((size_t)(i / D) * a.B + b) * D + (i % D)];
  __syncthreads();
  const float beta1 = a.beta[b * 2 + 0], beta2 = a.beta[b * 2 + 1];
  float s1 = 0.f, s2 = 0.f;
  for (int i = warp * 2; i < n; i += NW * 2) {
    float d1[2] = {0.f, 0.f}, d2[2] = {0.f, 0.f};
    constexpr int MAXJ = 8;              // D <= 256
    float eav[2][MAXJ], eiv[2][MAXJ];
#pragma unroll
    for (int u = 0; u < 2; ++u) {        // loads first (memory-level parallelism)
      const float* ea = a.enc_a + ((size_t)b * Lt + t0 + min(i + u, n - 1)) * D;
      const float* ei = a.enc_i + ((size_t)b * Lt + t0 + min(i + u, n - 1)) * D;
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        const int d = lane + 32 * j;
        eav[u][j] = d < D ? ea[d] : 0.f;
        eiv[u][j] = d < D ? ei[d] : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        const int d = lane + 32 * j;
        if (d < D) {
          d1[u] = fmaf(dc[d], eav[u][j], d1[u]);
          d2[u] = fmaf(dc[D + d], eiv[u][j], d2[u]);
        }
      }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float x1 = warp_sum(d1[u]), x2 = warp_sum(d2[u]);
      if (lane == 0 && i + u < n) {
        const int t = t0 + i + u;
        const float g = a.datt[(size_t)b * Lt + t];
        const float da1 = x1 + beta1 * g, da2 = x2 + beta2 * g;
        a.d_alpha[((size_t)b * 2 + 0) * Lt + t] = da1;
        a.d_alpha[((size_t)b * 2 + 1) * Lt + t] = da2;
        s1 = fmaf(a.alpha[((size_t)b * 2 + 0) * Lt + t], da1, s1);
        s2 = fmaf(a.alpha[((size_t)b * 2 + 1) * Lt + t], da2, s2);
      }
    }
  }
  s1 = block_sum(s1, red);
  s2 = block_sum(s2, red);
  if (tid == 0) {
    a.spart[((size_t)b * a.nch + c) * 2 + 0] = s1;
    a.spart[((size_t)b * a.nch + c) * 2 + 1] = s2;
  }
}

// 6: reduce the chunk partials: d (W h + b) rows for the final GEMM, parameter-gradient accumulators.  Run by the LAST
// sweep-2 block of a video to finish.
__device__ __forceinline__ void reduce_video(int b, const float* colp, const float* separt,   /* other blocks' partials */
                                                             const float* __restrict__ d_pre_b, float* __restrict__ d_hw4,
                                                             float* __restrict__ vec_acc, float* __restrict__ scal_acc, int B,
                                                             int D, int nch, int ldhw) {
  const int tid = threadIdx.x;
  for (int i = tid; i < 2 * D; i += NT) {
    const int m = i / D, d = i - m * D;
    float x = 0.f, y = 0.f, z = 0.f;
    constexpr int CB = 8;                                                  // chunk partials in flight (the sum order is unchanged)
    for (int c0 = 0; c0 < nch; c0 += CB) {
      float xs[CB], ys[CB], zs[CB];
#pragma unroll
      for (int u = 0; u < CB; ++u) {
        const float* q = colp + ((((size_t)b * nch + min(c0 + u, nch - 1)) * 2 + m) * 3) * D;
        xs[u] = q[d];
        ys[u] = q[D + d];
        zs[u] = q[2 * D + d];
      }
#pragma unroll
      for (int u = 0; u < CB; ++u)
        if (c0 + u < nch) {
          x += xs[u];
          y += ys[u];
          z += zs[u];
        }
    }
    d_hw4[(size_t)b * ldhw + m * D + d] = x;                              // d (W2 h) | d (W4 h)
    d_hw4[(size_t)b * ldhw + (2 + m) * D + d] = d_pre_b[((size_t)m * B + b) * D + d];    // d (W_beta_2 h) | d (W_beta_4 h)
    vec_acc[((size_t)b * 6 + m) * D + d] += y;                            // d Wc weight
    vec_acc[((size_t)b * 6 + 2 + m) * D + d] += z;                        // d v weight
  }
  if (tid < 64) {                                                          // warps 0, 1: lane pairs (chunk, k) loaded in parallel
    const int warp = tid >> 5, lane = tid & 31;
    float v0 = lane < nch ? separt[((size_t)b * nch + lane) * 2 + warp] : 0.f;
    float v1 = lane + 32 < nch ? separt[((size_t)b * nch + lane + 32) * 2 + warp] : 0.f;
    float s = 0.f;
    for (int c = 0; c < nch; ++c) s += __shfl_sync(0xffffffffu, c < 32 ? v0 : v1, c & 31);   // fixed order
    if (lane == 0) scal_acc[b * 4 + warp] += s;                           // d v bias (identically 0 up to rounding)
  }
}


// 5: sweep 2 over the projections of a chunk: soft-max backward, tanh backward, d proj (+=), d cov, column partials
__global__ void __launch_bounds__(NT) dec_attn_sweep2_kernel(const SweepArgs a) {
  const int D = a.D, Lt = a.Lt;
  const int c = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t0 = c * a.chunk, t1 = min(Lt, t0 + a.chunk), n = t1 - t0;
  extern __shared__ __align__(16) float smem[];
  float* vec = smem;                     // [6][D]: v1 | wc1 | hw1 | v2 | wc2 | hw2
  float* red = vec + 6 * D;              // [32]
  float* part = red + 32;                // [NW][3][D]
  float* rowacc = part + NW * 3 * D;     // [chunk] d cov accumulation
  for (int i = tid; i < D; i += NT) {
    vec[i] = a.v1[i];
    vec[D + i] = a.wc1[i];
    vec[2 * D + i] = a.hw[(size_t)b * 4 * D + i];
    vec[3 * D + i] = a.v2[i];
    vec[4 * D + i] = a.wc2[i];
    vec[5 * D + i] = a.hw[(size_t)b * 4 * D + D + i];
  }
  __shared__ float stot[2];
  if (tid < 64) {                        // warps 0, 1: the chunk partials of sum_t alpha d alpha, loaded in parallel, summed in order
    float v0 = lane < a.nch ? a.spart[((size_t)b * a.nch + lane) * 2 + warp] : 0.f;
    float v1 = lane + 32 < a.nch ? a.spart[((size_t)b * a.nch + lane + 32) * 2 + warp] : 0.f;
    float s = 0.f;
    for (int cc = 0; cc < a.nch; ++cc) s += __shfl_sync(0xffffffffu, cc < 32 ? v0 : v1, cc & 31);
    if (lane == 0) stot[warp] = s;
  }
  for (int i = tid; i < n; i += NT) rowacc[i] = a.d_cov_out ? a.d_cov_out[(size_t)b * Lt + t0 + i] : 0.f;
  __syncthreads();
  constexpr int MAXJ = 8;                // D <= 256
  for (int m = 0; m < 2; ++m) {
    const float* proj = (m == 0 ? a.proj_a : a.proj_i) + ((size_t)b * Lt + t0) * D;
    float* dproj = (m == 0 ? a.d_proj_a : a.d_proj_i) + ((size_t)b * Lt + t0) * D;
    const float* vv = vec + 3 * m * D;
    const float* wc = vv + D;
    const float* hwm = vv + 2 * D;
    const float stm = stot[m];
    float c_dz[MAXJ], c_cov[MAXJ], c_v[MAXJ];
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) c_dz[j] = c_cov[j] = c_v[j] = 0.f;
    float se = 0.f;
    // two sentences per warp iteration: every load of both rows is in flight before the first tanh
    for (int i0 = warp * 2; i0 < n; i0 += NW * 2) {
      float cvs[2], dets[2], pv[2][MAXJ], dpv[2][MAXJ];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int i = min(i0 + u, n - 1), t = t0 + i;
        cvs[u] = a.cov[(size_t)b * Lt + t];
        dets[u] = a.alpha[((size_t)b * 2 + m) * Lt + t] * (a.d_alpha[((size_t)b * 2 + m) * Lt + t] - stm);
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) {
          const int d = lane + 32 * j;
          pv[u][j] = d < D ? proj[(size_t)i * D + d] : 0.f;
          dpv[u][j] = d < D ? dproj[(size_t)i * D + d] : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int i = i0 + u;
        if (i >= n) break;
        const float cv = cvs[u], det = dets[u];
        float row = 0.f;
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) {
          const int d = lane + 32 * j;
          if (d < D) {
            const float tz = tanh_fast((pv[u][j] + hwm[d]) + cv * wc[d]);
            const float dz = det * vv[d] * (1.f - tz * tz);
            dproj[(size_t)i * D + d] = dpv[u][j] + dz;
            c_dz[j] += dz;
            c_cov[j] = fmaf(dz, cv, c_cov[j]);
            c_v[j] = fmaf(det, tz, c_v[j]);
            row = fmaf(dz, wc[d], row);
          }
        }
        row = warp_sum(row);
        if (lane == 0) {
          rowacc[i] += row;
          se += det;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      const int d = lane + 32 * j;
      if (d < D) {
        part[(warp * 3 + 0) * D + d] = c_dz[j];
        part[(warp * 3 + 1) * D + d] = c_cov[j];
        part[(warp * 3 + 2) * D + d] = c_v[j];
      }
    }
    se = block_sum(se, red);                                    // (contains the __syncthreads that publishes `part`)
    if (tid == 0) a.separt[((size_t)b * a.nch + c) * 2 + m] = se;
    for (int i = tid; i < 3 * D; i += NT) {
      float x = 0.f;
      for (int w = 0; w < NW; ++w) x += part[w * 3 * D + i];
      a.colp[((((size_t)b * a.nch + c) * 2 + m) * 3) * D + i] = x;
    }
    __syncthreads();
  }
  for (int i = tid; i < n; i += NT) a.d_cov[(size_t)b * Lt + t0 + i] = rowacc[i];
  if (last_block_of_video(a.counters + b, a.nch))
    reduce_video(b, a.colp, a.separt, a.d_pre_b, a.d_hw4, a.vec_acc, a.scal_acc, a.B, D, a.nch, a.ldhw);
}

}  // namespace
}  // namespace mmb

using namespace mmb;

extern "C" int mmb_decoder_chunks(int B, int Lt) {
  // as many (chunk, video) CTAs as fit in ONE wave at two CTAs per SM (sweep 2 needs 127 registers x 256 threads): 2 x 148
  // slots, rounded DOWN -- 320 CTAs (10 chunks x 32 videos) ran as a full wave plus a 24-CTA tail that doubled the time;
  // at least 16 sentences per chunk, at most 64 chunks
  int nch = 296 / B;
  nch = nch < 1 ? 1 : nch > 64 ? 64 : nch;
  const int max_by_len = (Lt + 15) / 16;
  return nch < max_by_len ? nch : (max_by_len < 1 ? 1 : max_by_len);
}

extern "C" int mmb_decoder_attn_fwd(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                    const float* hw, const float* coverage, const float* v1, const float* wc1,
                                    const float* v2, const float* wc2, const float* v1b, const float* v2b, float* p,
                                    float* stats, float* ctxp, float* ctx12, float* scale, int* counters, int B, int Lt, int D,
                                    int nch, mmb_stream_t stream) {
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && hw && coverage && v1 && wc1 && v2 && wc2 && v1b && v2b && p && stats &&
                  ctxp && ctx12 && scale && counters,
              MMB_ERR_INVALID, "mmb_decoder_attn_fwd: null pointer");
  MMB_REQUIRE(B > 0 && Lt > 0 && D > 0 && nch > 0 && nch <= 64, MMB_ERR_INVALID, "mmb_decoder_attn_fwd: bad sizes");
  MMB_REQUIRE(D <= NT, MMB_ERR_UNSUPPORTED, "mmb_decoder_attn_fwd: 2H=%d > %d", D, NT);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int chunk = (Lt + nch - 1) / nch;
  // with D % 4 == 0 every row start keeps the base pointer's alignment: float4 context loads when the bases are 16-byte aligned
  const int vec4 = D % 4 == 0 && ((reinterpret_cast<uintptr_t>(enc_a) | reinterpret_cast<uintptr_t>(enc_i)) & 15) == 0;
  PartialArgs a{proj_a, proj_i, enc_a, enc_i, hw, coverage, v1, wc1, v2, wc2, v1b, v2b, p, stats, ctxp, ctx12, scale, counters,
                B, Lt, D, chunk, nch, vec4};
  const int groups = vec4 ? NT / (D / 4) : NT / D;
  const size_t smem = sizeof(float) * ((size_t)groups * 2 * D + 6 * D + 32 + 2 * chunk);
  MMB_REQUIRE(smem <= 227 * 1024, MMB_ERR_UNSUPPORTED, "mmb_decoder_attn_fwd: chunk %d too large", chunk);
  MMB_CUDA(cudaFuncSetAttribute(dec_attn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dec_attn_partial_kernel<<<dim3(nch, B), NT, smem, st>>>(a);
  return check_launch("dec_attn_partial_kernel");
}

extern "C" int mmb_decoder_attn_finish(const float* pb, const float* hw, const float* ctx12, const float* scale,
                                       const float* coverage, const float* sent, const float* h, const float* vb1,
                                       const float* vb2, const float* vb1b, const float* vb2b, float* p_alpha, float* xcat,
                                       float* att_cov, float* cov_out, float* beta, float* cov_loss, int B, int Lt, int D,
                                       int E, int H, int nch, mmb_stream_t stream) {
  MMB_REQUIRE(pb && hw && ctx12 && scale && coverage && sent && h && vb1 && vb2 && vb1b && vb2b && p_alpha && xcat &&
                  att_cov && cov_out && beta,
              MMB_ERR_INVALID, "mmb_decoder_attn_finish: null pointer");
  const int chunk = (Lt + nch - 1) / nch;
  FinishArgs a{pb, hw, ctx12, scale, coverage, sent, h, vb1, vb2, vb1b, vb2b, p_alpha, xcat, att_cov, cov_out, beta,
               cov_loss, B, Lt, D, E, H, chunk, nch};
  dec_attn_finish_kernel<<<B, NT, 0, static_cast<cudaStream_t>(stream)>>>(a);
  return check_launch("dec_attn_finish_kernel");
}

extern "C" int mmb_decoder_cell_fwd(float* gates, const float* cell, float* h_out, float* cell_out, int B, int H,
                                    mmb_stream_t stream) {
  MMB_REQUIRE(gates && cell && h_out && cell_out && B > 0 && H > 0, MMB_ERR_INVALID, "mmb_decoder_cell_fwd: bad arguments");
  dec_cell_pointwise_kernel<<<(B * H + NT - 1) / NT, NT, 0, static_cast<cudaStream_t>(stream)>>>(gates, cell, h_out, cell_out, B, H);
  return check_launch("dec_cell_pointwise_kernel");
}

extern "C" int mmb_decoder_out_softmax(float* logits, const uint8_t* mask, long long* argmax, const long long* target,
                                       float* nll, int B, int M, mmb_stream_t stream) {
  MMB_REQUIRE(logits && mask && B > 0 && M > 0 && (!target || nll), MMB_ERR_INVALID, "mmb_decoder_out_softmax: bad arguments");
  dec_out_softmax_kernel<<<B, NT, 0, static_cast<cudaStream_t>(stream)>>>(logits, mask, argmax, target, nll, M);
  return check_launch("dec_out_softmax_kernel");
}

extern "C" int mmb_decoder_out_softmax_bwd(const float* probs, const float* d_probs, const long long* target,
                                           const float* g_nll, float* d_logits, int ldd, int B, int M, mmb_stream_t stream) {
  MMB_REQUIRE(probs && d_logits && B > 0 && M > 0 && ldd >= M && (!target || g_nll), MMB_ERR_INVALID,
              "mmb_decoder_out_softmax_bwd: bad arguments");
  dec_out_softmax_bwd_kernel<<<B, NT, 0, static_cast<cudaStream_t>(stream)>>>(probs, d_probs, target, g_nll, d_logits, ldd, M);
  return check_launch("dec_out_softmax_bwd_kernel");
}

extern "C" int mmb_decoder_cell_bwd(float* gates, const float* cell_in, const float* cell_out, const float* d_h,
                                    const float* d_h2, const float* d_cell_out, float* d_gates, int ldg, float* d_cell, int B,
                                    int H, mmb_stream_t stream) {
  MMB_REQUIRE(gates && cell_in && cell_out && d_h && d_gates && d_cell && B > 0 && H > 0 && ldg >= 4 * H, MMB_ERR_INVALID,
              "mmb_decoder_cell_bwd: bad arguments");
  dec_cell_bwd_kernel<<<(B * H + NT - 1) / NT, NT, 0, static_cast<cudaStream_t>(stream)>>>(
      gates, cell_in, cell_out, d_h, d_h2, d_cell_out, d_gates, ldg, d_cell, B, H);
  return check_launch("dec_cell_bwd_kernel");
}

extern "C" int mmb_decoder_attn_finish_bwd(const float* d_xcat, int ldx, const float* d_att_cov, const float* d_cov_out,
                                           const float* alpha, const float* beta, const float* ctx12, const float* pb,
                                           const float* hw, const float* vb1, const float* vb2, float* datt, float* d_pre_b,
                                           float* d_ctx12, float* vec_acc, float* scal_acc, const float* att_cov,
                                           const float* cov_out, const float* g_cov, float* dcov_tot, int B, int Lt, int D,
                                           mmb_stream_t stream) {
  MMB_REQUIRE(d_xcat && alpha && beta && ctx12 && pb && hw && vb1 && vb2 && datt && d_pre_b && d_ctx12 && vec_acc &&
                  scal_acc && dcov_tot && (!g_cov || (att_cov && cov_out)),
              MMB_ERR_INVALID, "mmb_decoder_attn_finish_bwd: null pointer");
  FinishBwdArgs a{d_xcat, d_att_cov, d_cov_out, alpha, beta, ctx12, pb, hw, vb1, vb2, datt, d_pre_b, d_ctx12, vec_acc,
                  scal_acc, att_cov, cov_out, g_cov, dcov_tot, B, Lt, D, ldx};
  dec_attn_finish_bwd_kernel<<<B, NT, 0, static_cast<cudaStream_t>(stream)>>>(a);
  return check_launch("dec_attn_finish_bwd_kernel");
}

extern "C" int mmb_decoder_attn_bwd(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                    const float* hw, const float* coverage, const float* alpha, const float* beta,
                                    const float* datt, const float* d_ctx12, const float* d_cov_out, const float* d_pre_b,
                                    const float* v1, const float* wc1, const float* v2, const float* wc2, float* d_alpha,
                                    float* spart, float* d_proj_a, float* d_proj_i, float* d_cov, float* colp, float* separt,
                                    float* d_hw4, int ldhw, float* vec_acc, float* scal_acc, int* counters, int B, int Lt,
                                    int D, int nch, mmb_stream_t stream) {
  MMB_REQUIRE(proj_a && proj_i && enc_a && enc_i && hw && coverage && alpha && beta && datt && d_ctx12 && d_pre_b && v1 &&
                  wc1 && v2 && wc2 && d_alpha && spart && d_proj_a && d_proj_i && d_cov && colp && separt && d_hw4 &&
                  vec_acc && scal_acc && counters,
              MMB_ERR_INVALID, "mmb_decoder_attn_bwd: null pointer");
  MMB_REQUIRE(D <= 256 && nch > 0 && nch <= 64, MMB_ERR_UNSUPPORTED, "mmb_decoder_attn_bwd: 2H=%d > 256 or bad chunks", D);
  MMB_REQUIRE(ldhw >= 4 * D, MMB_ERR_INVALID, "mmb_decoder_attn_bwd: ldhw=%d < 4 * 2H", ldhw);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int chunk = (Lt + nch - 1) / nch;
  SweepArgs a{proj_a, proj_i, enc_a, enc_i, hw, coverage, alpha, beta, datt, d_ctx12, d_cov_out, v1, wc1, v2, wc2,
              d_alpha, spart, d_proj_a, d_proj_i, d_cov, colp, separt, d_pre_b, d_hw4, vec_acc, scal_acc, counters,
              ldhw, B, Lt, D, chunk, nch};
  {
    const size_t smem = sizeof(float) * (2 * (size_t)D + 32);
    dec_attn_sweep1_kernel<<<dim3(nch, B), NT, smem, st>>>(a);
    if (int rc = check_launch("dec_attn_sweep1_kernel")) return rc;
  }
  {
    const size_t smem = sizeof(float) * (6 * (size_t)D + 32 + (size_t)NW * 3 * D + chunk);
    MMB_REQUIRE(smem <= 227 * 1024, MMB_ERR_UNSUPPORTED, "mmb_decoder_attn_bwd: chunk %d too large", chunk);
    MMB_CUDA(cudaFuncSetAttribute(dec_attn_sweep2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dec_attn_sweep2_kernel<<<dim3(nch, B), NT, smem, st>>>(a);
    return check_launch("dec_attn_sweep2_kernel");
  }
}
