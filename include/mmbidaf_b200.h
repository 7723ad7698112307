/*
 * mmbidaf_b200 -- C ABI of the B200 (sm_100a) kernels behind the MMBiDAF hot path.
 *
 * The reference (amankhullar/MMBiDAF) is pure Python: it has no FFI.  The boundary a
 * maintainer would bind is therefore the set of torch calls made inside
 *   layers/attention.py::BiDAFAttention.forward            (attention.py:37-75)
 *   layers/attention.py::masked_softmax                    (attention.py:78-98)
 *   layers/attention.py::MultimodalAttentionDecoder.forward (attention.py:145-186)
 *   layers/encoding.py::RNNEncoder.forward                 (encoding.py:83-108)
 * Each entry point below names the reference lines it replaces.  INTEGRATION.md shows
 * the ctypes stub that binds them from the reference's own layers/*.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous, row-major memory unless it says
 *     "host"; floats are fp32; masks / keep-masks are one byte per element (0 or 1);
 *   - nothing here allocates, synchronises or keeps global mutable state: the caller
 *     owns outputs and workspaces and passes the CUDA stream to launch on;
 *   - every function returns 0 on success, a non-zero mmb_status otherwise, and leaves a
 *     message readable through mmb_last_error() (thread local);
 *   - unsupported shapes are an error (MMB_ERR_UNSUPPORTED); there is no CPU fallback.
 */
#ifndef MMBIDAF_B200_H_
#define MMBIDAF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MMB_API __attribute__((visibility("default")))
#else
#define MMB_API
#endif

typedef void* mmb_stream_t;          /* a cudaStream_t */

enum mmb_status {
  MMB_OK = 0,
  MMB_ERR_INVALID = 1,               /* null pointer / non-positive size */
  MMB_ERR_UNSUPPORTED = 2,           /* shape or precision this build has no kernel for */
  MMB_ERR_CUDA = 3                   /* a CUDA runtime call failed (message has the cudaError) */
};

enum mmb_precision {
  MMB_PREC_FP32 = 0,                 /* fp32 FFMA contractions: rel <= 1e-5 tier */
  MMB_PREC_BF16 = 1                  /* tcgen05 bf16 contractions, fp32 accumulate: rel <= 2e-2 tier */
};

MMB_API int mmb_version(void);
MMB_API const char* mmb_last_error(void);
/* 1 if the current device is sm_100 (B200); the python loader refuses anything else. */
MMB_API int mmb_device_supported(void);

/* --------------------------------------------------------------------------------------
 * BiDAF attention, forward.  Replaces attention.py:37-54 + :56-75 + two masked_softmax
 * calls (:43-44).  S is never written to memory.
 *   text (B,Lc,d)  modality (B,Lq,d)  text_mask (B,Lc)  modality_mask (B,Lq)
 *   w_text (d) = text_weight, w_modality (d) = modality_weight, w_cross (d) =
 *   text_modality_weight, bias (1)                              (attention.py:30-35)
 *   keep_text / keep_modality: optional (NULL in eval) dropout keep-masks (B,L,d) for the
 *   inputs of the similarity only (attention.py:66-67); keep_scale = 1/(1-p).
 * Outputs
 *   out (B,Lc,4d) = [c, a, c*a, c*b]                                    (attention.py:52)
 *   q2c (B,Lq,d) = s2^T c, lse_row (B,Lc), lse_col (B,Lq): log-sum-exp of the row / column
 *   soft-max -- saved for the backward pass; bm (B,Lc,d) = s1 q2c (the b of attention.py:50 before the
 *   product with c), optional (NULL in inference), also for the backward pass.  MMB_PREC_FP32: d % 4 == 0, d <= 256 (workspace may be NULL).
 *   MMB_PREC_BF16 (tcgen05 + TMEM + TMA): d % 8 == 0, d <= 200, workspace of mmb_bidaf_workspace_bytes().
  * On the bf16 tier q2c, lse_row and lse_col may be NULL (inference: only `out` is written).
 */
MMB_API int mmb_bidaf_fwd(const float* text, const float* modality, const uint8_t* text_mask, const uint8_t* modality_mask,
                  const float* w_text, const float* w_modality, const float* w_cross, const float* bias,
                  const uint8_t* keep_text, const uint8_t* keep_modality, float keep_scale,
                  float* out, float* q2c, float* bm, float* lse_row, float* lse_col, void* workspace,
                  int B, int Lc, int Lq, int d, int precision, mmb_stream_t stream);

/* Bytes of scratch `workspace` mmb_bidaf_fwd needs (0 for MMB_PREC_FP32).  The bf16 tier keeps bf16 copies of
 * its operands there in tensor-core order; dropout != 0 when keep_modality will be non-NULL. */
MMB_API size_t mmb_bidaf_workspace_bytes(int B, int Lc, int Lq, int d, int precision, int dropout);

/* BiDAF attention, backward: the gradient of attention.py:37-75 that the reference obtains from autograd
 * (loss.backward(), train.py:148).  S, both soft-maxes and dS are recomputed on chip from lse_row / lse_col;
 * nothing of size Lc x Lq is read or written.
 *   grad_out (B,Lc,4d); text, modality, masks, weights, keep masks, keep_scale: as given to mmb_bidaf_fwd;
 *   out, bm, q2c, lse_row, lse_col: as produced by mmb_bidaf_fwd; fwd_workspace: the workspace of that call,
 *   untouched since (MMB_PREC_BF16: it holds the bf16 operands; MMB_PREC_FP32: NULL);
 *   workspace: mmb_bidaf_bwd_workspace_bytes().  MMB_PREC_FP32: d % 4 == 0, d <= 208; MMB_PREC_BF16: d % 8 == 0, d <= 200.
 * Outputs (all overwritten): d_text (B,Lc,d), d_modality (B,Lq,d), d_w_text (d), d_w_modality (d), d_w_cross (d), d_bias (1).
 */
MMB_API int mmb_bidaf_bwd(const float* grad_out, const float* text, const float* modality,
                  const uint8_t* text_mask, const uint8_t* modality_mask, const float* w_text,
                  const float* w_modality, const float* w_cross, const float* bias, const uint8_t* keep_text,
                  const uint8_t* keep_modality, float keep_scale, const float* out, const float* bm, const float* q2c,
                  const float* lse_row, const float* lse_col, const void* fwd_workspace, void* workspace,
                  float* d_text, float* d_modality, float* d_w_text, float* d_w_modality, float* d_w_cross, float* d_bias,
                  int B, int Lc, int Lq, int d, int precision, mmb_stream_t stream);
MMB_API size_t mmb_bidaf_bwd_workspace_bytes(int B, int Lc, int Lq, int d, int precision);

/* --------------------------------------------------------------------------------------
 * Length-aware LSTM recurrence of one layer, 1 or 2 directions.  Replaces the nn.LSTM call of
 * encoding.py:96 together with the sort / pack / pad / unsort gathers of encoding.py:91-101.
 *   gates (B,L,ndir,4H): on entry x W_ih^T + b_ih + b_hh (gate order i,f,g,o; a plain GEMM done
 *     by the caller); with save != 0 it holds the ACTIVATED gates on exit (for the backward pass)
 *   w_hh (ndir,4H,H)   lengths (B) int32   order (B) int32 permutation, longest first, or NULL
 *   out (B,L,ndir*H): hidden states, exact zeros past each length (pad_packed_sequence)
 *   h_n, c_n (B,ndir,H): state after each sample's last valid step, in BATCH order
 *   cell (B,L,ndir,H): cell states, written when save != 0 (may be NULL otherwise).  H <= 104.
 */
MMB_API int mmb_bilstm_fwd(float* gates, const float* w_hh, const int32_t* lengths, const int32_t* order, float* out,
                           float* h_n, float* c_n, float* cell, int B, int L, int H, int ndir, int save,
                           mmb_stream_t stream);

/* Backward through time of the same layer.  `gates` (activated gates from the forward pass) is
 * overwritten with d(loss)/d(pre-activation) (zeros past each length); dout (B,L,ndir*H);
 * dh_n / dc_n (B,ndir,H) may be NULL.  dW_ih, dx, db and dW_hh are GEMMs over `gates` for the caller.
 */
MMB_API int mmb_bilstm_bwd(float* gates, const float* cell, const float* w_hh, const int32_t* lengths,
                           const int32_t* order, const float* dout, const float* dh_n, const float* dc_n, int B, int L,
                           int H, int ndir, mmb_stream_t stream);

/* Dropout on a recurrent layer's OUTPUT applied inside the recurrence kernels (layers/encoding.py:104 `F.dropout(x, drop_prob, training)`
 * after the nn.LSTM call, and nn.LSTM's own inter-layer dropout, encoding.py:77-81): the forward kernel writes y = keep ? out / keep_prob : 0
 * beside the un-dropped `out` (which the recurrence and the weight gradients need); the backward kernel takes d y.  The keep bit of
 * element i of (B, L, ndir H) is a counter-based hash of (i, *rng_key): no mask tensor, no separate launch.  mmb_dropout_mask writes the
 * same bits as bytes (tests: parity GIVEN the mask); mmb_rng_next draws n_keys fresh keys from a device-resident state (splitmix64), so a
 * CUDA-graph replay gets new masks without host involvement.  Not ATen's Philox stream (DESIGN.md section 1). */
MMB_API int mmb_bilstm_fwd_dropout(float* gates, const float* w_hh, const int32_t* lengths, const int32_t* order, float* out, float* y,
                                   float* h_n, float* c_n, float* cell, const unsigned long long* rng_key, float keep_prob, int B,
                                   int L, int H, int ndir, int save, mmb_stream_t stream);
MMB_API int mmb_bilstm_bwd_dropout(float* gates, const float* cell, const float* w_hh, const int32_t* lengths, const int32_t* order,
                                   const float* dy, const float* dh_n, const float* dc_n, const unsigned long long* rng_key,
                                   float keep_prob, int B, int L, int H, int ndir, mmb_stream_t stream);
MMB_API int mmb_dropout_mask(const unsigned long long* rng_key, float keep_prob, long long n, uint8_t* mask, mmb_stream_t stream);
MMB_API int mmb_rng_next(unsigned long long* state, unsigned long long* key_out, int n_keys, mmb_stream_t stream);
/* layers/encoding.py:26 `F.dropout(x, self.drop_prob, self.training)` on the embedding inputs: y[i] = keep(i) ? x[i] / keep_prob : 0 with
 * the same counter-based bits (one launch, no mask tensor; y may alias x; x, y 16-byte aligned, n < 2^32).  Its backward is the same call
 * on the gradient with the same key.  The BiDAF kernels (attention.py:66-67) take mmb_dropout_mask's bytes as keep_text / keep_modality. */
MMB_API int mmb_dropout_apply(const float* x, float* y, const unsigned long long* rng_key, float keep_prob, long long n,
                              mmb_stream_t stream);

/* --------------------------------------------------------------------------------------
 * Multimodal attention decoder, one step (replaces attention.py:145-186).
 *
 * The step is a chain of chunk-parallel kernels around small batched GEMMs that the caller issues with its
 * BLAS (they are plain (B x K) x (K x N) products over the whole batch):
 *   hw    (B,4*2H) = h [W2;W4;W_beta_2;W_beta_4]^T + [b2+bc1; b4+bc2; bb2; bb4]
 *   mmb_decoder_attn_fwd      energies + un-masked soft-max over the text axis + contexts c1,c2 (attention.py:147-156)
 *   pb    (2,B,2H) = c_k W_beta_{1,3}^T (+ bias, unless the caller adds it with hw's third / fourth block: same tanh)
 *   mmb_decoder_attn_finish   2-way modality soft-max, attended context, att_cov, coverage (attention.py:161-177);
 *                             also assembles xcat (B, 2H+E+H) = [ctx | sent_embed | h]
 *   gates (B,4H)   = xcat [W_ih | W_hh]^T + b_ih + b_hh
 *   mmb_decoder_cell_fwd      LSTM cell point-wise part (attention.py:181); gates become the activated gates
 *   logits (B,M)   = h' out.weight^T + out.bias
 *   mmb_decoder_out_softmax   masked soft-max (attention.py:184) in place + first-max arg-max; with `target` (B) it
 *                             also emits the per-video loss term nll = -log(p[target] + 1e-12)  (models.py:168-170)
 * mmb_decoder_attn_finish likewise emits cov_loss (B) = sum_t min(att_cov, coverage') (models.py:177) when non-NULL.
 * proj_a = W1(enc_a) + b1 and proj_i = W3(enc_i) + b3 are step invariant and computed once by the caller.
 * Vectors v1, wc1 (= Wc1.weight), v2, wc2, vb1 (= v_beta_1.weight), vb2 have 2H entries; *b are 1-element biases.
 * nch = mmb_decoder_chunks(B, Lt) is the number of text chunks (scratch sizes depend on it):
 *   p (B,2,Lt)  stats (B,nch,4)  ctxp (B,nch,2,2H)  ctx12 (2,B,2H)  scale (B,2,nch)
 */
MMB_API int mmb_decoder_chunks(int B, int Lt);
/*
 * The same step as ONE kernel (north_star item 3; csrc/decoder_fused.cu): a thread-block cluster per video splits the text axis and
 * the output neurons of the step's mat-vecs and exchanges the small vectors through distributed shared memory.  Takes the weights in
 * the TRANSPOSED layouts of ops.DecoderWeights (consecutive threads read consecutive output neurons): Wh4t (H,4D) = [W2; W4; W_beta_2;
 * W_beta_4]^T with bh4 (4D) = the biases that land in the same tanh, Wb13t (2,D,D) = [W_beta_1^T; W_beta_3^T], Wcatt (D+E+H, 4H) =
 * [lstm.weight_ih | lstm.weight_hh]^T with bcat = b_ih + b_hh, out_wt (H,M) = out.weight^T.
 * Writes the step's outputs and everything mmb_decoder_*_bwd wants saved: hw (B,4D), alpha (B,2,Lt), beta (B,2), ctx12 (2,B,D),
 * pb (2,B,D), xcat (B,D+E+H) = [c3 | sent | h], gates (B,4H) activated.  argmax, target / nll and cov_loss may be NULL.
 * When D is a multiple of 4 and proj / enc are 16-byte aligned, each CTA stages its rows of proj_a / proj_i (then enc_a / enc_i) in shared
 * memory by bulk copies issued at kernel start (two buffers of ceil(Lt / cluster) x D floats; skipped when they do not fit in 227 KB, and
 * with MMB_DEC_STAGE=0, read once per process): the results of reading the rows from L2 (bit for bit when D >= 86, where the backward's
 * mat-vecs split K the same way on both), with fewer L2 round trips.
 * mmb_decoder_step_fused_bwd stages enc then proj the same way and adds its d z rows into d_proj_a / d_proj_i with one bulk reduction
 * per modality (d_proj_* must then be 16-byte aligned too).  Rows need only 4-byte alignment: when enc_a / enc_i are not 16-byte aligned
 * (or D is not a multiple of 4) the weighted contexts read them one float at a time, in this kernel and in mmb_decoder_attn_fwd, which
 * splits the rows over the threads differently: the same values up to fp32 rounding, not bit for bit.
 */
MMB_API int mmb_decoder_step_fused_fwd(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                       const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                       const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                       const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                       const float* out_wt, const float* out_b, const float* sent, const float* h, const float* cell,
                                       const float* cov, const uint8_t* mask, const long long* target, float* probs, float* h_out,
                                       float* cell_out, float* att_cov, float* cov_out, long long* argmax, float* nll,
                                       float* cov_loss, float* hw, float* alpha, float* beta, float* ctx12, float* pb, float* xcat,
                                       float* gates, int B, int Lt, int D, int H, int E, int M, mmb_stream_t stream);
/*
 * Greedy summary roll-out: all S = max_dec_len decoder steps of evaluation mode in ONE launch.  Replaces the decode loop of
 * models.py:156-199 in eval mode (the `else` branches: each step's arg-max row of the text is the next input, models.py:184,193)
 * -- S calls of attention.py:145-186, S arg-maxes and gathers, the torch.stack of the distributions.  Same cluster kernel as
 * mmb_decoder_step_fused_fwd (same weight layouts, stages, reduction order and shape limits: the per-step values are bit for bit the
 * step kernel's); the state between the steps (h', the cell, the coverage, the arg-max) stays on chip.  Start state as
 * models.py:145-149: h0 (B,H) = the sum of the two modality encoders' h_n (models.py:143), zero cell, coverage and input row.
 *   emb_text (B,Lt,E)  the embedded text (the next inputs are its rows)     mask (B,M)
 *   probs (B,S,M)      every step's distribution, in the layout MMBiDAF.forward returns
 *   argmax (B,S)       every step's first maximal index
 *   target (B,T) with T >= S, or NULL; then loss_terms (S,2,B) = per step [nll | coverage term] (models.py:168-170, :177), else unused.
 * Nothing the backward pass would need is written.
 */
MMB_API int mmb_decoder_greedy_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                     const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                     const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                     const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                     const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                     const uint8_t* mask, const long long* target, float* probs, long long* argmax, float* loss_terms,
                                     int B, int Lt, int D, int H, int E, int M, int S, int T, mmb_stream_t stream);
/*
 * Beam summary roll-out: the decode loop of models.py:156-199 in eval mode with K hypotheses per video instead of one, all S steps
 * in ONE launch of the same cluster kernel (one cluster per video holds every slot); the beam alternative to evaluate.py:185-202's
 * greedy pick.  This is the project's own beam rule; it does not claim parity with the reference's evaluate.py::beam_search.
 *   Slots: K per video, each live, finished (its last token was the EOS row text_len[b] - 1) or empty.  Before step 0 slot 0 is live
 *   with score 0 and the greedy start state (h0, zero cell, coverage and input row), the others empty with score -inf.
 *   Step: a live slot runs the decoder step from its own state -- bit for bit what mmb_decoder_step_fused_fwd computes from it -- and
 *   offers (slot, m) for every m with p[m] > 0, scored score + logf(p[m]) in fp32; a finished slot offers one carry (slot, EOS) with
 *   its score and step probability 1; empty slots offer nothing.  The candidates rank by score descending, then step probability
 *   descending, then parent slot ascending, then sentence ascending; the first K become the new slots 0..K-1, the rest stay empty.
 *   No length normalisation.  With K = 1 this is the greedy roll-out.
 *   text_len (B) int32   tokens / parents / scores (B,S,K) int64 / int32 / fp32: each new slot's token, previous slot and score
 *                        (-1, -1, -inf for an empty slot)
 *   probs (B,S,K,M)      the distribution slot j's parent produced at step s (zero for carries and empty slots)
 *   best (B,S) int64     the tokens of slot 0's path after the last step;  path (B,S) int32: the slot of that path at every step
 * 1 <= K <= 8.  Shapes as mmb_decoder_greedy_fused; the per-slot state lives in shared memory, so a width whose state does not fit
 * beside the step's arrays returns MMB_ERR_UNSUPPORTED with the byte count.
 */
MMB_API int mmb_decoder_beam_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                   const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                   const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                   const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                   const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                   const uint8_t* mask, const int32_t* text_len, long long* tokens, int32_t* parents, float* scores,
                                   float* probs, long long* best, int32_t* path, int B, int Lt, int D, int H, int E, int M, int K,
                                   int S, mmb_stream_t stream);
/*
 * Constrained summary roll-outs: mmb_decoder_greedy_fused and mmb_decoder_beam_fused with two constraints on the pick, each in ONE
 * launch of the same cluster kernel.  This is the project's own rule; like the beam rule it claims no parity with the reference.
 *   Per video b let eos = text_len[b] - 1.  Each hypothesis keeps `kept`, the number of its picks so far with index < eos (repeats
 *   counted), and used[m], set when m < eos was picked earlier on its path.  Parameters: no_repeat (0 or 1), min_sentences (>= 0).
 *   avail = eos - (no_repeat ? kept : 0), the non-EOS sentences the hypothesis could still add.  Sentence m is ELIGIBLE when mask[b,m]
 *   is set and either m < eos and not (no_repeat and used[m]), or m == eos and (kept >= min_sentences or avail == 0).  Rows past eos
 *   are never eligible.
 *   Greedy: the pick is the first maximal p[m] over the eligible m; with none eligible (only when the mask hides rows below eos) the
 *   pick is eos.  The roll-out goes on after EOS with the same rule.
 *   Beam: a live slot offers (slot, m) for every eligible m with p[m] > 0; everything else is mmb_decoder_beam_fused's rule (scores,
 *   carries, ranking, empty slots).  A new slot inherits used and kept from its parent, then adds its own token.
 *   The distributions are not changed: probs are the model's masked soft-max, bit for bit the step kernel's, and scores use that p.
 *   no_repeat = 0, min_sentences = 0 is exactly the unconstrained rule; the constrained beam with K = 1 is the constrained greedy.
 *   So: with no_repeat no summary holds a sentence twice, and a summary holds at least min(min_sentences, S, eos) sentences.
 * Greedy: arguments of mmb_decoder_greedy_fused without target / loss_terms (the eval loss is the unconstrained roll-out's), plus
 * text_len (B) int32; M / cluster size <= 16384.  Beam: arguments of mmb_decoder_beam_fused; the eligible bits and kept count of every
 * slot add to its shared memory (MMB_ERR_UNSUPPORTED with the byte count when a width does not fit).
 */
MMB_API int mmb_decoder_greedy_constrained_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                                 const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                                 const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                                 const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt,
                                                 const float* bcat, const float* out_wt, const float* out_b, const float* emb_text,
                                                 const float* h0, const uint8_t* mask, const int32_t* text_len, float* probs,
                                                 long long* argmax, int B, int Lt, int D, int H, int E, int M, int S, int no_repeat,
                                                 int min_sentences, mmb_stream_t stream);
MMB_API int mmb_decoder_beam_constrained_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                               const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                               const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                               const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                               const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                               const uint8_t* mask, const int32_t* text_len, long long* tokens, int32_t* parents,
                                               float* scores, float* probs, long long* best, int32_t* path, int B, int Lt, int D, int H,
                                               int E, int M, int K, int S, int no_repeat, int min_sentences, mmb_stream_t stream);
/*
 * Stochastic beam summary roll-outs: K DISTINCT summaries per video, an exact sample without replacement from the model's tempered,
 * renormalised sequence distribution, in ONE launch of the beam's cluster kernel (Kool, van Hoof and Welling, "Stochastic Beams and
 * Where to Find Them", ICML 2019).  This is the project's own rule; no reference parity is claimed.  Per video b: eos = text_len[b] - 1,
 * K slots, S steps, temperature T, a 64-bit key on the device (*key, as mmb_decoder_sample_fused takes it).
 *   Slots: the beam's (token, parent, status live / finished / empty, score = the sum of logf(p) along the path), plus two fp32 values:
 *   phi, the path's log-probability under the sampling distribution, and key, its perturbed log-probability.  Before step 0 slot 0 is
 *   live with score = phi = 0, key = -logf(-logf(u)) (a Gumbel(0) draw, u as below with the counter B S K M + b) and the greedy start
 *   state; the others are empty with all three -inf.  (The root's key must be a draw, not 0: with the root fixed, the final keys are
 *   conditioned on their maximum and the inclusion probabilities below would be wrong; the sample itself does not depend on it.)
 *   Candidates of a live slot k: the beam's -- every m with p[m] > 0, or under no_repeat / min_sentences the eligible m with p[m] > 0
 *   (the constrained beam's rule); p is the step kernel's distribution, bit for bit.
 *   Sampling distribution, exact and independent of how the cluster splits M:
 *     1. l[m] = logf(p[m]) * (1 / T) in fp32;  mu = the max of l over the candidates.
 *     2. q[m] = floor(expf(l[m] - mu) 2^24), Q = the sum of q as a uint64 (exact in any order; the max candidate has q = 2^24).
 *     3. lam = mu + logf((float)Q * 2^-24); the child's phi' = phi_k + (l[m] - lam).
 *   Perturbation: u as the sampled rule's step 2 with the counter c = ((b S + s) K + k) M + m (uint32; K = 1 is the counter of
 *   mmb_decoder_sample_fused with N = 1); G = phi' + -logf(-logf(u)); Z_k = the max of G over slot k's candidates.
 *   Child key: G truncated to at most the parent's key, key' = (key_k - fmaxf(v, 0)) - log1pf(expf(-fabsf(v))) with
 *   v = (key_k - G) + log1mexp(G - Z_k), log1mexp(a) = a > -ln 2 ? logf(-expm1f(a)) : log1pf(-expf(a)) (all fp32).  The child with
 *   G = Z_k gets exactly key_k.
 *   A finished slot offers one carry (slot, eos) with its score, phi and key and step probability 1; empty slots offer nothing.
 *   Selection: key descending, then step probability descending, then parent ascending, then sentence ascending (the beam's order with
 *   key in place of score); the first K become the new slots, the rest stay empty.  A new slot's score is score_k + logf(p[m]), its
 *   phi phi', its key key' (a carry keeps all three).
 *   Threshold: kappa[b] = the largest key, over the steps, of the (K + 1)-th entry of that step's ranking (the best candidate the
 *   step prunes), -inf when no step ranks more than K.  A pruned candidate's subtree holds a sequence with exactly its key and none
 *   with a larger one, so kappa is the (K + 1)-th largest key of all sequences.
 * So the K final slots are distinct token rows; the inclusion probability of final slot i is 1 - exp(-exp(phi_i - kappa)), and
 * exp(phi_i) over it is an unbiased importance weight.
 * Arguments of mmb_decoder_beam_constrained_fused (text_len required; no_repeat = min_sentences = 0 is the unconstrained rule) plus key
 * and T.  Writes the beam's tokens / parents / scores (B,S,K) and probs (B,S,K,M), plus phi and keys (B,S,K) fp32, paths (B,K,S) int64
 * (every final slot's tokens, step order), path_slots (B,K,S) int32 (its slot at every step) and kappa (B) fp32.  An empty final slot's
 * path is eos at every step and its path_slots -1; its phi, key and score are -inf.  MMB_ERR_INVALID: K outside 1..8, S <= 0, T not
 * finite and > 0, or a constraint out of range; MMB_ERR_UNSUPPORTED: B S K M + B > 2^32 (the counters of a key), or the shared memory of
 * the width (with the byte count), as for the beam.
 */
MMB_API int mmb_decoder_beam_sample_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                          const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                          const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                          const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                          const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                          const uint8_t* mask, const int32_t* text_len, const unsigned long long* key, long long* tokens,
                                          int32_t* parents, float* scores, float* probs, float* phi, float* keys, long long* paths,
                                          int32_t* path_slots, float* kappa, int B, int Lt, int D, int H, int E, int M, int K, int S,
                                          float T, int no_repeat, int min_sentences, mmb_stream_t stream);
/*
 * Sampled summary roll-outs: N summaries per video, each the greedy roll-out (or the constrained one) with the pick DRAWN, all in ONE
 * launch of the same cluster kernel (one cluster per (video, sample); the encoder outputs are read per video, not replicated).  This
 * is the project's own rule.  Inputs: N in 1..64; temperature T finite and > 0; top_k 0 (off) or 1..8; a 64-bit key on the device
 * (*key, as the dropout entry points take it); no_repeat / min_sentences as above (either set: the constrained candidates).
 * Roll-out (b, n) runs exactly the greedy roll-out's stages; its distributions are the step kernel's masked soft-max, bit for bit.
 * Only the pick of step s changes:
 *   1. Candidates: every sentence 0..M-1; with a constraint set, the eligible sentences of the rule above; with top_k > 0, only the
 *      top_k of those ranked first by (p descending, m ascending).
 *   2. Uniform: c = ((b N + n) S + s) M + m as a uint32; u = ((hash32(c, key) >> 9) + 0.5f) 2^-23, exact in fp32 and in
 *      [2^-24, 1 - 2^-24].  hash32 is the mixing function of the dropout keep bits.
 *   3. Score: z = logf(p[m]) (1 / T) - logf(-logf(u)) in fp32 (Gumbel-max); p = 0 gives -inf, p > 0 a finite z.
 *   4. Pick: the candidate with the largest z, ties to the smaller m.  With no candidate (only under a constraint, when the mask hides
 *      the rows below eos) the pick is eos, as in the constrained greedy.  The roll-out goes on after EOS with the same rule.
 * So the pick is distributed as p^(1/T) over the candidates; top_k = 1 is the greedy pick (the constrained greedy pick under a
 * constraint) whatever the key and T; the same key and inputs give the same samples, bit for bit.
 * Arguments of mmb_decoder_greedy_constrained_fused (text_len may be null without a constraint) plus key, N, T, top_k.  Writes
 * probs (B,N,S,M) and tokens (B,N,S) int64.  MMB_ERR_INVALID: N, T, top_k or a constraint out of range; MMB_ERR_UNSUPPORTED:
 * B N S M > 2^32 (the counters of a key), or under a constraint M / cluster size > 16384.
 */
MMB_API int mmb_decoder_sample_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                     const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                     const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                     const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                     const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                     const uint8_t* mask, const int32_t* text_len, const unsigned long long* key, float* probs,
                                     long long* tokens, int B, int Lt, int D, int H, int E, int M, int S, int N, float T, int top_k,
                                     int no_repeat, int min_sentences, mmb_stream_t stream);
/*
 * Steps 1 to 4 of the sampled pick above for given rows, one CTA per row, with the roll-out kernel's score function: the reference
 * of the tests.  probs (R,M); eligible (R,M) uint8 or null (null: every sentence is a candidate; else the candidates are the rows'
 * nonzero entries); row r is sample r % N of video row_base[r], i.e. roll-out row_base[r] N + r % N, at step s of S.
 * picks (R) int64: the pick, or -1 for a row without a candidate.
 */
MMB_API int mmb_sample_pick(const float* probs, const uint8_t* eligible, const unsigned long long* key, const int32_t* row_base, int R,
                            int M, int S, int s, int N, float T, int top_k, long long* picks, mmb_stream_t stream);
/*
 * Nucleus (top-p) summary roll-outs: mmb_decoder_sample_fused with the draw limited to the smallest set of the likeliest candidates
 * that holds top_p of their mass, cut inside the same one-launch cluster kernel.  This is the project's own rule.  Per step of roll-out
 * (b, n), the candidates C are step 1 of the sampled rule above (every sentence or the eligible ones, cut to the first top_k in
 * (p descending, m ascending) order when top_k > 0).  Then, for top_p < 1:
 *   1. Each candidate has the integer mass q[m] = floor(p[m] 2^24), exact from the fp32 p; Q = sum of q over C.
 *   2. P = rint(top_p 2^24) from the fp32 top_p (round half to even).
 *   3. The NUCLEUS is the first n candidates in that order, n the smallest n >= 1 with 2^24 (sum of the first n q) >= P Q.  Integer
 *      sums do not depend on their order: the set is the same however the cluster splits the sentences, and a host recomputes it
 *      exactly from the probs the kernel writes.
 *   4. The draw is steps 2 to 4 of the sampled rule over the nucleus: the largest z = logf(p) (1 / T) - logf(-logf(u)), same counter
 *      and key, ties to the smaller m; no candidate: eos.
 * The nucleus is cut from the model's p, not from p^(1/T): the set comes from the model and T only shapes the draw inside it.  (This
 * differs from tempering first and cutting after, when T != 1.)  So P Q <= 2^24 q of the first candidate gives n = 1, and the pick is
 * the (constrained) greedy pick whatever T and the key; a small enough top_p always gets there.  top_p = 1 is no cut: the call is
 * mmb_decoder_sample_fused's, with its samples bit for bit (a cut at P = 2^24 would drop candidates whose q is 0).
 * Arguments of mmb_decoder_sample_fused plus top_p.  MMB_ERR_INVALID: top_p outside (0, 1], or any error of mmb_decoder_sample_fused;
 * MMB_ERR_UNSUPPORTED: M >= 65536 with top_p < 1 (P Q must fit 64 bits), a row of M floats that does not fit in shared memory beside
 * the step's arrays, or any reason of mmb_decoder_sample_fused.
 */
MMB_API int mmb_decoder_sample_nucleus_fused(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                             const float* Wh4t, const float* bh4, const float* v1, const float* wc1, const float* v2,
                                             const float* wc2, const float* v1b, const float* v2b, const float* Wb13t, const float* vb1,
                                             const float* vb2, const float* vb1b, const float* vb2b, const float* Wcatt, const float* bcat,
                                             const float* out_wt, const float* out_b, const float* emb_text, const float* h0,
                                             const uint8_t* mask, const int32_t* text_len, const unsigned long long* key, float* probs,
                                             long long* tokens, int B, int Lt, int D, int H, int E, int M, int S, int N, float T,
                                             int top_k, int no_repeat, int min_sentences, float top_p, mmb_stream_t stream);
/*
 * mmb_sample_pick with the nucleus rule above: the reference of the tests for mmb_decoder_sample_nucleus_fused.  top_p = 1 is
 * mmb_sample_pick.  MMB_ERR_INVALID: top_p outside (0, 1] or any error of mmb_sample_pick; MMB_ERR_UNSUPPORTED: M >= 65536 with
 * top_p < 1.
 */
MMB_API int mmb_sample_pick_nucleus(const float* probs, const uint8_t* eligible, const unsigned long long* key, const int32_t* row_base,
                                    int R, int M, int S, int s, int N, float T, int top_k, long long* picks, float top_p,
                                    mmb_stream_t stream);
/*
 * Greedy sentence selection (evaluate.py:185-202, decode.greedy_search) on the device.  Per video, in step order over argmax (B,S):
 * the EOS row text_len[b] - 1 ends the summary, an index past it is skipped, any other is kept (repeats too).
 *   sel (B,S) int32 = the kept indices, then -1;  count (B) int32 = how many were kept.
 */
MMB_API int mmb_greedy_select(const long long* argmax, const int32_t* text_len, int32_t* sel, int32_t* count, int B, int S,
                              mmb_stream_t stream);

MMB_API int mmb_decoder_attn_fwd(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                 const float* hw, const float* coverage, const float* v1, const float* wc1,
                                 const float* v2, const float* wc2, const float* v1b, const float* v2b, float* p,
                                 float* stats, float* ctxp, float* ctx12, float* scale, int* counters, int B, int Lt, int D,
                                 int nch, mmb_stream_t stream);
/* p_alpha: in = p from mmb_decoder_attn_fwd, out = the attention weights alpha (B,2,Lt). */
MMB_API int mmb_decoder_attn_finish(const float* pb, const float* hw, const float* ctx12, const float* scale,
                                    const float* coverage, const float* sent, const float* h, const float* vb1,
                                    const float* vb2, const float* vb1b, const float* vb2b, float* p_alpha, float* xcat,
                                    float* att_cov, float* cov_out, float* beta, float* cov_loss, int B, int Lt, int D,
                                    int E, int H, int nch, mmb_stream_t stream);
MMB_API int mmb_decoder_cell_fwd(float* gates, const float* cell, float* h_out, float* cell_out, int B, int H,
                                 mmb_stream_t stream);
MMB_API int mmb_decoder_out_softmax(float* logits, const uint8_t* mask, long long* argmax, const long long* target,
                                    float* nll, int B, int M, mmb_stream_t stream);

/* Backward of the step, same structure in reverse (GEMMs by the caller between the kernels):
 *   mmb_decoder_out_softmax_bwd   d_logits = p (d_probs - sum p d_probs)            [d_probs may be NULL = 0]
 *                                 d_logits has row stride ldd >= M; columns M..ldd-1 are written as zeros (so that the
 *                                 caller can keep the K of d_logits out.weight a multiple of 4 when M is odd)
 *   d_h'   = d_h_out + d_logits out.weight
 *   mmb_decoder_cell_bwd          activated gates -> d pre-activations d_gates (B,4H; row stride ldg), d_cell; the hidden-state
 *                                 gradient is d_h + d_h2 (d_h2 may be NULL)
 *   d_xcat = d_gates [W_ih | W_hh]                 (its first 2H columns are d ctx, row stride ldx)
 *   mmb_decoder_attn_finish_bwd   dcov_tot (B,Lt) = d_cov_out + d cov_loss, datt (B,Lt) = d_att_cov + d cov_loss + dcov_tot
 *                                 (g_cov (B) = gradient of the fused coverage-loss term; ties of min() split evenly),
 *                                 d_pre_b (2,B,2H) = d(W_beta tanh argument),
 *                                 d_ctx12 (2,B,2H) = beta_k d ctx   (the caller adds d_pre_b W_beta_{1,3})
 *   mmb_decoder_attn_bwd          (d_cov_out = dcov_tot) sweeps over the text chunks: d_alpha, soft-max / tanh backward, d_cov,
 *                                 d_proj_a / d_proj_i ACCUMULATED in place (+=), d_hw4 (B,4*2H; row stride ldhw) = d(hw)
 *   (with d_gates and d_hw4 side by side in one (B, 4H + 4*2H) buffer, d_h is ONE GEMM against [W_hh ; Wh4])
 *   d_h    = d_xcat[:, 2H+E:] + d_hw4 [W2;W4;W_beta_2;W_beta_4]
 * vec_acc (B,6,2H) += [dWc1, dWc2, dv1, dv2, dv_beta_1, dv_beta_2]; scal_acc (B,4) += their scalar biases.
 * Scratch: d_alpha (B,2,Lt)  spart (B,nch,2)  colp (B,nch,2,3,2H)  separt (B,nch,2).
 * counters (B) int32 of mmb_decoder_attn_fwd / _bwd: zero before the first call, left at zero by every call (the last chunk
 * block of a video to finish merges that video's chunk partials, so neither function needs a second launch for it).
 */
/* The head of a backward step as ONE cluster kernel (csrc/decoder_fused.cu): mmb_decoder_out_softmax_bwd, d h = d_logits out.weight,
 * mmb_decoder_cell_bwd, d c3 = d_gates W_ih[:, :D], mmb_decoder_attn_finish_bwd and d c_k += W_beta_k^T d_pre_k -- same arguments and
 * results as those calls and the three library GEMMs between them (out_w (M,H), Wcat_ctx (4H,D), Wb13 (2,D,D) row-major).  The text
 * sweeps (mmb_decoder_attn_bwd) and the final d h GEMM follow it unchanged. */
MMB_API int mmb_decoder_bwd_head(const float* probs, const float* d_probs, const long long* target, const float* g_nll,
                                 const float* g_cov, const float* out_w, const float* gates, const float* cell_in,
                                 const float* cell_out, const float* d_h_out, const float* d_cell_out, const float* Wcat_ctx,
                                 const float* d_att_cov, const float* d_cov_out, const float* alpha, const float* beta,
                                 const float* ctx12, const float* pb, const float* hw, const float* vb1, const float* vb2,
                                 const float* att, const float* cov_out, const float* Wb13, float* d_logits, int ldd, float* d_gates,
                                 int ldg, float* d_cell, float* datt, float* dcov_tot, float* d_pre_b, float* d_ctx12, float* vec_acc,
                                 float* scal_acc, int B, int Lt, int D, int H, int M, mmb_stream_t stream);
MMB_API int mmb_decoder_out_softmax_bwd(const float* probs, const float* d_probs, const long long* target,
                                        const float* g_nll, float* d_logits, int ldd, int B, int M, mmb_stream_t stream);
MMB_API int mmb_decoder_cell_bwd(float* gates, const float* cell_in, const float* cell_out, const float* d_h,
                                 const float* d_h2, const float* d_cell_out, float* d_gates, int ldg, float* d_cell,
                                 int B, int H, mmb_stream_t stream);
MMB_API int mmb_decoder_attn_finish_bwd(const float* d_xcat, int ldx, const float* d_att_cov, const float* d_cov_out,
                                        const float* alpha, const float* beta, const float* ctx12, const float* pb,
                                        const float* hw, const float* vb1, const float* vb2, float* datt, float* d_pre_b,
                                        float* d_ctx12, float* vec_acc, float* scal_acc, const float* att_cov,
                                        const float* cov_out, const float* g_cov, float* dcov_tot, int B, int Lt, int D,
                                        mmb_stream_t stream);
/* The whole backward step of layers/attention.py:145-186 as ONE cluster kernel: mmb_decoder_bwd_head, the two text sweeps of
 * mmb_decoder_attn_bwd and d h = [d_gates | d_hw4] Wh_stack (Wh_stack (4H + 4D, H) = [lstm.weight_hh; W2; W4; W_beta_2; W_beta_4]).
 * d_gates is a (B, ldg) buffer with ldg >= 4H + 4D: d_hw4 (B, 4D) is written beside d_gates.  d_proj_a / d_proj_i, vec_acc and
 * scal_acc are accumulated in place; d_cov (B, Lt) and d_h (B, H) are written. */
MMB_API int mmb_decoder_step_fused_bwd(const float* probs, const float* d_probs, const long long* target, const float* g_nll,
                                       const float* g_cov, const float* out_w, const float* gates, const float* cell_in,
                                       const float* cell_out, const float* d_h_out, const float* d_cell_out, const float* Wcat_ctx,
                                       const float* d_att_cov, const float* d_cov_out, const float* alpha, const float* beta,
                                       const float* ctx12, const float* pb, const float* hw, const float* vb1, const float* vb2,
                                       const float* att, const float* cov_out, const float* Wb13, float* d_logits, int ldd,
                                       float* d_gates, int ldg, float* d_cell, float* datt, float* dcov_tot, float* d_pre_b,
                                       float* d_ctx12, float* vec_acc, float* scal_acc, const float* proj_a, const float* proj_i,
                                       const float* enc_a, const float* enc_i, const float* coverage, const float* v1, const float* wc1,
                                       const float* v2, const float* wc2, float* d_proj_a, float* d_proj_i, float* d_cov,
                                       const float* Wh_stack, float* d_h, int B, int Lt, int D, int H, int M, mmb_stream_t stream);

MMB_API int mmb_decoder_attn_bwd(const float* proj_a, const float* proj_i, const float* enc_a, const float* enc_i,
                                 const float* hw, const float* coverage, const float* alpha, const float* beta,
                                 const float* datt, const float* d_ctx12, const float* d_cov_out, const float* d_pre_b,
                                 const float* v1, const float* wc1, const float* v2, const float* wc2, float* d_alpha,
                                 float* spart, float* d_proj_a, float* d_proj_i, float* d_cov, float* colp, float* separt,
                                 float* d_hw4, int ldhw, float* vec_acc, float* scal_acc, int* counters, int B, int Lt,
                                 int D, int nch, mmb_stream_t stream);

/* --------------------------------------------------------------------------------------
 * masked_softmax over the last axis (attention.py:78-98): y = softmax(mask ? x : -1e30), or
 * log_softmax when log_mode != 0.  x, y (rows,n); mask (rows,n) bytes.  Backward returns
 * dx = mask * dsoftmax (the reference's d(mask*x)/dx = mask).
 */
MMB_API int mmb_masked_softmax_fwd(const float* x, const uint8_t* mask, float* y, long long rows, int n, int log_mode,
                                   mmb_stream_t stream);
MMB_API int mmb_masked_softmax_bwd(const float* y, const float* dy, const uint8_t* mask, float* dx, long long rows,
                                   int n, int log_mode, mmb_stream_t stream);

/* --------------------------------------------------------------------------------------
 * Highway layer (encoding.py:52-59), point-wise part.  pre (n,2H) = x [gates.k.weight; transforms.k.weight]^T + bias
 * is one GEMM by the caller; y = sigmoid(pre_g) * relu(pre_t) + (1 - sigmoid(pre_g)) * x.  Backward returns
 * d_pre (n,2H) (for dW = d_pre^T x, dx += d_pre W) and the direct path dx_direct = dy (1 - g).
 */
MMB_API int mmb_highway_fwd(const float* pre, const float* x, float* y, long long n, int H, mmb_stream_t stream);
MMB_API int mmb_highway_bwd(const float* pre, const float* x, const float* dy, float* d_pre, float* dx_direct,
                            long long n, int H, mmb_stream_t stream);

/* --------------------------------------------------------------------------------------
 * Mask / length plumbing on the device.  Replaces models.py:86-92 (`get_mask`: arange < len on the CPU, then .to(device),
 * models.py:126-129), models.py:119-123 (decoder mask: zeros + cast + cat on the CPU) and the scheduling use of the
 * descending-length order of encoding.py:91.  One launch from an int32 device vector of lengths:
 *   mask (B, L) uint8 = pos < len[b];  dec_mask (B, M) uint8 (optional, M >= L) = the same, zero beyond L;
 *   order (B) int32 (optional) = videos by descending length, ties in batch order (stable) -- used only to schedule the
 *   longest recurrences first; the hidden-state permutation of encoding.py:99-106 keeps coming from the host's torch.sort.
 */
MMB_API int mmb_length_plan(const int32_t* lengths, uint8_t* mask, uint8_t* dec_mask, int32_t* order, int B, int L, int M,
                            mmb_stream_t stream);

/* --------------------------------------------------------------------------------------
 * Column sums of a tall matrix: out (p) = sum over the n rows of a (n, p).  Every bias gradient of the training step is one
 * (the autograd gradient of nn.LSTM's b_ih / b_hh, encoding.py:76-81; of the highway biases, encoding.py:52-59; of the
 * decoder's hoisted projections W1 / W3, attention.py:152-157) -- in the reference an ATen reduction inside
 * loss.backward() (train.py:148).  Deterministic two-stage sum; partial: workspace of mmb_col_sum_blocks(n, p) * p floats.
 * Any p; the float4 kernel runs when p % 4 == 0 and a, partial are 16-byte aligned, a one-column-per-thread kernel otherwise.
 */
MMB_API int mmb_col_sum_blocks(long long n, int p);
MMB_API int mmb_col_sum(const float* a, float* partial, float* out, long long n, int p, mmb_stream_t stream);

/* train.py:148-155 hands ~110 per-parameter gradients to clip_grad_norm_ / the optimizer; here they are gathered into the flat gradient
 * buffer the fused update below runs over.  srcs / dst_offsets / sizes are HOST arrays of n_segs entries (device source pointers, element
 * offsets into dst that are multiples of 4, element counts); a null source zero-fills its segment; every segment is zero-padded up to a
 * multiple of 4 elements.  One launch per 120 segments; the pointers travel as kernel parameters. */
MMB_API int mmb_pack_segments(const float* const* srcs, const long long* dst_offsets, const long long* sizes, int n_segs, float* dst,
                              mmb_stream_t stream);

/* --------------------------------------------------------------------------------------
 * Parameter update of the training step (train.py:154-155 with the optimiser of train.py:110): clip_grad_norm_ followed by
 * one Adadelta step, fused into one pass over flat buffers of n floats (n % 4 == 0, 16-byte aligned):
 *   coef = min(max_norm / (grad_norm[0] + 1e-6), 1); grad *= coef (written back); g = grad + weight_decay * param;
 *   square_avg = rho square_avg + (1 - rho) g^2; delta = sqrt(acc_delta + eps) / sqrt(square_avg + eps) * g;
 *   acc_delta = rho acc_delta + (1 - rho) delta^2; param -= lr * delta.
 * grad_norm: device scalar, the 2-norm of grad (after the all-reduce when data parallel).
 */
MMB_API int mmb_adadelta_clip_step(float* param, float* grad, float* square_avg, float* acc_delta, const float* grad_norm,
                                   float max_norm, float lr, float rho, float eps, float weight_decay, long long n,
                                   mmb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MMBIDAF_B200_H_ */
