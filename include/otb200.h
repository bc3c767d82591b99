/*
 * libotb200 -- B200 (sm_100a) hot path for the OpenTransformer speech transformer, C ABI.
 *
 * The reference has no FFI / operator API: its boundary is the Python nn.Module surface
 * (SURVEY.md 8b).  Every entry point below therefore names the reference *module method* whose
 * per-call compute it replaces (file:line under the reference tree); the Python classes in
 * opentransformer_b200/ keep the reference's constructor kwargs / state_dict keys and call these
 * functions through ctypes (see INTEGRATION.md for the binding a maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated; "bf16" buffers are uint16 bfloat16, row-major
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream)
 *   - functions return 0 on success, non-zero on error; otb_last_error() gives the message
 *     (thread-local).  Nothing aborts; kernels are asynchronous on `stream`.
 *   - the library keeps no global mutable state besides the per-thread error string and lazily
 *     set function attributes, so one thread per GPU (nn.DataParallel, trainer.py:65) is safe.
 */
#ifndef OTB200_H_
#define OTB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OTB_VERSION 1

/* GEMM epilogues (otb_linear) */
enum {
    OTB_EPI_BIAS = 0,     /* y = x W^T + b                                   nn.Linear                          */
    OTB_EPI_RELU = 1,     /* relu(.)                                          ffn.py:16, conv.py:64              */
    OTB_EPI_GLU = 2,      /* W has 2N rows: (a + b_a) * sigmoid(g + b_g)      ffn.py:18 F.glu, conformer.py:45   */
    OTB_EPI_TABLE = 3,    /* (.) * alpha + table[row % period]                pos.py:56  x*sqrt(d)+PE            */
    OTB_EPI_RESID = 4,    /* resid + alpha * (.)                              encoder/conformer.py:53,72         */
    OTB_EPI_RESID_LN = 5, /* LayerNorm(resid + (.)) * gamma + beta            encoder/transformer.py:54-56,61-63 */
    OTB_EPI_SWISH = 6,    /* v * sigmoid(v)                                   ffn.py:20                          */
    OTB_EPI_GELU = 7,     /* F.gelu                                           ffn.py:17                          */
    OTB_EPI_TANH = 8      /* tanh                                             ffn.py:19                          */
};

const char* otb_last_error(void);
int otb_version(void);
int otb_num_sms(void);
/* Tiling policy of small GEMMs (M <= 512 rows, the decode step): 0 (default) = shortest launch -- narrow tiles, the
 * residual+LayerNorm row split over a 4-CTA cluster; 1 = least SM-time -- the widest tile on the fewest CTAs, for
 * servers that keep several utterance batches in flight on separate streams (+10-15 % aggregate throughput, +30 %
 * latency of a lone batch on B200).  Process-wide; set it before CUDA graphs are captured. */
int otb_set_tile_policy(int policy);
/* Profiling aid: buf (device, u64 [grid*8]) receives per-CTA clock64 phase stamps of the next GEMMs; NULL disables. */
int otb_debug_gemm_timing(unsigned long long* buf);
/* Profiling aid: 0 = normal, 1 = GEMM mainloop without TMA traffic, 2 = without MMAs (results are garbage). */
int otb_debug_gemm_mode(int mode);
/* Profiling aid: buf (device, u64 [>= 256]) receives clock64 stamps at every phase boundary of decode step `step`
 * of the next otb_decode_persistent launches (group 0, CTA 0); NULL disables. */
int otb_debug_decode_timing(unsigned long long* buf, int step);
/* Serving knob of otb_decode_persistent (no counterpart in the reference): how the 16 CTAs of a row group synchronise.
 * 1 = thread-block cluster of 16 + barrier.cluster (lowest latency; one cluster per GPC, i.e. at most 8 groups in flight),
 * 0 = plain CTAs + a release/acquire counter in L2 (all 148 SMs usable: best throughput with 3 batches in flight),
 * -1 = default (clusters when the device grants them, unless OTB_DG_CLUSTER=0).  Process-wide. */
int otb_set_decode_barrier(int kind);

/* Conv2dLayer output geometry, kernel 3, stride 2, padding (0,1)  (frontend/conv.py:10-11,27):
 * T1 = (T-3)/2+1, F1 = (F-1)/2+1, T2 = (T1-3)/2+1, F2 = (F1-1)/2+1.  The conv1 activation buffer is
 * NHWC bf16 [B, 2*(T2+1), 2*F2, C1]. */
int otb_conv_geometry(int T, int F, int* T1, int* F1, int* T2, int* F2);

/* Conv2dLayer.forward #1 (frontend/conv.py:50-76; C_in = 1): relu(conv2d(x, w) + b).
 * x f32 [B,T,F]; w f32 [C1,1,3,3]; bias f32 [C1]; out bf16 NHWC [B, 2*(T2+1), 2*F2, C1]. */
int otb_conv1_relu(const float* x, const float* w, const float* bias, void* out, int B, int T, int F, int C1,
                   void* stream);

/* Conv2dLayer.forward #2 + the transpose/reshape of ConvFrontEnd.forward (frontend/conv.py:63-64,145)
 * as a tcgen05 implicit GEMM.  in = conv1 buffer; w bf16 [C2, 9*C1] with k = (kh*3+kw)*C1 + c;
 * out bf16 [B*T2, F2*C2] with feature index f*C2 + c (the caller permutes output_layer.weight columns
 * from the reference's c*F2 + f order once at load time). */
int otb_conv2_relu(const void* in, const void* w, const float* bias, void* out, int B, int T, int F, int C1, int C2,
                   void* stream);

/* nn.Linear with a fused epilogue on tcgen05 tensor cores: out[M,N] = epi(a[M,K] w[N(,2N),K]^T + bias).
 * a, w bf16 (lda, ldw in elements, multiples of 8); out bf16 or f32 (out_f32); unused pointers NULL.
 * row_len/row_period: optional key-padding mask, rows with (m % row_period) >= row_len[m / row_period]
 * produce 0 before the residual is added (conformer.py:46,55 masked_fill).
 * Replaces attention.py:68,128-129,44; ffn.py:39-41; frontend/conv.py:146; decoder/transformer.py:181. */
int otb_linear(const void* a, int lda, const void* w, int ldw, const float* bias, void* out, int ldc, int M, int N,
               int K, int epilogue, int out_f32, const void* resid, int ldr, const float* gamma, const float* beta,
               float eps, float alpha, const float* table, int period, const int* row_len, int row_period,
               void* stream);

/* Training-mode residual connection with nn.Dropout on the sub-layer output (encoder/transformer.py:32-33,54,61;
 * decoder/transformer.py:36-38 `residual_dropout`): out bf16 = resid + alpha * keep * (a w^T + bias) / (1 - p), where
 * keep(seed, site, row, col) is a counter-based Bernoulli(1-p) mask (csrc/dropout.cuh) -- a pure function of the per-step
 * seed (*seed is read on the DEVICE at run time, so a captured CUDA graph draws a fresh mask per replay), the dropout
 * site id and the element, so the backward replays it instead of storing it. */
int otb_linear_dropout_resid(const void* a, int lda, const void* w, int ldw, const float* bias, void* out, int ldc, int M, int N,
                             int K, const void* resid, int ldr, float alpha, float p, const uint32_t* seed, uint32_t site,
                             void* stream);
/* Backward of that dropout: out = dy * keep / (1 - p) (bf16 [M,N]); mask (optional, u8 [M,N]) receives keep -- with dy / out
 * NULL this only exports the mask (parity tests replay it in the oracle). */
int otb_dropout_bwd(const void* dy, int lddy, void* out, int ldo, uint8_t* mask, int M, int N, float p, const uint32_t* seed,
                    uint32_t site, void* stream);

/* Fused masked multi-head attention, d_k = 64 (attention.py:80,34-41): for batch b, head h
 *   out[b*Tq+i, h*64:(h+1)*64] = softmax_j((q_i . k_j + bd) / 8, j < kv_len[b], causal: j <= i) V
 * q/k/v are row-major bf16 matrices; batch b owns rows [b*Tq, (b+1)*Tq) of q and [b*Tk, (b+1)*Tk) of k,v;
 * head h starts at column q_col0/k_col0/v_col0 + 64*h.  bd (optional, f32 [H,B,Tq,ldbd]) holds
 * relative-position scores, bias(i,j) = bd[h,b,i, j-i+Tq-1] (the gather of attention.py:196-215 done by
 * indexing).  resid (optional, bf16 [B*Tq, ldr]) is added to the output (the rel-pos attention of the
 * shipped Conformer has no output projection, SURVEY.md 8a quirks). */
int otb_attention(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                  void* out, int ldo, int B, int H, int Tq, int Tk, const int* kv_len, int causal, int q_col0,
                  int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, void* stream);
/* otb_attention with the head width as an argument: head_dim 64 or 96 (d_model 384 with 4 heads, the Conformer
 * recipe); head h starts at column *_col0 + head_dim*h and the scores are scaled by 1/sqrt(head_dim).  Any other
 * head_dim returns a non-zero status (otb_last_error) without launching.  otb_attention is head_dim = 64. */
int otb_attention_hd(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                     void* out, int ldo, int B, int H, int head_dim, int Tq, int Tk, const int* kv_len, int causal,
                     int q_col0, int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr,
                     void* stream);

/* ConformerConvolutionModule middle (module/conformer.py:48-52): depthwise Conv1d(k, pad (k-1)/2) over time +
 * eval-mode BatchNorm1d + swish.  x, out bf16 [B*T, d]; w f32 [k, d] and b f32 [d] carry the BatchNorm affine
 * folded in by the caller (w' = w * gamma/sqrt(var+eps), b' = (b - mean) * gamma/sqrt(var+eps) + beta). */
int otb_dwconv_swish(const void* x, const float* w, const float* b, void* out, int B, int T, int d, int k,
                     void* stream);

/* nn.LayerNorm (eps as given), optionally two in a row (encoder/conformer.py:87-89). g2/b2 may be NULL. */
int otb_layernorm(const void* x, int ldx, void* out, int ldo, int out_f32, const float* g1, const float* b1,
                  const float* g2, const float* b2, float eps, int M, int N, void* stream);

/* PositionalEncoding.forward stand-alone (module/pos.py:56): out bf16 = x * alpha + table[row % period];
 * x is f32 (x_f32 != 0) or bf16; table may be NULL (pure scale / dtype conversion). */
int otb_scale_add_table(const void* x, int ldx, int x_f32, void* out, int ldo, float alpha, const float* table,
                        int period, int M, int N, void* stream);

/* PositionalEncoding._embedding_from_positions (module/pos.py:30-42): out f32 [n_pos, d] for positions
 * first_pos .. first_pos + n_pos - 1 (negative allowed). */
int otb_sinusoid_table(float* out, int n_pos, int d, int first_pos, void* stream);

/* embedding + PositionalEncoding.forward (decoder/transformer.py:163,169; pos.py:56):
 * out[n] = emb[tok[n*tok_stride]] * sqrt(d) + table[pos], pos = step_ptr ? *step_ptr : n % period. */
int otb_embed_posenc(const int64_t* tok, int tok_stride, const void* emb, const float* table, void* out, int N,
                     int d, int period, const int* step_ptr, int vocab, void* stream);

/* F.log_softmax over the last dim, fp32 (decoder/transformer.py:206). */
int otb_log_softmax(const float* x, int ldx, float* out, int ldo, int rows, int V, void* stream);

/* Decode-step self-attention over a per-hypothesis KV cache (the cache API the reference left as a
 * stub, decoder/transformer.py:92-126,188-203): qkv bf16 [N,3d] of the newest token; kc/vc bf16
 * [Lmax,N,d]; anc i32 [2,N,Lmax]; *step_ptr = 0-based position; out bf16 [N,d]. */
int otb_decode_self_attn(const void* qkv, void* kc, void* vc, const int* anc, const int* step_ptr, void* out, int N,
                         int H, int Lmax, void* stream);
/* otb_decode_self_attn with the head width as an argument (64 or 96; d = H * head_dim).  otb_decode_self_attn is
 * head_dim = 64. */
int otb_decode_self_attn_hd(const void* qkv, void* kc, void* vc, const int* anc, const int* step_ptr, void* out, int N,
                            int H, int head_dim, int Lmax, void* stream);

/* LabelSmoothingLoss.forward (module/loss.py:21-48) fused: per-token KL(smoothed one-hot || softmax), PAD rows 0,
 * mean over non-PAD tokens.  logits f32 [rows, ldl]; targets i64 [rows]; tok_loss f32 [rows]; loss f32 [1];
 * n_valid i32 [1]; dlogits (optional, f32 [rows, ldd]) receives d loss / d logits. */
int otb_ls_ce(const float* logits, int ldl, const int64_t* targets, int rows, int V, float smoothing, int pad_id,
              float* tok_loss, float* loss, int32_t* n_valid, float* dlogits, int ldd, void* stream);

/* Device-resident beam-search state, N = B*beam hypotheses (all device pointers). */
typedef struct {
    int32_t* tok_hist;  /* [Lmax, N] */
    int32_t* par_hist;  /* [Lmax, N] */
    int64_t* last_tok;  /* [N]       */
    float* scores;      /* [N]       */
    uint8_t* flag;      /* [N]       */
    int32_t* anc;       /* [2, N, Lmax] */
    int32_t* ctrl;      /* [4] = {step, done, ended_now, -} */
    int32_t N, beam, Lmax;
} otb_beam_state;

/* recognize() initial state (recognize/speech2text.py:54-58). */
int otb_beam_init(const otb_beam_state* st, void* stream);
/* SpeechToTextRecognizer.decode_step after the decoder call (recognize/speech2text.py:102-153,156-192).
 * logp f32 [N, ldl] log-probs; lm_logp optional (shallow fusion, :102-105).  dbg_ktok i64 [N,beam] and
 * dbg_offs i32 [N] (optional) receive last_k_preds / offset_k_indices for parity traces. */
int otb_beam_step(const float* logp, int ldl, int V, const float* lm_logp, int ld_lm, float lm_weight,
                  const otb_beam_state* st, int64_t* dbg_ktok, int32_t* dbg_offs, void* stream);
/* Fused log_softmax (+ lm_weight * lm_logp) + per-row top-k (decoder/transformer.py:206 + speech2text.py:102-112):
 * logits f32 [rows, ldl] -> out_val f32 [rows,k] (log-prob values, descending), out_idx i32 [rows,k];
 * out_logp (optional, f32 [rows, ld_logp]) additionally receives the full log-prob rows. */
int otb_logsoftmax_topk(const float* logits, int ldl, int V, const float* lm_logp, int ld_lm, float lm_weight, int k,
                        int rows, float* out_val, int32_t* out_idx, float* out_logp, int ld_logp, void* stream);
/* otb_beam_step with the per-hypothesis top-k already computed by otb_logsoftmax_topk (k == beam). */
int otb_beam_step_topk(const float* topk_val, const int32_t* topk_idx, const otb_beam_state* st, int64_t* dbg_ktok,
                       int32_t* dbg_offs, void* stream);
/* Materialise preds i64 [N, ld] (column 0 = BOS) after `steps` steps from the back-pointers. */
int otb_beam_reconstruct(const otb_beam_state* st, int64_t* preds, int ld, int steps, void* stream);
/* Tail of recognize() (recognize/speech2text.py:70-91). out_preds i64 [B,nbest,Lmax], out_scores f32 [B,nbest]. */
int otb_beam_finalize(const otb_beam_state* st, float penalty, float lamda, int nbest, int64_t* out_preds,
                      float* out_scores, void* stream);

/* ---- Persistent decode loop --------------------------------------------------------------------------------
 * The whole loop of SpeechToTextRecognizer.recognize (recognize/speech2text.py:60-68: decode_step :95-153 ->
 * TransformerDecoder.inference, decoder/transformer.py:185-208) for ALL steps in one launch (csrc/decode_group.cu):
 * the hypotheses of up to 128 / beam utterances form one 128-row tcgen05 tile owned by a group of 16 co-operating CTAs
 * (projections split by output column / contraction slice, weights streamed from L2 by TMA, accumulators in TMEM,
 * activations exchanged through L2 behind a group-local barrier), search state on the device, no kernel launch or host
 * round trip inside the loop.  Post-norm GLU decoder, d_model 256, 4 heads, d_ff 2048, beam <= 16, T <= 256 memory
 * frames, max_steps <= st->Lmax <= 128, ceil(B / (128 / beam)) * 16 <= number of SMs (other configurations: per-step
 * calls above).  All pointers are device pointers; weights bf16 [N,K] row-major exactly as nn.Linear stores them. */
#define OTB_MEGA_MAX_LAYERS 8
typedef struct {
    const void *wqkv, *wo, *wq, *wo2, *w1, *w2;                 /* slf_attn.qvk_proj, .output_proj, src_attn.q_proj, .output_proj, feed_forward.w_1, .w_2 */
    const float *bqkv, *bo, *bq, *bo2, *b1, *b2;
    const float *g1, *be1, *g2, *be2, *g3, *be3;                /* norm1/2/3 weight, bias */
} otb_mega_layer;
typedef struct {
    int32_t n_layers, d_model, n_heads, d_ff, vocab;
    const void* emb;       /* embedding.weight bf16 [V, d] */
    const void* wout;      /* output_layer.weight bf16 [V, d] (== emb when tied, decoder/transformer.py:156-158) */
    const float* bout;     /* output_layer.bias [V] or NULL */
    const float* pe;       /* sinusoid table f32 [>= max_steps, d] (otb_sinusoid_table) */
    otb_mega_layer layers[OTB_MEGA_MAX_LAYERS];
    float ln_eps;
} otb_mega_model;
/* Scratch the launch needs (activations, partial sums, barrier counters, TMA descriptors), in bytes; -1 on bad arguments. */
long long otb_decode_persistent_workspace(int N, int n_layers, int Lmax, int B, int beam, int vocab);
/* kvx bf16 [n_layers, B*T, 2d]: src_attn.vk_proj(memory) per layer (K | V, attention.py:134), projected once per
 * utterance by otb_linear; mem_len i32 [B]; kc/vc bf16 [n_layers, st->Lmax, N, d] self-attention cache (scratch);
 * st: search state, initialised by otb_beam_init (ctrl zeroed); workspace: 256-byte aligned device scratch of at least
 * otb_decode_persistent_workspace() bytes.  On return tok_hist / par_hist hold max_steps steps (a group of utterances
 * that ended early is padded with EOS / identity parents, exactly what the reference's finished-hypothesis masking
 * produces), scores / flag / last_tok the final state, ctrl[0] the reference's executed step count (first step at which
 * every hypothesis of every utterance has ended, else max_steps).
 * dbg_logp (optional, f32 [max_steps, N, vocab]) receives every step's log-probs, dbg_scores (optional, f32
 * [max_steps, N]) every step's hypothesis scores -- parity traces. */
int otb_decode_persistent(const otb_mega_model* model, const void* kvx, const int32_t* mem_len, void* kc, void* vc,
                          const otb_beam_state* st, int B, int T, int max_steps, void* workspace, long long workspace_bytes,
                          float* dbg_logp, float* dbg_scores, void* stream);

/* ---- Training step (SpeechToText.forward + loss.backward() + clip + Adam, model/speech2text.py:39-64,
 * train/trainer.py:206-234).  The reference differentiates through torch autograd; the entry points below are the
 * hand-written backward of each forward op above.  bf16 activations / gradients, fp32 parameter gradients. */

/* otb_attention that also stores the per-row log-sum-exp (log2 units) [B,H,Tq] the backward needs. */
int otb_attention_lse(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                      void* out, int ldo, int B, int H, int Tq, int Tk, const int* kv_len, int causal, int q_col0,
                      int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, float* lse,
                      void* stream);
/* otb_attention_lse with the head width as an argument (64 or 96, as otb_attention_hd). */
int otb_attention_lse_hd(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                         void* out, int ldo, int B, int H, int head_dim, int Tq, int Tk, const int* kv_len, int causal,
                         int q_col0, int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, float* lse,
                         void* stream);
/* Backward of otb_attention, head_dim = 64 only (no bd / resid): dq, dk, dv written at column offsets d*_col0 + 64*h of their matrices
 * (e.g. the three thirds of one [M,3d] dqkv buffer).  dsum f32 [B,H,Tq] is scratch.  tcgen05, scores recomputed. */
int otb_attention_bwd(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                      const void* out, int ldo, const void* dout, int lddo, const float* lse, float* dsum, void* dq,
                      int lddq, int dq_col0, void* dk, int lddk, int dk_col0, void* dv, int lddv, int dv_col0, int B, int H,
                      int Tq, int Tk, const int* kv_len, int causal, int q_col0, int k_col0, int v_col0, void* stream);
/* nn.Linear weight gradient dW[N,K] (fp32) = dy[M,N]^T x[M,K] (bf16), tcgen05 with MN-major operands + split-K.
 * (The input gradient dx = dy W is otb_linear with the transposed weight.)  accumulate != 0: dW += ... (gradient
 * accumulation straight into the optimizer's flat gradient buffer, the way autograd accumulates into .grad). */
int otb_linear_wgrad(const void* dy, int lddy, const void* x, int ldx, float* dw, int lddw, int M, int N, int K, int accumulate,
                     void* stream);
/* nn.Linear bias gradient: out[n] (+)= sum_m x[m,n]. */
int otb_colsum(const void* x, int ldx, float* out, int M, int N, int accumulate, void* stream);
/* nn.LayerNorm backward (N <= 256): dz, dgamma (+)=, dbeta (+)= from dy and the pre-norm input z. */
int otb_layernorm_bwd(const void* dy, int lddy, const void* z, int ldz, const float* gamma, void* dz, int lddz,
                      float* dgamma, float* dbeta, float eps, int M, int N, int accumulate, void* stream);
/* F.glu (ffn.py:18) un-fused for training: u = [a | g] bf16 [M,2F] -> h [M,F]; and its backward. */
int otb_glu_fwd(const void* u, void* h, int M, int F, void* stream);
int otb_glu_bwd(const void* dh, const void* u, void* du, int M, int F, void* stream);
/* ReLU backward through the output (frontend/conv.py:64). */
int otb_relu_bwd(const void* dy, const void* y, void* dx, long long n, void* stream);
/* nn.Embedding backward: dE[tok[n]] += scale * dx[n]  (fp32 atomics). */
int otb_embed_bwd(const int64_t* tok, const void* dx, float* dE, int N, int d, int vocab, float scale, void* stream);
/* otb_ls_ce that also writes d(mean loss)/dlogits as bf16 [rows, ldd] (zero-padded columns) for the backward GEMMs. */
int otb_ls_ce_train(const float* logits, int ldl, const int64_t* targets, int rows, int V, float smoothing, int pad_id,
                    float* tok_loss, float* loss, int32_t* n_valid, void* dlogits_bf16, int ldd, void* stream);
/* out (+)= sum g^2 over a flat fp32 buffer (global gradient norm, trainer.py:221). */
int otb_sumsq(const float* g, long long n, float* out, int zero_first, void* stream);
/* clip_grad_norm_(max_norm) + torch.optim.Adam step on flat fp32 buffers; a non-finite norm skips the update
 * (trainer.py:229-230).  `sumsq` is the device scalar written by otb_sumsq; `step` is the 1-based update count. */
int otb_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* sumsq, float max_norm, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int step, void* stream);

/* otb_adam_step with the step counters and the LR schedule on the DEVICE (no host sync, CUDA-graph friendly):
 * counters i32 [3] = {optimizer steps, scheduler global_step, skipped steps}; when sqrt(*sumsq) is finite both counts
 * advance and lr = factor * model_size^-0.5 * min(s^-0.5, s * warmup^-1.5) (TransformerScheduler, train/scheduler.py:137-138;
 * warmup_steps <= 0: lr = base_lr), else only `skipped` advances and nothing is updated -- the reference skips
 * scheduler.step() and optimizer.step() together (trainer.py:229-233).  hyper f32 [4] receives {lr, 1-b1^t, 1-b2^t, applied}. */
int otb_adam_step_sched(float* p, const float* g, float* m, float* v, long long n, const float* sumsq, float max_norm,
                        float base_lr, float model_size, float warmup_steps, float factor, float beta1, float beta2, float eps,
                        float weight_decay, int32_t* counters, float* hyper, void* stream);

/* Log-mel filterbank features on the device (data/audio.py:117-120: ta.compliance.kaldi.fbank with Kaldi defaults, dither 0):
 * wave f32 [B, ld_wave] (zero padded), n_samples i32 [B]; window f32 [frame_len] (povey); bank f32 [F, 256] triangular mel
 * weights over the first 256 bins of the 512-point spectrum and bank_range i32 [F, 2] their non-zero [lo, hi) ranges (built
 * by opentransformer_b200/features.py); out f32 [B, Tmax, F], frames >= 1 + (n - frame_len) / frame_shift are zero. */
int otb_fbank(const float* wave, int ld_wave, const int32_t* n_samples, int B, const float* window, const float* bank,
              const int32_t* bank_range, float* out, int Tmax, int F, int frame_len, int frame_shift, float preemph, void* stream);
/* `normalization` (data/audio.py:22-24): (x - mean) / std over all valid elements of each utterance (unbiased std), in place;
 * or, with gmean / gstd f32 [F], the global CMVN of audio.py:131-132.  x f32 [B, Tmax, F], n_frames i32 [B]. */
int otb_utt_cmvn(float* x, int B, int Tmax, int F, const int32_t* n_frames, const float* gmean, const float* gstd, void* stream);

/* Joint-CTC loss of SpeechToText.forward (model/speech2text.py:60-72 -> CTCAssistor.compute_loss, model/ctc.py:48-52):
 * nn.CTCLoss(blank, reduction 'mean', zero_infinity = True) and its gradient with respect to the LOGITS.
 * logp f32 [B*T, ldl] = log_softmax of the assistor's logits (otb_log_softmax); in_len i32 [B] valid frames; targets i64
 * [B, ldt] label rows (the first tgt_len[b] entries count); max_tgt >= every tgt_len (<= 64); nll f32 [B] per-utterance
 * negative log-likelihood (+inf if infeasible); loss f32 [1]; ws f32 [B, T, 2 max_tgt + 1] scratch (alpha + beta);
 * dlogits_bf16 (optional, bf16 [B*T, ldd]) = grad_scale * d loss / d logits (padded frames / infeasible utterances: 0). */
int otb_ctc_loss(const float* logp, int ldl, int B, int T, int V, const int32_t* in_len, const int64_t* targets, int ldt,
                 const int32_t* tgt_len, int max_tgt, int blank, float* nll, float* loss, float* ws, void* dlogits_bf16, int ldd,
                 float grad_scale, void* stream);

/* Conv2d front end backward (frontend/conv.py:50-76 under autograd).  h1 = conv1 activation buffer (layout of
 * otb_conv1_relu).  col bf16 [B*T2*F2, 9*C1] = im2col of h1 for conv2 (k = (kh*3+kw)*C1 + c): conv2's weight gradient is
 * otb_linear_wgrad(dpre2, col) and its input gradient dcol = otb_linear(dpre2, W2^T).  otb_conv_col2im_relu folds dcol
 * back onto the conv1 grid and applies ReLU' -> dpre1 (h1 layout).  otb_conv1_wgrad: out f32 [C1, 10] = 9 tap
 * gradients + the bias gradient of conv1 (C_in = 1). */
int otb_conv_im2col(const void* h1, void* col, int B, int T, int F, int C1, void* stream);
int otb_conv_col2im_relu(const void* dcol, const void* h1, void* dpre1, int B, int T, int F, int C1, void* stream);
int otb_conv1_wgrad(const void* dpre1, const float* x, float* out, int B, int T, int F, int C1, void* stream);

/* SpecAugment (data/augment.py:9-41) applied on the device: zero n_freq frequency bands and n_time time bands per
 * utterance.  x f32 [B,T,F] in place; bands i32 [B, 2*(n_freq+n_time)] = (f0, width)*n_freq, (t0, width)*n_time drawn
 * on the host with the reference's RNG call order. */
int otb_spec_augment(float* x, const int32_t* bands, int B, int T, int F, int n_freq, int n_time, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OTB200_H_ */
