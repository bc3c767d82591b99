// Internal declarations shared by the .cu translation units of libotb200.so.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace otb {

typedef __nv_bfloat16 bf16;

// ---- epilogues of the tcgen05 GEMM (C = A[M,K] * W[N,K]^T, fp32 accumulate in TMEM) ----
enum Epilogue : int {
    EPI_BIAS = 0,      // out = acc + bias
    EPI_RELU = 1,      // out = relu(acc + bias)
    EPI_GLU = 2,       // W has 2*Nh rows; out[:, j] = (acc_j + b_j) * sigmoid(acc_{Nh+j} + b_{Nh+j})
    EPI_TABLE = 3,     // out = (acc + bias) * alpha + table[(row % period) * N + col]     (x*sqrt(d)+PE)
    EPI_RESID = 4,     // out = resid + alpha * (acc + bias)
    EPI_RESID_LN = 5,  // out = LayerNorm(resid + acc + bias) * gamma + beta   (tile spans the whole row)
    EPI_SWISH = 6,     // out = v * sigmoid(v), v = acc + bias
    EPI_GELU = 7,      // out = gelu(v) (erf form, as F.gelu)
    EPI_TANH = 8,      // out = tanh(v)
};

struct GemmParams {
    int M, N, K;  // N = number of output columns (for GLU: Nh); K multiple of 8
    const float* bias;
    void* out;
    int ldc;
    int out_f32;
    const bf16* resid;
    int ldr;
    const float* gamma;
    const float* beta;
    float eps;
    float alpha;
    const float* table;
    int period;
    const int* row_len;  // optional: rows with (m % row_period) >= row_len[m / row_period] produce 0 (before resid)
    int row_period;
    // implicit-GEMM 3x3/stride-2 convolution mode (A operand gathered by a 5-D TMA map)
    int conv;
    int conv_F2;       // output frequency bins
    int conv_R;        // output time rows per M tile (R * F2 <= 128)
    int conv_T1h;      // (padded input time rows) / 2
    int conv_T2;       // valid output time rows per utterance
    int conv_B;        // batch
    int conv_cchunks;  // C_in / 64
    int splitk;        // TN (weight-gradient) mode: number of contraction splits (fp32 atomics when > 1)
    int accum;         // TN mode: add into `out` instead of overwriting it
    // training-mode dropout of the projection BEFORE the residual add (EPI_RESID only): out = resid + alpha * keep * (.) / (1-p)
    const unsigned* drop_seed;    // device scalar, null = no dropout
    unsigned drop_site, drop_thresh;
    float drop_scale;
    unsigned long long* dbg;  // optional [grid][8] clock64 phase stamps (otb_debug_gemm_timing)
    int dbg_mode;             // 0 normal; 1 = no TMA traffic (MMA-only cadence); 2 = no MMA (TMA-only cadence)
};

const char* gemm_launch(cudaStream_t st, const void* A, int lda, const void* W, int ldw, int w_rows, int epi,
                        GemmParams p, const CUtensorMap* conv_map);

const char* gemm_wgrad_launch(cudaStream_t st, const void* dY, int lddy, const void* X, int ldx, float* out, int ldc,
                              int Mact, int Nw, int Kw, int accumulate);

// encode helpers (driver entry point fetched at runtime; libcuda is not a link-time dependency)
// swizzle_bytes: 128 (box of <= 64 columns) or 64 (box of <= 32 columns)
const char* encode_tmap_2d(CUtensorMap* m, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems,
                           uint32_t box_cols, uint32_t box_rows, int swizzle_bytes = 128);
const char* encode_tmap_2d_f32(CUtensorMap* m, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems,
                               uint32_t box_cols, uint32_t box_rows);
const char* encode_tmap_conv5d(CUtensorMap* m, const void* base, int C, int F1h, int T1h_total, uint32_t boxF,
                               uint32_t boxR);

struct AttnParams {
    int B, H, Tq, Tk;
    const int* kv_len;  // [B] or null
    int causal;
    float scale_log2;   // (1/sqrt(dk)) * log2(e)
    bf16* out;
    int ldo;
    int q_col0, k_col0, v_col0;
    const float* bd;    // optional relative-position scores, [H,B,Tq,ldbd]; bias(i,j) = bd[h,b,i, j - i + Tq - 1]
    int ldbd;
    const bf16* resid;  // optional: out = resid + softmax(..)V   (rel-pos attention has no output projection)
    int ldr;
    float* lse;         // optional [B,H,Tq]: row log-sum-exp of the scaled scores in log2 units (saved for the backward)
};

struct AttnBwdParams {
    int B, H, Tq, Tk;
    const int* kv_len;
    int causal;
    float scale_log2;
    int q_col0, k_col0, v_col0;
    const bf16* o;      // forward output [B*Tq, ldo]
    int ldo;
    const bf16* dout;   // gradient of the forward output [B*Tq, lddo]
    int lddo;
    const float* lse;   // [B,H,Tq] from the forward
    float* dsum;        // [B,H,Tq] scratch: D_i = dO_i . O_i (written by the dQ kernel, read by the dK/dV kernel)
    bf16* dq; int lddq, dq_col0;
    bf16* dk; int lddk, dk_col0;
    bf16* dv; int lddv, dv_col0;
};
const char* attn_bwd_launch(cudaStream_t st, const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows,
                            const void* v, int ldv, const AttnBwdParams& p);
const char* colsum_launch(cudaStream_t st, const bf16* x, int ldx, float* out, int M, int N, int accumulate);
const char* layernorm_bwd_launch(cudaStream_t st, const bf16* dy, int lddy, const bf16* z, int ldz, const float* gamma,
                                 bf16* dz, int lddz, float* dgamma, float* dbeta, float eps, int M, int N, int accumulate);
const char* glu_launch(cudaStream_t st, const bf16* u, const bf16* dh, bf16* out, int M, int F);
const char* relu_bwd_launch(cudaStream_t st, const bf16* dy, const bf16* y, bf16* dx, size_t n);
const char* dropout_bwd_launch(cudaStream_t st, const bf16* dy, int lddy, bf16* out, int ldo, unsigned char* mask, int M, int N, float p,
                               const unsigned* seed, unsigned site);
const char* embed_bwd_launch(cudaStream_t st, const long long* tok, const bf16* dx, float* dE, int N, int d, int vocab, float scale);
const char* im2col_s2_launch(cudaStream_t st, const bf16* h1, bf16* col, int B, int T2, int F2, int C);
const char* col2im_s2_relu_launch(cudaStream_t st, const bf16* dcol, const bf16* h1, bf16* dpre1, int B, int T1, int F1, int T2,
                                  int F2, int C);
const char* conv1_wgrad_launch(cudaStream_t st, const bf16* dpre1, const float* x, float* out, int B, int T, int F, int T1,
                               int F1, int T2, int F2, int C);
const char* spec_augment_launch(cudaStream_t st, float* x, const int* bands, int B, int T, int F, int nf, int nt);
const char* sumsq_launch(cudaStream_t st, const float* g, size_t n, float* out, int zero_first);
const char* adam_launch(cudaStream_t st, float* p, const float* g, float* m, float* v, size_t n, const float* sumsq,
                        float max_norm, float lr, float b1, float b2, float eps, float wd, int step);
const char* adam_sched_launch(cudaStream_t st, float* p, const float* g, float* m, float* v, size_t n, const float* sumsq,
                              float max_norm, float base_lr, float model_size, float warmup, float factor, float b1, float b2,
                              float eps, float wd, int* counters, float* hyper);

struct BeamState {
    int* tok_hist;
    int* par_hist;
    long long* last_tok;
    float* scores;
    unsigned char* flag;
    int* anc;
    int* ctrl;
    int N, beam, Lmax;
};

// ---- persistent decode kernel (decode_mega.cu)
static constexpr int OTB_MEGA_MAX_LAYERS_INT = 8;
struct MegaLayer {   // one TransformerDecoderLayer: bf16 weights [N,K] row-major, fp32 biases / LayerNorm affine
    const bf16 *wqkv, *wo, *wq, *wo2, *w1, *w2;
    const float *bqkv, *bo, *bq, *bo2, *b1, *b2;
    const float *g1, *be1, *g2, *be2, *g3, *be3;
};
struct MegaParams {
    int n_layers, d, H, dff, V;
    const bf16* emb;      // [V, d] embedding
    const bf16* wout;     // [V, d] output layer (== emb when tied)
    const float* bout;    // [V] or null
    const float* pe;      // [>= max_steps, d] sinusoid table
    MegaLayer layers[OTB_MEGA_MAX_LAYERS_INT];
    const bf16* kvx;      // [n_layers, B*T, 2d] cross-attention K | V
    const int* mem_len;   // [B]
    bf16* kc;             // [n_layers, Lmax, N, d]
    bf16* vc;
    BeamState st;
    int B, T, max_steps;
    float eps;
    float* dbg_logp;      // optional [max_steps, N, V]
    float* dbg_scores;    // optional [max_steps, N]
};
// ---- persistent decode kernel, round 2 (decode_group.cu): row groups of <= 128 hypotheses x 16 CTAs, tcgen05 GEMMs
struct DgLayer {
    const float *bqkv, *bo, *bq, *bo2, *b1, *b2;
    const float *g1, *be1, *g2, *be2, *g3, *be3;
};
struct DgParams {
    int n_layers, V, G, utts_per_group;
    int cluster;               // 1: launched as thread-block clusters of 16 (group == cluster, hardware barrier)
    const bf16* emb;
    const float* bout;
    const float* pe;
    DgLayer layers[OTB_MEGA_MAX_LAYERS_INT];
    const CUtensorMap* maps;   // device array: per layer {wqkv, wo, wq, wo2, w1, w2}, then wout, ctx, kvx
    const int* mem_len;
    bf16* kc;
    bf16* vc;
    BeamState st;
    int B, T, max_steps;
    float eps;
    bf16* qbuf;                // [N, d]   self-attention queries of the newest token
    bf16* ctx;                 // [N + 128, d] attention context (self, then cross)
    bf16* xbuf;                // [N + 128, d] layer input x (embedding / LayerNorm 3 of the previous layer)
    bf16* x2buf;               // [N, d]   LayerNorm 2 output (residual of the feed-forward)
    float* pre;                // [N, d]   pre-LayerNorm rows (residual + projection + bias), fp32
    bf16* q2;                  // [N, d]   cross-attention queries
    int flags;                 // experiment switches (OTB_DG_FLAGS)
    float* part;               // [16 slices][groups][64 column groups][128 rows][4] w_2 partial products (fp32)
    float* logits;             // [N, ldv] output-layer logits of the step
    int ldv;
    int* bar;                  // [G, 32]  group barrier counters
    int* gstate;               // [G, Lmax] ended-hypothesis count per step
    float* dbg_logp;
    float* dbg_scores;
    unsigned long long* dbg_clk;
    int dbg_step;
};
extern unsigned long long* g_dg_dbg;
extern int g_dg_dbg_step;
extern int g_dg_barrier;
size_t decode_group_workspace_bytes(int N, int n_layers, int Lmax, int B, int beam, int V);
const char* decode_group_launch(cudaStream_t st, const MegaParams& p, void* workspace, size_t workspace_bytes);

const char* attn_launch(cudaStream_t st, const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows,
                        const void* v, int ldv, const AttnParams& p, int head_dim);   // head_dim 64 or 96
const char* conv1_launch(cudaStream_t st, const float* x, const float* w, const float* bias, bf16* out, int B, int T,
                         int F, int T1, int F1, int T1pad, int F1pad, int C1);
const char* layernorm_launch(cudaStream_t st, const bf16* x, int ldx, void* out, int ldo, int out_f32, const float* g1,
                             const float* b1, const float* g2, const float* b2, float eps, int M, int N);
const char* scale_add_table_launch(cudaStream_t st, const void* x, int ldx, int x_f32, bf16* out, int ldo, float alpha,
                                   const float* table, int period, int M, int N);
const char* dwconv_swish_launch(cudaStream_t st, const bf16* x, const float* w, const float* b, bf16* out, int B, int T,
                                int d, int k);
const char* sinusoid_table_launch(cudaStream_t st, float* out, int n_pos, int d, int first_pos);
const char* embed_posenc_launch(cudaStream_t st, const long long* tok, int tok_stride, const bf16* emb,
                                const float* table, bf16* out, int N, int d, int period, const int* step_ptr,
                                int vocab);
const char* log_softmax_launch(cudaStream_t st, const float* x, int ldx, float* out, int ldo, int rows, int V);
const char* decode_self_attn_launch(cudaStream_t st, const bf16* qkv, bf16* kc, bf16* vc, const int* anc,
                                    const int* step_ptr, bf16* out, int N, int H, int Lmax, int head_dim);
const char* beam_init_launch(cudaStream_t stream, BeamState st);
const char* beam_step_launch(cudaStream_t stream, const float* logp, int ldl, int V, const float* lm_logp, int ld_lm,
                             float lm_weight, BeamState st, long long* dbg_ktok, int* dbg_offs, const float* pre_val,
                             const int* pre_idx);
const char* logsoftmax_topk_launch(cudaStream_t stream, const float* logits, int ldl, int V, const float* lm_logp,
                                   int ld_lm, float lm_weight, int k, int rows, float* out_val, int* out_idx,
                                   float* out_logp, int ld_logp);
const char* beam_reconstruct_launch(cudaStream_t stream, BeamState st, long long* preds, int ld, int steps);
const char* beam_finalize_launch(cudaStream_t stream, BeamState st, float penalty, float lamda, int nbest,
                                 long long* out_preds, float* out_scores);

const char* ls_ce_launch(cudaStream_t st, const float* logits, int ldl, const long long* tgt, int rows, int V, float eps,
                         int pad_id, float* tok_loss, float* loss, int* n_valid, float* dlogits, int ldd,
                         bf16* dlogits_bf16 = nullptr);

const char* ctc_launch(cudaStream_t st, const float* logp, int ldl, int B, int T, int V, const int* in_len, const long long* targets,
                       int ldt, const int* tgt_len, int max_tgt, int blank, float* nll, float* loss, float* ws, bf16* dlogits, int ldd,
                       float grad_scale);

const char* fbank_launch(cudaStream_t st, const float* wave, int ld_wave, const int* n_samples, int B, const float* window,
                         const float* bank, const int* bank_range, float* out, int Tmax, int F, int frame_len, int frame_shift,
                         float preemph);
const char* utt_cmvn_launch(cudaStream_t st, float* x, int B, int Tmax, int F, const int* n_frames, const float* gmean, const float* gstd);

int num_sms();
extern unsigned long long* g_gemm_dbg;
extern int g_gemm_dbg_mode;
extern int g_tile_policy;
void set_error(const char* msg);

}  // namespace otb
