// extern "C" boundary of libotb200.so (declared in include/otb200.h).  Argument checking, error
// reporting (thread-local string, integer status, no aborts) and dispatch to the kernel launchers.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include "../../include/otb200.h"
#include "dropout.cuh"
#include "otb_internal.h"

namespace otb {


static thread_local char g_err[512] = "";
void set_error(const char* msg) {
    strncpy(g_err, msg ? msg : "", sizeof(g_err) - 1);
    g_err[sizeof(g_err) - 1] = 0;
}
static int fail(const char* where, const char* msg) {
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s", where, msg);
    set_error(buf);
    return 1;
}
static BeamState to_state(const otb_beam_state* s) {
    BeamState b;
    b.tok_hist = s->tok_hist; b.par_hist = s->par_hist; b.last_tok = (long long*)s->last_tok;
    b.scores = s->scores; b.flag = s->flag; b.anc = s->anc; b.ctrl = s->ctrl;
    b.N = s->N; b.beam = s->beam; b.Lmax = s->Lmax;
    return b;
}

}  // namespace otb

using namespace otb;
#define ST(s) reinterpret_cast<cudaStream_t>(s)
#define RET(where, expr)                      \
    do {                                      \
        const char* _e = (expr);              \
        if (_e) return fail(where, _e);       \
        return 0;                             \
    } while (0)

extern "C" {

const char* otb_last_error(void) { return g_err; }
int otb_version(void) { return OTB_VERSION; }
int otb_num_sms(void) { return num_sms(); }

/* debug / profiling aid: when buf != NULL every GEMM CTA writes 8 clock64 phase stamps to buf[cta*8 ..] */
int otb_debug_gemm_timing(unsigned long long* buf) {
    g_gemm_dbg = buf;
    return 0;
}
int otb_set_tile_policy(int policy) {
    if (policy != 0 && policy != 1) return fail("otb_set_tile_policy", "policy must be 0 (latency) or 1 (throughput)");
    g_tile_policy = policy;
    return 0;
}
int otb_debug_gemm_mode(int mode) {
    g_gemm_dbg_mode = mode;
    return 0;
}

int otb_debug_decode_timing(unsigned long long* buf, int step) {
    g_dg_dbg = buf;
    g_dg_dbg_step = step;
    return 0;
}

int otb_set_decode_barrier(int kind) {
    if (kind < -1 || kind > 1) return fail("otb_set_decode_barrier", "kind must be -1 (default), 0 (software) or 1 (cluster)");
    g_dg_barrier = kind;
    return 0;
}

int otb_conv_geometry(int T, int F, int* T1, int* F1, int* T2, int* F2) {
    if (T < 7 || F < 1) return fail("otb_conv_geometry", "need T >= 7 and F >= 1");
    const int t1 = (T - 3) / 2 + 1, f1 = (F - 1) / 2 + 1;
    const int t2 = (t1 - 3) / 2 + 1, f2 = (f1 - 1) / 2 + 1;
    if (T1) *T1 = t1;
    if (F1) *F1 = f1;
    if (T2) *T2 = t2;
    if (F2) *F2 = f2;
    return 0;
}

int otb_conv1_relu(const float* x, const float* w, const float* bias, void* out, int B, int T, int F, int C1,
                   void* stream) {
    int T1, F1, T2, F2;
    if (otb_conv_geometry(T, F, &T1, &F1, &T2, &F2)) return 1;
    if (!x || !w || !bias || !out || B < 1) return fail("otb_conv1_relu", "null pointer or empty batch");
    RET("otb_conv1_relu",
        conv1_launch(ST(stream), x, w, bias, reinterpret_cast<bf16*>(out), B, T, F, T1, F1, 2 * (T2 + 1), 2 * F2, C1));
}

int otb_conv2_relu(const void* in, const void* w, const float* bias, void* out, int B, int T, int F, int C1, int C2,
                   void* stream) {
    int T1, F1, T2, F2;
    if (otb_conv_geometry(T, F, &T1, &F1, &T2, &F2)) return 1;
    if (!in || !w || !bias || !out || B < 1) return fail("otb_conv2_relu", "null pointer or empty batch");
    if (C1 % 64) return fail("otb_conv2_relu", "C1 must be a multiple of 64 (one 128-byte tap per k-block)");
    if (C2 % 8) return fail("otb_conv2_relu", "C2 must be a multiple of 8");
    if (F2 > 128) return fail("otb_conv2_relu", "F2 > 128 not supported");
    const int T1h = T2 + 1;
    int R = 128 / F2;
    if (R > T1h) R = T1h;
    if (R > 256) R = 256;
    CUtensorMap cmap;
    const char* e = encode_tmap_conv5d(&cmap, in, C1, F2, B * T1h, (uint32_t)F2, (uint32_t)R);
    if (e) return fail("otb_conv2_relu", e);
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = B * T2 * F2;
    p.N = C2;
    p.K = 9 * C1;
    p.bias = bias;
    p.out = out;
    p.ldc = C2;
    p.alpha = 1.f;
    p.conv = 1;
    p.conv_F2 = F2;
    p.conv_R = R;
    p.conv_T1h = T1h;
    p.conv_T2 = T2;
    p.conv_B = B;
    p.conv_cchunks = C1 / 64;
    RET("otb_conv2_relu", gemm_launch(ST(stream), nullptr, 0, w, 9 * C1, C2, EPI_RELU, p, &cmap));
}

int otb_linear(const void* a, int lda, const void* w, int ldw, const float* bias, void* out, int ldc, int M, int N,
               int K, int epilogue, int out_f32, const void* resid, int ldr, const float* gamma, const float* beta,
               float eps, float alpha, const float* table, int period, const int* row_len, int row_period,
               void* stream) {
    if (!a || !w || !out) return fail("otb_linear", "null operand");
    if (epilogue < 0 || epilogue > EPI_TANH) return fail("otb_linear", "unknown epilogue");
    if ((epilogue == EPI_RESID || epilogue == EPI_RESID_LN) && !resid) return fail("otb_linear", "residual epilogue without resid");
    if (epilogue == EPI_RESID_LN && (!gamma || !beta)) return fail("otb_linear", "LayerNorm epilogue without gamma/beta");
    if (epilogue == EPI_TABLE && (!table || period < 1)) return fail("otb_linear", "table epilogue without table/period");
    if (row_len && row_period < 1) return fail("otb_linear", "row_len without row_period");
    if (out_f32 ? (ldc < N) : (ldc < N)) return fail("otb_linear", "ldc < N");
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = M; p.N = N; p.K = K;
    p.bias = bias;
    p.out = out; p.ldc = ldc; p.out_f32 = out_f32;
    p.resid = reinterpret_cast<const bf16*>(resid); p.ldr = ldr;
    p.gamma = gamma; p.beta = beta; p.eps = eps; p.alpha = alpha;
    p.table = table; p.period = period;
    p.row_len = row_len; p.row_period = row_period;
    const int w_rows = (epilogue == EPI_GLU) ? 2 * N : N;
    RET("otb_linear", gemm_launch(ST(stream), a, lda, w, ldw, w_rows, epilogue, p, nullptr));
}

int otb_linear_dropout_resid(const void* a, int lda, const void* w, int ldw, const float* bias, void* out, int ldc, int M, int N, int K,
                             const void* resid, int ldr, float alpha, float p_drop, const uint32_t* seed, uint32_t site, void* stream) {
    if (!a || !w || !out || !resid || !seed) return fail("otb_linear_dropout_resid", "null operand");
    if (!(p_drop >= 0.f && p_drop < 1.f)) return fail("otb_linear_dropout_resid", "p must be in [0, 1)");
    if (ldc < N) return fail("otb_linear_dropout_resid", "ldc < N");
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = M; p.N = N; p.K = K;
    p.bias = bias;
    p.out = out; p.ldc = ldc; p.out_f32 = 0;
    p.resid = reinterpret_cast<const bf16*>(resid); p.ldr = ldr;
    p.alpha = alpha;
    p.drop_seed = seed; p.drop_site = site; p.drop_thresh = drop_threshold(p_drop); p.drop_scale = 1.0f / (1.0f - p_drop);
    RET("otb_linear_dropout_resid", gemm_launch(ST(stream), a, lda, w, ldw, N, EPI_RESID, p, nullptr));
}

int otb_dropout_bwd(const void* dy, int lddy, void* out, int ldo, uint8_t* mask, int M, int N, float p, const uint32_t* seed,
                    uint32_t site, void* stream) {
    if ((!dy || !out) && !mask) return fail("otb_dropout_bwd", "nothing to do");
    RET("otb_dropout_bwd", dropout_bwd_launch(ST(stream), reinterpret_cast<const bf16*>(dy), lddy, reinterpret_cast<bf16*>(out), ldo, mask, M, N,
                                              p, seed, site));
}

int otb_attention(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                  void* out, int ldo, int B, int H, int Tq, int Tk, const int* kv_len, int causal, int q_col0,
                  int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, void* stream) {
    return otb_attention_lse_hd(q, ldq, q_rows, k, ldk, k_rows, v, ldv, out, ldo, B, H, 64, Tq, Tk, kv_len, causal, q_col0,
                                k_col0, v_col0, bd, ldbd, resid, ldr, nullptr, stream);
}

int otb_attention_hd(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                     void* out, int ldo, int B, int H, int head_dim, int Tq, int Tk, const int* kv_len, int causal, int q_col0,
                     int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, void* stream) {
    return otb_attention_lse_hd(q, ldq, q_rows, k, ldk, k_rows, v, ldv, out, ldo, B, H, head_dim, Tq, Tk, kv_len, causal, q_col0,
                                k_col0, v_col0, bd, ldbd, resid, ldr, nullptr, stream);
}

int otb_attention_lse(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                      void* out, int ldo, int B, int H, int Tq, int Tk, const int* kv_len, int causal, int q_col0,
                      int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, float* lse,
                      void* stream) {
    return otb_attention_lse_hd(q, ldq, q_rows, k, ldk, k_rows, v, ldv, out, ldo, B, H, 64, Tq, Tk, kv_len, causal, q_col0,
                                k_col0, v_col0, bd, ldbd, resid, ldr, lse, stream);
}

int otb_attention_lse_hd(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                         void* out, int ldo, int B, int H, int head_dim, int Tq, int Tk, const int* kv_len, int causal,
                         int q_col0, int k_col0, int v_col0, const float* bd, int ldbd, const void* resid, int ldr, float* lse,
                         void* stream) {
    if (head_dim != 64 && head_dim != 96) return fail("otb_attention", "head_dim must be 64 or 96");
    if (!q || !k || !v || !out) return fail("otb_attention", "null operand");
    if (q_col0 % 8 || k_col0 % 8 || v_col0 % 8 || ldo % 8) return fail("otb_attention", "column offsets / ldo must be multiples of 8");
    AttnParams p;
    p.B = B; p.H = H; p.Tq = Tq; p.Tk = Tk;
    p.kv_len = kv_len; p.causal = causal;
    p.scale_log2 = (head_dim == 64 ? 0.125f : 1.0f / sqrtf((float)head_dim)) * 1.4426950408889634f;
    p.out = reinterpret_cast<bf16*>(out); p.ldo = ldo;
    p.q_col0 = q_col0; p.k_col0 = k_col0; p.v_col0 = v_col0;
    p.bd = bd; p.ldbd = ldbd;
    p.resid = reinterpret_cast<const bf16*>(resid); p.ldr = ldr;
    p.lse = lse;
    if (resid && (ldr % 8)) return fail("otb_attention", "ldr must be a multiple of 8");
    RET("otb_attention", attn_launch(ST(stream), q, ldq, q_rows, k, ldk, k_rows, v, ldv, p, head_dim));
}

int otb_layernorm(const void* x, int ldx, void* out, int ldo, int out_f32, const float* g1, const float* b1,
                  const float* g2, const float* b2, float eps, int M, int N, void* stream) {
    if (!x || !out || !g1 || !b1) return fail("otb_layernorm", "null operand");
    if ((g2 == nullptr) != (b2 == nullptr)) return fail("otb_layernorm", "g2/b2 must both be given");
    RET("otb_layernorm", layernorm_launch(ST(stream), reinterpret_cast<const bf16*>(x), ldx, out, ldo, out_f32, g1, b1,
                                          g2, b2, eps, M, N));
}

int otb_scale_add_table(const void* x, int ldx, int x_f32, void* out, int ldo, float alpha, const float* table,
                        int period, int M, int N, void* stream) {
    if (!x || !out || M < 1 || N < 1) return fail("otb_scale_add_table", "bad arguments");
    if (table && period < 1) return fail("otb_scale_add_table", "table without period");
    RET("otb_scale_add_table", scale_add_table_launch(ST(stream), x, ldx, x_f32, reinterpret_cast<bf16*>(out), ldo, alpha,
                                                      table, period, M, N));
}

int otb_dwconv_swish(const void* x, const float* w, const float* b, void* out, int B, int T, int d, int k,
                     void* stream) {
    if (!x || !w || !b || !out || B < 1 || T < 1) return fail("otb_dwconv_swish", "bad arguments");
    RET("otb_dwconv_swish", dwconv_swish_launch(ST(stream), reinterpret_cast<const bf16*>(x), w, b,
                                                reinterpret_cast<bf16*>(out), B, T, d, k));
}

int otb_sinusoid_table(float* out, int n_pos, int d, int first_pos, void* stream) {
    if (!out || n_pos < 1 || d < 2 || (d & 1)) return fail("otb_sinusoid_table", "bad arguments");
    RET("otb_sinusoid_table", sinusoid_table_launch(ST(stream), out, n_pos, d, first_pos));
}

int otb_embed_posenc(const int64_t* tok, int tok_stride, const void* emb, const float* table, void* out, int N,
                     int d, int period, const int* step_ptr, int vocab, void* stream) {
    if (!tok || !emb || !table || !out) return fail("otb_embed_posenc", "null operand");
    if (!step_ptr && period < 1) return fail("otb_embed_posenc", "need period or step_ptr");
    RET("otb_embed_posenc",
        embed_posenc_launch(ST(stream), reinterpret_cast<const long long*>(tok), tok_stride,
                            reinterpret_cast<const bf16*>(emb), table, reinterpret_cast<bf16*>(out), N, d, period,
                            step_ptr, vocab));
}

int otb_log_softmax(const float* x, int ldx, float* out, int ldo, int rows, int V, void* stream) {
    if (!x || !out || rows < 1 || V < 1) return fail("otb_log_softmax", "bad arguments");
    RET("otb_log_softmax", log_softmax_launch(ST(stream), x, ldx, out, ldo, rows, V));
}

int otb_decode_self_attn(const void* qkv, void* kc, void* vc, const int* anc, const int* step_ptr, void* out, int N,
                         int H, int Lmax, void* stream) {
    return otb_decode_self_attn_hd(qkv, kc, vc, anc, step_ptr, out, N, H, 64, Lmax, stream);
}

int otb_decode_self_attn_hd(const void* qkv, void* kc, void* vc, const int* anc, const int* step_ptr, void* out, int N,
                            int H, int head_dim, int Lmax, void* stream) {
    if (head_dim != 64 && head_dim != 96) return fail("otb_decode_self_attn", "head_dim must be 64 or 96");
    if (!qkv || !kc || !vc || !anc || !step_ptr || !out) return fail("otb_decode_self_attn", "null operand");
    RET("otb_decode_self_attn",
        decode_self_attn_launch(ST(stream), reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(kc),
                                reinterpret_cast<bf16*>(vc), anc, step_ptr, reinterpret_cast<bf16*>(out), N, H, Lmax, head_dim));
}

int otb_ls_ce(const float* logits, int ldl, const int64_t* targets, int rows, int V, float smoothing, int pad_id,
              float* tok_loss, float* loss, int32_t* n_valid, float* dlogits, int ldd, void* stream) {
    if (!logits || !targets || !tok_loss || !loss || !n_valid) return fail("otb_ls_ce", "null operand");
    RET("otb_ls_ce", ls_ce_launch(ST(stream), logits, ldl, reinterpret_cast<const long long*>(targets), rows, V, smoothing,
                                  pad_id, tok_loss, loss, n_valid, dlogits, ldd));
}

int otb_beam_init(const otb_beam_state* st, void* stream) {
    if (!st) return fail("otb_beam_init", "null state");
    RET("otb_beam_init", beam_init_launch(ST(stream), to_state(st)));
}

int otb_beam_step(const float* logp, int ldl, int V, const float* lm_logp, int ld_lm, float lm_weight,
                  const otb_beam_state* st, int64_t* dbg_ktok, int32_t* dbg_offs, void* stream) {
    if (!st || !logp) return fail("otb_beam_step", "null operand");
    RET("otb_beam_step", beam_step_launch(ST(stream), logp, ldl, V, lm_logp, ld_lm, lm_weight, to_state(st),
                                          reinterpret_cast<long long*>(dbg_ktok), dbg_offs, nullptr, nullptr));
}

int otb_beam_step_topk(const float* topk_val, const int32_t* topk_idx, const otb_beam_state* st, int64_t* dbg_ktok,
                       int32_t* dbg_offs, void* stream) {
    if (!st || !topk_val || !topk_idx) return fail("otb_beam_step_topk", "null operand");
    RET("otb_beam_step_topk", beam_step_launch(ST(stream), nullptr, 0, 0, nullptr, 0, 0.f, to_state(st),
                                               reinterpret_cast<long long*>(dbg_ktok), dbg_offs, topk_val, topk_idx));
}

int otb_logsoftmax_topk(const float* logits, int ldl, int V, const float* lm_logp, int ld_lm, float lm_weight, int k,
                        int rows, float* out_val, int32_t* out_idx, float* out_logp, int ld_logp, void* stream) {
    if (!logits || !out_val || !out_idx || rows < 1) return fail("otb_logsoftmax_topk", "bad arguments");
    RET("otb_logsoftmax_topk", logsoftmax_topk_launch(ST(stream), logits, ldl, V, lm_logp, ld_lm, lm_weight, k, rows,
                                                      out_val, out_idx, out_logp, ld_logp));
}

int otb_beam_reconstruct(const otb_beam_state* st, int64_t* preds, int ld, int steps, void* stream) {
    if (!st || !preds) return fail("otb_beam_reconstruct", "null operand");
    RET("otb_beam_reconstruct", beam_reconstruct_launch(ST(stream), to_state(st), reinterpret_cast<long long*>(preds), ld, steps));
}

int otb_beam_finalize(const otb_beam_state* st, float penalty, float lamda, int nbest, int64_t* out_preds,
                      float* out_scores, void* stream) {
    if (!st || !out_preds || !out_scores) return fail("otb_beam_finalize", "null operand");
    RET("otb_beam_finalize", beam_finalize_launch(ST(stream), to_state(st), penalty, lamda, nbest,
                                                  reinterpret_cast<long long*>(out_preds), out_scores));
}

long long otb_decode_persistent_workspace(int N, int n_layers, int Lmax, int B, int beam, int vocab) {
    if (N < 1 || n_layers < 1 || Lmax < 1 || B < 1 || beam < 1 || beam > 16 || vocab < 1) return -1;
    return (long long)decode_group_workspace_bytes(N, n_layers, Lmax, B, beam, vocab);
}

int otb_decode_persistent(const otb_mega_model* model, const void* kvx, const int32_t* mem_len, void* kc, void* vc,
                          const otb_beam_state* st, int B, int T, int max_steps, void* workspace, long long workspace_bytes,
                          float* dbg_logp, float* dbg_scores, void* stream) {
    if (!model || !kvx || !mem_len || !kc || !vc || !st || !workspace) return fail("otb_decode_persistent", "null operand");
    if (model->n_layers < 1 || model->n_layers > OTB_MEGA_MAX_LAYERS) return fail("otb_decode_persistent", "1..8 decoder layers");
    MegaParams p;
    memset(&p, 0, sizeof(p));
    p.n_layers = model->n_layers; p.d = model->d_model; p.H = model->n_heads; p.dff = model->d_ff; p.V = model->vocab;
    p.emb = reinterpret_cast<const bf16*>(model->emb);
    p.wout = reinterpret_cast<const bf16*>(model->wout);
    p.bout = model->bout;
    p.pe = model->pe;
    if (!p.emb || !p.wout || !p.pe) return fail("otb_decode_persistent", "null model tensor");
    for (int l = 0; l < model->n_layers; ++l) {
        const otb_mega_layer& s = model->layers[l];
        MegaLayer& d = p.layers[l];
        d.wqkv = (const bf16*)s.wqkv; d.wo = (const bf16*)s.wo; d.wq = (const bf16*)s.wq; d.wo2 = (const bf16*)s.wo2;
        d.w1 = (const bf16*)s.w1; d.w2 = (const bf16*)s.w2;
        d.bqkv = s.bqkv; d.bo = s.bo; d.bq = s.bq; d.bo2 = s.bo2; d.b1 = s.b1; d.b2 = s.b2;
        d.g1 = s.g1; d.be1 = s.be1; d.g2 = s.g2; d.be2 = s.be2; d.g3 = s.g3; d.be3 = s.be3;
        const void* need[18] = {s.wqkv, s.wo, s.wq, s.wo2, s.w1, s.w2, s.bqkv, s.bo, s.bq, s.bo2, s.b1, s.b2,
                                s.g1, s.be1, s.g2, s.be2, s.g3, s.be3};
        for (int i = 0; i < 18; ++i)
            if (!need[i]) return fail("otb_decode_persistent", "null layer tensor (biases are required)");
    }
    p.kvx = reinterpret_cast<const bf16*>(kvx);
    p.mem_len = mem_len;
    p.kc = reinterpret_cast<bf16*>(kc);
    p.vc = reinterpret_cast<bf16*>(vc);
    p.st = to_state(st);
    p.B = B; p.T = T; p.max_steps = max_steps;
    p.eps = model->ln_eps;
    p.dbg_logp = dbg_logp; p.dbg_scores = dbg_scores;
    RET("otb_decode_persistent", decode_group_launch(ST(stream), p, workspace, (size_t)workspace_bytes));
}

int otb_attention_bwd(const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows, const void* v, int ldv,
                      const void* out, int ldo, const void* dout, int lddo, const float* lse, float* dsum, void* dq,
                      int lddq, int dq_col0, void* dk, int lddk, int dk_col0, void* dv, int lddv, int dv_col0, int B, int H,
                      int Tq, int Tk, const int* kv_len, int causal, int q_col0, int k_col0, int v_col0, void* stream) {
    if (!q || !k || !v || !out || !dout || !lse || !dsum || !dq || !dk || !dv) return fail("otb_attention_bwd", "null operand");
    if ((q_col0 | k_col0 | v_col0 | dq_col0 | dk_col0 | dv_col0 | ldo | lddo | lddq | lddk | lddv) % 8)
        return fail("otb_attention_bwd", "column offsets / leading dimensions must be multiples of 8");
    AttnBwdParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.H = H; p.Tq = Tq; p.Tk = Tk; p.kv_len = kv_len; p.causal = causal;
    p.scale_log2 = 0.125f * 1.4426950408889634f;
    p.q_col0 = q_col0; p.k_col0 = k_col0; p.v_col0 = v_col0;
    p.o = reinterpret_cast<const bf16*>(out); p.ldo = ldo;
    p.dout = reinterpret_cast<const bf16*>(dout); p.lddo = lddo;
    p.lse = lse; p.dsum = dsum;
    p.dq = reinterpret_cast<bf16*>(dq); p.lddq = lddq; p.dq_col0 = dq_col0;
    p.dk = reinterpret_cast<bf16*>(dk); p.lddk = lddk; p.dk_col0 = dk_col0;
    p.dv = reinterpret_cast<bf16*>(dv); p.lddv = lddv; p.dv_col0 = dv_col0;
    RET("otb_attention_bwd", attn_bwd_launch(ST(stream), q, ldq, q_rows, k, ldk, k_rows, v, ldv, p));
}

int otb_linear_wgrad(const void* dy, int lddy, const void* x, int ldx, float* dw, int lddw, int M, int N, int K, int accumulate,
                     void* stream) {
    if (!dy || !x || !dw) return fail("otb_linear_wgrad", "null operand");
    RET("otb_linear_wgrad", gemm_wgrad_launch(ST(stream), dy, lddy, x, ldx, dw, lddw, M, N, K, accumulate));
}

int otb_colsum(const void* x, int ldx, float* out, int M, int N, int accumulate, void* stream) {
    if (!x || !out || M < 1 || N < 1) return fail("otb_colsum", "bad arguments");
    RET("otb_colsum", colsum_launch(ST(stream), reinterpret_cast<const bf16*>(x), ldx, out, M, N, accumulate));
}

int otb_layernorm_bwd(const void* dy, int lddy, const void* z, int ldz, const float* gamma, void* dz, int lddz,
                      float* dgamma, float* dbeta, float eps, int M, int N, int accumulate, void* stream) {
    if (!dy || !z || !gamma || !dz || !dgamma || !dbeta) return fail("otb_layernorm_bwd", "null operand");
    RET("otb_layernorm_bwd", layernorm_bwd_launch(ST(stream), reinterpret_cast<const bf16*>(dy), lddy,
                                                  reinterpret_cast<const bf16*>(z), ldz, gamma, reinterpret_cast<bf16*>(dz),
                                                  lddz, dgamma, dbeta, eps, M, N, accumulate));
}

int otb_glu_fwd(const void* u, void* h, int M, int F, void* stream) {
    if (!u || !h || M < 1 || F < 8) return fail("otb_glu_fwd", "bad arguments");
    RET("otb_glu_fwd", glu_launch(ST(stream), reinterpret_cast<const bf16*>(u), nullptr, reinterpret_cast<bf16*>(h), M, F));
}

int otb_glu_bwd(const void* dh, const void* u, void* du, int M, int F, void* stream) {
    if (!dh || !u || !du || M < 1 || F < 8) return fail("otb_glu_bwd", "bad arguments");
    RET("otb_glu_bwd", glu_launch(ST(stream), reinterpret_cast<const bf16*>(u), reinterpret_cast<const bf16*>(dh),
                                  reinterpret_cast<bf16*>(du), M, F));
}

int otb_relu_bwd(const void* dy, const void* y, void* dx, long long n, void* stream) {
    if (!dy || !y || !dx || n < 8) return fail("otb_relu_bwd", "bad arguments");
    RET("otb_relu_bwd", relu_bwd_launch(ST(stream), reinterpret_cast<const bf16*>(dy), reinterpret_cast<const bf16*>(y),
                                        reinterpret_cast<bf16*>(dx), (size_t)n));
}

int otb_embed_bwd(const int64_t* tok, const void* dx, float* dE, int N, int d, int vocab, float scale, void* stream) {
    if (!tok || !dx || !dE || N < 1) return fail("otb_embed_bwd", "bad arguments");
    RET("otb_embed_bwd", embed_bwd_launch(ST(stream), reinterpret_cast<const long long*>(tok), reinterpret_cast<const bf16*>(dx),
                                          dE, N, d, vocab, scale));
}

int otb_ls_ce_train(const float* logits, int ldl, const int64_t* targets, int rows, int V, float smoothing, int pad_id,
                    float* tok_loss, float* loss, int32_t* n_valid, void* dlogits_bf16, int ldd, void* stream) {
    if (!logits || !targets || !tok_loss || !loss || !n_valid || !dlogits_bf16) return fail("otb_ls_ce_train", "null operand");
    if (ldd < V || ldd % 8) return fail("otb_ls_ce_train", "ldd must be >= V and a multiple of 8");
    RET("otb_ls_ce_train", ls_ce_launch(ST(stream), logits, ldl, reinterpret_cast<const long long*>(targets), rows, V, smoothing,
                                        pad_id, tok_loss, loss, n_valid, nullptr, ldd, reinterpret_cast<bf16*>(dlogits_bf16)));
}

int otb_sumsq(const float* g, long long n, float* out, int zero_first, void* stream) {
    if (!g || !out || n < 1) return fail("otb_sumsq", "bad arguments");
    RET("otb_sumsq", sumsq_launch(ST(stream), g, (size_t)n, out, zero_first));
}

int otb_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* sumsq, float max_norm, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int step, void* stream) {
    if (!p || !g || !m || !v || !sumsq || n < 1) return fail("otb_adam_step", "bad arguments");
    RET("otb_adam_step", adam_launch(ST(stream), p, g, m, v, (size_t)n, sumsq, max_norm, lr, beta1, beta2, eps, weight_decay, step));
}

int otb_adam_step_sched(float* p, const float* g, float* m, float* v, long long n, const float* sumsq, float max_norm,
                        float base_lr, float model_size, float warmup_steps, float factor, float beta1, float beta2, float eps,
                        float weight_decay, int32_t* counters, float* hyper, void* stream) {
    if (!p || !g || !m || !v || !sumsq || !counters || !hyper || n < 1) return fail("otb_adam_step_sched", "bad arguments");
    RET("otb_adam_step_sched", adam_sched_launch(ST(stream), p, g, m, v, (size_t)n, sumsq, max_norm, base_lr, model_size, warmup_steps,
                                                 factor, beta1, beta2, eps, weight_decay, counters, hyper));
}

int otb_fbank(const float* wave, int ld_wave, const int32_t* n_samples, int B, const float* window, const float* bank,
              const int32_t* bank_range, float* out, int Tmax, int F, int frame_len, int frame_shift, float preemph, void* stream) {
    if (!wave || !n_samples || !window || !bank || !bank_range || !out) return fail("otb_fbank", "null operand");
    RET("otb_fbank", fbank_launch(ST(stream), wave, ld_wave, n_samples, B, window, bank, bank_range, out, Tmax, F, frame_len, frame_shift, preemph));
}

int otb_utt_cmvn(float* x, int B, int Tmax, int F, const int32_t* n_frames, const float* gmean, const float* gstd, void* stream) {
    if (!x || !n_frames) return fail("otb_utt_cmvn", "null operand");
    RET("otb_utt_cmvn", utt_cmvn_launch(ST(stream), x, B, Tmax, F, n_frames, gmean, gstd));
}

int otb_ctc_loss(const float* logp, int ldl, int B, int T, int V, const int32_t* in_len, const int64_t* targets, int ldt,
                 const int32_t* tgt_len, int max_tgt, int blank, float* nll, float* loss, float* ws, void* dlogits_bf16, int ldd,
                 float grad_scale, void* stream) {
    if (!logp || !in_len || !targets || !tgt_len || !nll || !loss || !ws) return fail("otb_ctc_loss", "null operand");
    if (ldl < V || (dlogits_bf16 && ldd < V)) return fail("otb_ctc_loss", "row pitch < V");
    RET("otb_ctc_loss", ctc_launch(ST(stream), logp, ldl, B, T, V, in_len, reinterpret_cast<const long long*>(targets), ldt, tgt_len, max_tgt,
                                   blank, nll, loss, ws, reinterpret_cast<bf16*>(dlogits_bf16), ldd, grad_scale));
}

int otb_conv_im2col(const void* h1, void* col, int B, int T, int F, int C1, void* stream) {
    int T1, F1, T2, F2;
    if (otb_conv_geometry(T, F, &T1, &F1, &T2, &F2)) return 1;
    if (!h1 || !col) return fail("otb_conv_im2col", "null operand");
    RET("otb_conv_im2col", im2col_s2_launch(ST(stream), reinterpret_cast<const bf16*>(h1), reinterpret_cast<bf16*>(col), B, T2, F2, C1));
}

int otb_conv_col2im_relu(const void* dcol, const void* h1, void* dpre1, int B, int T, int F, int C1, void* stream) {
    int T1, F1, T2, F2;
    if (otb_conv_geometry(T, F, &T1, &F1, &T2, &F2)) return 1;
    if (!dcol || !h1 || !dpre1) return fail("otb_conv_col2im_relu", "null operand");
    RET("otb_conv_col2im_relu", col2im_s2_relu_launch(ST(stream), reinterpret_cast<const bf16*>(dcol), reinterpret_cast<const bf16*>(h1),
                                                      reinterpret_cast<bf16*>(dpre1), B, T1, F1, T2, F2, C1));
}

int otb_conv1_wgrad(const void* dpre1, const float* x, float* out, int B, int T, int F, int C1, void* stream) {
    int T1, F1, T2, F2;
    if (otb_conv_geometry(T, F, &T1, &F1, &T2, &F2)) return 1;
    if (!dpre1 || !x || !out) return fail("otb_conv1_wgrad", "null operand");
    RET("otb_conv1_wgrad", conv1_wgrad_launch(ST(stream), reinterpret_cast<const bf16*>(dpre1), x, out, B, T, F, T1, F1, T2, F2, C1));
}

int otb_spec_augment(float* x, const int32_t* bands, int B, int T, int F, int n_freq, int n_time, void* stream) {
    if (!x || !bands || B < 1 || T < 1 || F < 1 || n_freq < 0 || n_time < 0) return fail("otb_spec_augment", "bad arguments");
    RET("otb_spec_augment", spec_augment_launch(ST(stream), x, bands, B, T, F, n_freq, n_time));
}

}  // extern "C"
