"""torch.Tensor-level wrappers around the C ABI (include/otb200.h).

PyTorch is plumbing here: it owns device memory and the current CUDA stream; all compute is in
libotb200.so.  Every wrapper launches on ``torch.cuda.current_stream()`` so the calls can be
captured into a CUDA graph (recognize.BeamDecoder captures a decode step, train.FusedTrainer a training micro-step).
"""
import ctypes
import math

import torch

from . import _lib
from ._lib import check

EPI_BIAS, EPI_RELU, EPI_GLU, EPI_TABLE, EPI_RESID, EPI_RESID_LN, EPI_SWISH, EPI_GELU, EPI_TANH = range(9)
ACT_EPILOGUE = {'relu': EPI_RELU, 'glu': EPI_GLU, 'swish': EPI_SWISH, 'gelu': EPI_GELU, 'tanh': EPI_TANH}
BF16 = torch.bfloat16


# ---- instrumentation (bench.py): kernel-launch counter and optional per-launch CUDA-event timing ----
COUNTERS = {'launches': 0}
PROFILE = None          # set to a list to collect (kind, algorithmic_flops, start_event, end_event) per GEMM launch


def _count(n=1):
    COUNTERS['launches'] += n


class _Timed:
    """Record CUDA events around one launch on the current stream when PROFILE is enabled."""

    def __init__(self, kind, flops, tag=None):
        self.kind, self.flops, self.tag = kind, flops, tag

    def __enter__(self):
        if PROFILE is not None and not torch.cuda.is_current_stream_capturing():
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        else:
            self.e0 = None

    def __exit__(self, *exc):
        if self.e0 is not None:
            self.e1.record()
            PROFILE.append((self.kind, self.flops, self.e0, self.e1, self.tag))


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _need(t, dtype, name):
    if not t.is_cuda:
        raise RuntimeError(f'{name} must be a CUDA tensor: the B200 hot path has no CPU fallback')
    if t.dtype != dtype:
        raise TypeError(f'{name} must be {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise ValueError(f'{name} must be contiguous')
    return t


def set_decode_barrier(kind):
    """'cluster', 'software' or 'default': group barrier of the persistent decode kernel (otb_set_decode_barrier)."""
    check(_lib.lib().otb_set_decode_barrier({'default': -1, 'software': 0, 'cluster': 1}[kind]), 'otb_set_decode_barrier')


def set_tile_policy(policy):
    """'latency' (default) or 'throughput': tiling of the small decode-step GEMMs (otb_set_tile_policy).  Takes effect for
    launches / graph captures made afterwards."""
    check(_lib.lib().otb_set_tile_policy({'latency': 0, 'throughput': 1}[policy]), 'otb_set_tile_policy')


def num_sms():
    return int(_lib.lib().otb_num_sms())


def conv_geometry(T, F):
    t1, f1, t2, f2 = (ctypes.c_int() for _ in range(4))
    check(_lib.lib().otb_conv_geometry(T, F, t1, f1, t2, f2), 'otb_conv_geometry')
    return t1.value, f1.value, t2.value, f2.value


def conv1_relu(x, w, bias, out=None):
    """x f32 [B,T,F]; w f32 [C1,1,3,3] -> bf16 NHWC [B, 2*(T2+1), 2*F2, C1]."""
    _need(x, torch.float32, 'x'); _need(w, torch.float32, 'w'); _need(bias, torch.float32, 'bias')
    B, T, F = x.shape
    C1 = w.shape[0]
    _, _, T2, F2 = conv_geometry(T, F)
    if out is None:
        out = torch.empty(B, 2 * (T2 + 1), 2 * F2, C1, dtype=BF16, device=x.device)
    check(_lib.lib().otb_conv1_relu(_p(x), _p(w), _p(bias), _p(out), B, T, F, C1, _stream()), 'otb_conv1_relu')
    _count()
    return out


def conv2_relu(h1, w, bias, B, T, F, out=None):
    """h1 = conv1 buffer; w bf16 [C2, 9*C1] (kh,kw,c order) -> bf16 [B*T2, F2*C2] (feature = f*C2 + c)."""
    _need(h1, BF16, 'h1'); _need(w, BF16, 'w'); _need(bias, torch.float32, 'bias')
    C2, K = w.shape
    C1 = K // 9
    _, _, T2, F2 = conv_geometry(T, F)
    if out is None:
        out = torch.empty(B * T2, F2 * C2, dtype=BF16, device=h1.device)
    with _Timed('conv2_gemm', 2.0 * B * T2 * F2 * C2 * K):
        check(_lib.lib().otb_conv2_relu(_p(h1), _p(w), _p(bias), _p(out), B, T, F, C1, C2, _stream()),
              'otb_conv2_relu')
    _count()
    return out


def linear(a, w, bias=None, epilogue=EPI_BIAS, out=None, out_f32=False, resid=None, gamma=None, beta=None,
           eps=1e-5, alpha=1.0, table=None, period=0, row_len=None, row_period=0, n_out=None):
    """out[M,N] = epi(a[M,K] @ w[N(,2N),K]^T + bias).  a, w bf16 2-D, unit column stride (row-strided views
    such as one head's 64 columns of a wider matrix are fine: the TMA map takes the row pitch)."""
    for t, n in ((a, 'a'), (w, 'w')):
        if not t.is_cuda:
            raise RuntimeError(f'{n} must be a CUDA tensor: the B200 hot path has no CPU fallback')
        if t.dtype != BF16 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError(f'{n} must be a 2-D bf16 tensor with unit column stride')
    M, K = a.shape
    N = w.shape[0] // 2 if epilogue == EPI_GLU else w.shape[0]
    if w.shape[1] != K:
        raise ValueError(f'linear: K mismatch {w.shape} vs {a.shape}')
    if out is None:
        ldc = n_out if n_out is not None else N
        out = torch.empty(M, ldc, dtype=torch.float32 if out_f32 else BF16, device=a.device)
    ldc = out.stride(0)
    with _Timed('gemm', 2.0 * M * w.shape[0] * K, (epilogue, M, w.shape[0], K, out.dtype == torch.float32)):
        check(_lib.lib().otb_linear(_p(a), a.stride(0), _p(w), w.stride(0), _p(bias), _p(out), ldc, M, N, K, epilogue,
                                    1 if out.dtype == torch.float32 else 0, _p(resid),
                                    resid.stride(0) if resid is not None else 0, _p(gamma), _p(beta), eps, alpha,
                                    _p(table), period, _p(row_len), row_period, _stream()), 'otb_linear')
    _count()
    return out


def linear_dropout_resid(a, w, bias, resid, p, seed, site, alpha=1.0, out=None):
    """out = resid + alpha * dropout_p(a @ w^T + bias): training-mode residual connection (otb_linear_dropout_resid).
    seed: int32/uint32 device tensor [1] (read at run time), site: dropout site id."""
    for t, n in ((a, 'a'), (w, 'w'), (resid, 'resid')):
        if not t.is_cuda or t.dtype != BF16 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError(f'{n} must be a 2-D bf16 CUDA tensor with unit column stride')
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, dtype=BF16, device=a.device)
    check(_lib.lib().otb_linear_dropout_resid(_p(a), a.stride(0), _p(w), w.stride(0), _p(bias), _p(out), out.stride(0), M, N, K,
                                              _p(resid), resid.stride(0), alpha, float(p), _p(seed), int(site), _stream()),
          'otb_linear_dropout_resid')
    _count()
    return out


def dropout_bwd(dy, p, seed, site):
    """dy * keep / (1 - p) with the mask of dropout site `site` replayed from (seed, site)."""
    _need(dy, BF16, 'dy')
    M, N = dy.shape
    out = torch.empty_like(dy)
    check(_lib.lib().otb_dropout_bwd(_p(dy), dy.stride(0), _p(out), out.stride(0), None, M, N, float(p), _p(seed), int(site),
                                     _stream()), 'otb_dropout_bwd')
    _count()
    return out


def dropout_mask(M, N, p, seed, site):
    """u8 [M,N] keep mask of a dropout site (parity tests replay it in the oracle)."""
    mask = torch.empty(M, N, dtype=torch.uint8, device=seed.device)
    check(_lib.lib().otb_dropout_bwd(None, 0, None, 0, _p(mask), M, N, float(p), _p(seed), int(site), _stream()),
          'otb_dropout_bwd')
    _count()
    return mask


def attention(q, k, v, B, H, Tq, Tk, kv_len=None, causal=False, q_col0=0, k_col0=0, v_col0=0, out=None, bd=None,
              resid=None, head_dim=64):
    """q/k/v: bf16 2-D matrices (may be the same [M,3d] buffer with different column offsets); head h reads columns
    *_col0 + head_dim*h (head_dim 64 or 96)."""
    for t, n in ((q, 'q'), (k, 'k'), (v, 'v')):
        _need(t, BF16, n)
    d = H * head_dim
    if out is None:
        out = torch.empty(B * Tq, d, dtype=BF16, device=q.device)
    if kv_len is not None:
        _need(kv_len, torch.int32, 'kv_len')
    check(_lib.lib().otb_attention_hd(_p(q), q.stride(0), q.shape[0], _p(k), k.stride(0), k.shape[0], _p(v), v.stride(0),
                                      _p(out), out.stride(0), B, H, head_dim, Tq, Tk, _p(kv_len), 1 if causal else 0, q_col0,
                                      k_col0, v_col0, _p(bd), bd.shape[-1] if bd is not None else 0, _p(resid),
                                      resid.stride(0) if resid is not None else 0, _stream()),
          'otb_attention')
    _count()
    return out


def dwconv_swish(x, w, b, B, T, out=None):
    """depthwise conv over time + folded BatchNorm + swish; x bf16 [B*T, d], w f32 [k, d], b f32 [d]."""
    _need(x, BF16, 'x'); _need(w, torch.float32, 'w'); _need(b, torch.float32, 'b')
    d = x.shape[1]
    if out is None:
        out = torch.empty_like(x)
    check(_lib.lib().otb_dwconv_swish(_p(x), _p(w), _p(b), _p(out), B, T, d, w.shape[0], _stream()),
          'otb_dwconv_swish')
    _count()
    return out


def layernorm(x, g1, b1, g2=None, b2=None, eps=1e-5, out=None, out_f32=False):
    _need(x, BF16, 'x')
    M, N = x.shape
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32 if out_f32 else BF16, device=x.device)
    check(_lib.lib().otb_layernorm(_p(x), x.stride(0), _p(out), out.stride(0), 1 if out.dtype == torch.float32 else 0,
                                   _p(g1), _p(b1), _p(g2), _p(b2), eps, M, N, _stream()), 'otb_layernorm')
    _count()
    return out


def scale_add_table(x, alpha=1.0, table=None, period=1, out=None):
    """bf16 out = x * alpha + table[row % period]; x f32 or bf16 2-D."""
    M, N = x.shape
    if out is None:
        out = torch.empty(M, N, dtype=BF16, device=x.device)
    check(_lib.lib().otb_scale_add_table(_p(x), x.stride(0), 1 if x.dtype == torch.float32 else 0, _p(out),
                                         out.stride(0), alpha, _p(table), period, M, N, _stream()),
          'otb_scale_add_table')
    _count()
    return out


_TABLES = {}


def sinusoid_table(n_pos, d, first_pos=0, device=None):
    """Cached f32 [n_pos, d] sinusoid table (module/pos.py:30-42), computed once on the device."""
    device = torch.device(device if device is not None else torch.cuda.current_device())
    key = (n_pos, d, first_pos, device.index if device.index is not None else torch.cuda.current_device())
    t = _TABLES.get(key)
    if t is None:
        t = torch.empty(n_pos, d, dtype=torch.float32, device=device)
        check(_lib.lib().otb_sinusoid_table(_p(t), n_pos, d, first_pos, _stream()), 'otb_sinusoid_table')
        _count()
        _TABLES[key] = t
    return t


def embed_posenc(tok, emb, table, N, d, period=1, tok_stride=1, step_ptr=None, out=None):
    _need(emb, BF16, 'emb')
    if out is None:
        out = torch.empty(N, d, dtype=BF16, device=emb.device)
    check(_lib.lib().otb_embed_posenc(_p(tok), tok_stride, _p(emb), _p(table), _p(out), N, d, period, _p(step_ptr),
                                      emb.shape[0], _stream()), 'otb_embed_posenc')
    _count()
    return out


def log_softmax(x, V, out=None):
    _need(x, torch.float32, 'x')
    rows = x.shape[0]
    if out is None:
        out = torch.empty(rows, V, dtype=torch.float32, device=x.device)
    check(_lib.lib().otb_log_softmax(_p(x), x.stride(0), _p(out), out.stride(0), rows, V, _stream()),
          'otb_log_softmax')
    _count()
    return out


def logsoftmax_topk(logits, V, k, lm_logp=None, lm_weight=0.0, out_val=None, out_idx=None, out_logp=None):
    """Fused log-softmax (+ LM shallow fusion) + per-row top-k.  logits f32 [rows, ld]."""
    _need(logits, torch.float32, 'logits')
    rows = logits.shape[0]
    if out_val is None:
        out_val = torch.empty(rows, k, dtype=torch.float32, device=logits.device)
    if out_idx is None:
        out_idx = torch.empty(rows, k, dtype=torch.int32, device=logits.device)
    check(_lib.lib().otb_logsoftmax_topk(_p(logits), logits.stride(0), V, _p(lm_logp),
                                         lm_logp.stride(0) if lm_logp is not None else 0, lm_weight, k, rows,
                                         _p(out_val), _p(out_idx), _p(out_logp),
                                         out_logp.stride(0) if out_logp is not None else 0, _stream()),
          'otb_logsoftmax_topk')
    _count()
    return out_val, out_idx


def ls_cross_entropy(logits, targets, V, smoothing=0.1, pad_id=0, want_grad=False):
    """Label-smoothed CE (module/loss.py:21-48).  logits f32 [rows, ld]; targets i64 [rows].
    Returns (loss f32 scalar tensor, dlogits f32 [rows, V] or None)."""
    _need(logits, torch.float32, 'logits')
    rows = logits.shape[0]
    targets = targets.contiguous().view(-1)
    dev = logits.device
    tok = torch.empty(rows, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    nv = torch.empty(1, dtype=torch.int32, device=dev)
    dl = torch.empty(rows, V, dtype=torch.float32, device=dev) if want_grad else None
    check(_lib.lib().otb_ls_ce(_p(logits), logits.stride(0), _p(targets), rows, V, smoothing, pad_id, _p(tok), _p(loss),
                               _p(nv), _p(dl), V if want_grad else 0, _stream()), 'otb_ls_ce')
    _count(3)
    return loss[0], dl


def decode_self_attn(qkv, kc, vc, anc, step_ptr, N, H, Lmax, out=None, head_dim=64):
    if out is None:
        out = torch.empty(N, H * head_dim, dtype=BF16, device=qkv.device)
    check(_lib.lib().otb_decode_self_attn_hd(_p(qkv), _p(kc), _p(vc), _p(anc), _p(step_ptr), _p(out), N, H, head_dim, Lmax,
                                             _stream()), 'otb_decode_self_attn')
    _count()
    return out


class BeamState:
    """Device-resident beam-search state (otb_beam_state)."""

    def __init__(self, batch, beam, max_len, device):
        self.B, self.beam, self.Lmax = batch, beam, max_len
        self.N = N = batch * beam
        kw = dict(device=device)
        self.tok_hist = torch.zeros(max_len, N, dtype=torch.int32, **kw)
        self.par_hist = torch.zeros(max_len, N, dtype=torch.int32, **kw)
        self.last_tok = torch.ones(N, dtype=torch.int64, **kw)
        self.scores = torch.zeros(N, dtype=torch.float32, **kw)
        self.flag = torch.zeros(N, dtype=torch.uint8, **kw)
        self.anc = torch.zeros(2, N, max_len, dtype=torch.int32, **kw)
        self.ctrl = torch.zeros(4, dtype=torch.int32, **kw)
        self.c = _lib.BeamStateC(self.tok_hist.data_ptr(), self.par_hist.data_ptr(), self.last_tok.data_ptr(),
                                 self.scores.data_ptr(), self.flag.data_ptr(), self.anc.data_ptr(),
                                 self.ctrl.data_ptr(), N, beam, max_len)

    @property
    def step_ptr(self):
        return self.ctrl  # ctrl[0] is the step counter

    def init(self):
        check(_lib.lib().otb_beam_init(ctypes.byref(self.c), _stream()), 'otb_beam_init')
        _count()

    def step(self, logp, V, lm_logp=None, lm_weight=0.0, dbg_ktok=None, dbg_offs=None):
        _need(logp, torch.float32, 'logp')
        check(_lib.lib().otb_beam_step(_p(logp), logp.stride(0), V, _p(lm_logp),
                                       lm_logp.stride(0) if lm_logp is not None else 0, lm_weight,
                                       ctypes.byref(self.c), _p(dbg_ktok), _p(dbg_offs), _stream()), 'otb_beam_step')
        _count()

    def step_topk(self, topk_val, topk_idx, dbg_ktok=None, dbg_offs=None):
        check(_lib.lib().otb_beam_step_topk(_p(topk_val), _p(topk_idx), ctypes.byref(self.c), _p(dbg_ktok),
                                            _p(dbg_offs), _stream()), 'otb_beam_step_topk')
        _count()

    def reconstruct(self, steps):
        preds = torch.empty(self.N, steps + 1, dtype=torch.int64, device=self.scores.device)
        check(_lib.lib().otb_beam_reconstruct(ctypes.byref(self.c), _p(preds), steps + 1, steps, _stream()),
              'otb_beam_reconstruct')
        _count()
        return preds

    def finalize(self, penalty, lamda, nbest):
        k = min(nbest, self.beam)
        out_preds = torch.empty(self.B, k, self.Lmax, dtype=torch.int64, device=self.scores.device)
        out_scores = torch.empty(self.B, k, dtype=torch.float32, device=self.scores.device)
        check(_lib.lib().otb_beam_finalize(ctypes.byref(self.c), float(penalty), float(lamda), k, _p(out_preds),
                                           _p(out_scores), _stream()), 'otb_beam_finalize')
        _count()
        return out_preds, out_scores


def decode_persistent_workspace(N, n_layers, Lmax, B, beam, vocab, device):
    n = int(_lib.lib().otb_decode_persistent_workspace(N, n_layers, Lmax, B, beam, vocab))
    if n < 0:
        raise ValueError('otb_decode_persistent_workspace: bad geometry')
    return torch.zeros(n, dtype=torch.uint8, device=device)


def decode_persistent(model_c, kvx, mem_len, kc, vc, state, B, T, max_steps, workspace, dbg_logp=None, dbg_scores=None):
    """The whole beam-search decode loop in one persistent kernel (otb_decode_persistent, csrc/decode_group.cu)."""
    _need(kvx, BF16, 'kvx'); _need(kc, BF16, 'kc'); _need(vc, BF16, 'vc'); _need(mem_len, torch.int32, 'mem_len')
    check(_lib.lib().otb_decode_persistent(ctypes.byref(model_c), _p(kvx), _p(mem_len), _p(kc), _p(vc), ctypes.byref(state.c),
                                           B, T, max_steps, _p(workspace), workspace.numel(), _p(dbg_logp), _p(dbg_scores),
                                           _stream()), 'otb_decode_persistent')
    _count()


# ------------------------------------------------------------------------------------------------
# training step: backward kernels (include/otb200.h "Training step")
# ------------------------------------------------------------------------------------------------
def attention_train(q, k, v, B, H, Tq, Tk, kv_len=None, causal=False, q_col0=0, k_col0=0, v_col0=0, head_dim=64):
    """otb_attention + the per-row log-sum-exp the backward needs -> (out bf16 [B*Tq, H*head_dim], lse f32 [B,H,Tq]).
    (attention_bwd is 64-wide only.)"""
    for t, n in ((q, 'q'), (k, 'k'), (v, 'v')):
        _need(t, BF16, n)
    out = torch.empty(B * Tq, H * head_dim, dtype=BF16, device=q.device)
    lse = torch.empty(B, H, Tq, dtype=torch.float32, device=q.device)
    check(_lib.lib().otb_attention_lse_hd(_p(q), q.stride(0), q.shape[0], _p(k), k.stride(0), k.shape[0], _p(v), v.stride(0),
                                          _p(out), out.stride(0), B, H, head_dim, Tq, Tk, _p(kv_len), 1 if causal else 0, q_col0,
                                          k_col0, v_col0, None, 0, None, 0, _p(lse), _stream()), 'otb_attention_lse')
    _count()
    return out, lse


def attention_bwd(q, k, v, out, dout, lse, B, H, Tq, Tk, dq, dk, dv, kv_len=None, causal=False, q_col0=0, k_col0=0,
                  v_col0=0, dq_col0=0, dk_col0=0, dv_col0=0):
    """Gradients of otb_attention written into dq/dk/dv (bf16 matrices, column offsets d*_col0)."""
    for t, n in ((q, 'q'), (k, 'k'), (v, 'v'), (out, 'out'), (dout, 'dout'), (dq, 'dq'), (dk, 'dk'), (dv, 'dv')):
        if not t.is_cuda or t.dtype != BF16 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError(f'{n} must be a 2-D bf16 CUDA tensor with unit column stride (no CPU fallback)')
    dsum = torch.empty(B, H, Tq, dtype=torch.float32, device=q.device)
    check(_lib.lib().otb_attention_bwd(_p(q), q.stride(0), q.shape[0], _p(k), k.stride(0), k.shape[0], _p(v), v.stride(0),
                                       _p(out), out.stride(0), _p(dout), dout.stride(0), _p(lse), _p(dsum),
                                       _p(dq), dq.stride(0), dq_col0, _p(dk), dk.stride(0), dk_col0, _p(dv), dv.stride(0),
                                       dv_col0, B, H, Tq, Tk, _p(kv_len), 1 if causal else 0, q_col0, k_col0, v_col0,
                                       _stream()), 'otb_attention_bwd')
    _count(2)


def linear_wgrad(dy, x, out=None, accumulate=False):
    """dW f32 [N,K] (+)= dy[M,N]^T x[M,K]  (bf16 2-D, unit column stride)."""
    for t, n in ((dy, 'dy'), (x, 'x')):
        if not t.is_cuda or t.dtype != BF16 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError(f'{n} must be a 2-D bf16 CUDA tensor with unit column stride')
    M, N = dy.shape
    K = x.shape[1]
    if x.shape[0] != M:
        raise ValueError('linear_wgrad: row mismatch')
    if out is None:
        out = torch.empty(N, K, dtype=torch.float32, device=dy.device)
    with _Timed('wgrad', 2.0 * M * N * K, (M, N, K)):
        check(_lib.lib().otb_linear_wgrad(_p(dy), dy.stride(0), _p(x), x.stride(0), _p(out), out.stride(0), M, N, K,
                                          1 if accumulate else 0, _stream()), 'otb_linear_wgrad')
    _count(2)
    return out


def colsum(x, out=None, accumulate=False):
    M, N = x.shape
    if out is None:
        out = torch.empty(N, dtype=torch.float32, device=x.device)
    check(_lib.lib().otb_colsum(_p(x), x.stride(0), _p(out), M, N, 1 if accumulate else 0, _stream()), 'otb_colsum')
    _count()
    return out


def layernorm_bwd(dy, z, gamma, eps=1e-5, dgamma=None, dbeta=None, accumulate=False):
    """-> (dz bf16 [M,N], dgamma f32 [N], dbeta f32 [N]); with accumulate the given dgamma / dbeta are added to."""
    _need(dy, BF16, 'dy'); _need(z, BF16, 'z')
    M, N = z.shape
    dz = torch.empty(M, N, dtype=BF16, device=z.device)
    dg = dgamma if dgamma is not None else torch.empty(N, dtype=torch.float32, device=z.device)
    db = dbeta if dbeta is not None else torch.empty(N, dtype=torch.float32, device=z.device)
    check(_lib.lib().otb_layernorm_bwd(_p(dy), dy.stride(0), _p(z), z.stride(0), _p(gamma), _p(dz), dz.stride(0), _p(dg),
                                       _p(db), eps, M, N, 1 if accumulate else 0, _stream()), 'otb_layernorm_bwd')
    _count()
    return dz, dg, db


def glu_fwd(u):
    _need(u, BF16, 'u')
    M, F2 = u.shape
    h = torch.empty(M, F2 // 2, dtype=BF16, device=u.device)
    check(_lib.lib().otb_glu_fwd(_p(u), _p(h), M, F2 // 2, _stream()), 'otb_glu_fwd')
    _count()
    return h


def glu_bwd(dh, u):
    _need(u, BF16, 'u'); _need(dh, BF16, 'dh')
    M, F2 = u.shape
    du = torch.empty(M, F2, dtype=BF16, device=u.device)
    check(_lib.lib().otb_glu_bwd(_p(dh), _p(u), _p(du), M, F2 // 2, _stream()), 'otb_glu_bwd')
    _count()
    return du


def relu_bwd(dy, y, out=None):
    _need(dy, BF16, 'dy'); _need(y, BF16, 'y')
    if out is None:
        out = torch.empty_like(dy)
    check(_lib.lib().otb_relu_bwd(_p(dy), _p(y), _p(out), dy.numel(), _stream()), 'otb_relu_bwd')
    _count()
    return out


def embed_bwd(tok, dx, dE, scale):
    """dE[tok[n]] += scale * dx[n]   (dE f32 [V,d], accumulated in place)."""
    _need(dx, BF16, 'dx'); _need(dE, torch.float32, 'dE')
    tok = tok.contiguous().view(-1)
    check(_lib.lib().otb_embed_bwd(_p(tok), _p(dx), _p(dE), tok.numel(), dx.shape[1], dE.shape[0], scale, _stream()),
          'otb_embed_bwd')
    _count()


def ls_cross_entropy_train(logits, targets, V, smoothing=0.1, pad_id=0):
    """-> (loss f32 scalar tensor, dlogits bf16 [rows, ld] with ld = logits.stride(0); pad columns zero)."""
    _need(logits, torch.float32, 'logits')
    rows, ld = logits.shape[0], logits.stride(0)
    targets = targets.contiguous().view(-1)
    dev = logits.device
    tok = torch.empty(rows, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    nv = torch.empty(1, dtype=torch.int32, device=dev)
    dl = torch.empty(rows, ld, dtype=BF16, device=dev)
    check(_lib.lib().otb_ls_ce_train(_p(logits), ld, _p(targets), rows, V, smoothing, pad_id, _p(tok), _p(loss), _p(nv),
                                     _p(dl), ld, _stream()), 'otb_ls_ce_train')
    _count(3)
    return loss[0], dl


def sumsq(g, out, zero_first=True):
    check(_lib.lib().otb_sumsq(_p(g), g.numel(), _p(out), 1 if zero_first else 0, _stream()), 'otb_sumsq')
    _count()


def adam_step(p, g, m, v, sumsq_buf, max_norm, lr, betas, eps, weight_decay, step):
    for t, n in ((p, 'p'), (g, 'g'), (m, 'm'), (v, 'v')):
        _need(t, torch.float32, n)
    check(_lib.lib().otb_adam_step(_p(p), _p(g), _p(m), _p(v), p.numel(), _p(sumsq_buf), max_norm, lr, betas[0], betas[1],
                                   eps, weight_decay, step, _stream()), 'otb_adam_step')
    _count()


def adam_step_sched(p, g, m, v, sumsq_buf, max_norm, base_lr, model_size, warmup_steps, factor, betas, eps, weight_decay,
                    counters, hyper):
    """clip + Adam with the step counters / Noam schedule evaluated on the device (otb_adam_step_sched)."""
    for t, n in ((p, 'p'), (g, 'g'), (m, 'm'), (v, 'v'), (hyper, 'hyper')):
        _need(t, torch.float32, n)
    _need(counters, torch.int32, 'counters')
    check(_lib.lib().otb_adam_step_sched(_p(p), _p(g), _p(m), _p(v), p.numel(), _p(sumsq_buf), max_norm, base_lr,
                                         float(model_size), float(warmup_steps or 0), factor, betas[0], betas[1], eps,
                                         weight_decay, _p(counters), _p(hyper), _stream()), 'otb_adam_step_sched')
    _count(2)


def ctc_loss(logits, B, T, V, in_len, targets, tgt_len, blank=0, want_grad=False, grad_scale=1.0):
    """nn.CTCLoss(blank, 'mean', zero_infinity=True) on logits f32 [B*T, ld] (model/ctc.py:48-52).
    -> (loss 0-d, nll f32 [B], dlogits bf16 [B*T, ld] or None)."""
    _need(logits, torch.float32, 'logits'); _need(in_len, torch.int32, 'in_len'); _need(tgt_len, torch.int32, 'tgt_len')
    targets = targets.contiguous()
    dev = logits.device
    ld = logits.stride(0)
    logp = torch.empty(B * T, ld, dtype=torch.float32, device=dev)
    check(_lib.lib().otb_log_softmax(_p(logits), ld, _p(logp), ld, B * T, V, _stream()), 'otb_log_softmax')
    max_tgt = targets.shape[1]
    nll = torch.empty(B, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = torch.empty(B, T, 2 * max_tgt + 1, dtype=torch.float32, device=dev)
    dl = torch.empty(B * T, ld, dtype=BF16, device=dev) if want_grad else None
    check(_lib.lib().otb_ctc_loss(_p(logp), ld, B, T, V, _p(in_len), _p(targets), targets.stride(0), _p(tgt_len), max_tgt, blank,
                                  _p(nll), _p(loss), _p(ws), _p(dl), ld if want_grad else 0, float(grad_scale), _stream()),
          'otb_ctc_loss')
    _count(4 if want_grad else 3)
    return loss[0], nll, dl


def conv_im2col(h1, B, T, F, C1):
    _, _, T2, F2 = conv_geometry(T, F)
    col = torch.empty(B * T2 * F2, 9 * C1, dtype=BF16, device=h1.device)
    check(_lib.lib().otb_conv_im2col(_p(h1), _p(col), B, T, F, C1, _stream()), 'otb_conv_im2col')
    _count()
    return col


def conv_col2im_relu(dcol, h1, B, T, F, C1):
    dpre1 = torch.empty_like(h1)
    check(_lib.lib().otb_conv_col2im_relu(_p(dcol), _p(h1), _p(dpre1), B, T, F, C1, _stream()), 'otb_conv_col2im_relu')
    _count()
    return dpre1


def conv1_wgrad(dpre1, x, B, T, F, C1):
    out = torch.empty(C1, 10, dtype=torch.float32, device=x.device)
    check(_lib.lib().otb_conv1_wgrad(_p(dpre1), _p(x), _p(out), B, T, F, C1, _stream()), 'otb_conv1_wgrad')
    _count()
    return out

