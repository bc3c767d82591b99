"""Host-side mirror of the reference's nn.Module surface for the hot path.

Same class names, constructor kwargs (the YAML sub-dicts verbatim) and ``state_dict()`` key names /
shapes as the reference so existing checkpoints load unchanged (SURVEY.md 8b):

    ConvFrontEnd        <- otrans/frontend/conv.py:86-159
    TransformerEncoder  <- otrans/encoder/transformer.py:93-134
    TransformerDecoder  <- otrans/decoder/transformer.py:129-208

The nn.Linear / nn.LayerNorm / nn.Conv2d / nn.Embedding objects below are *parameter holders*
only (they give identical key names and default init); their ``forward`` is never called.  All
compute goes through ``ops`` -> libotb200.so (hand-written sm_100a kernels).  There is no CPU path:
calling a module with CPU tensors raises.

Numerics: GEMM operands / activations are bf16, accumulation fp32, LayerNorm / softmax statistics
fp32 (DESIGN.md "rounding points").  The module-level forward is the inference path; training goes through
``SpeechToText.forward`` in train mode -> train.py (hand-written backward).
"""
import math

import torch
import torch.nn as nn

from . import ops
from .ops import BF16, EPI_BIAS, EPI_GLU, EPI_RELU, EPI_RESID, EPI_RESID_LN, EPI_TABLE, ACT_EPILOGUE


def _lengths(mask):
    """bool [B,T] prefix mask -> int32 [B] lengths (masks are contiguous prefixes, SURVEY.md 8a)."""
    return mask.sum(dim=1).to(torch.int32).contiguous()


_PARAM_GENERATION = [0]


def bump_param_generation():
    """Invalidate every bf16 shadow copy: called after parameters were updated outside torch's version tracking
    (the fused Adam kernel of train.FusedTrainer writes the flat fp32 buffer directly)."""
    _PARAM_GENERATION[0] += 1


class _Packed:
    """bf16 shadow copies of fp32 master parameters, refreshed when any parameter changes
    (load_state_dict / optimizer steps bump ``Tensor._version``)."""

    def __init__(self, module, builder):
        self._module, self._builder, self._sig, self._val = module, builder, None, None

    def get(self):
        sig = (_PARAM_GENERATION[0],) + tuple((p.data_ptr(), p._version) for p in self._module.parameters())
        if self._val is None or sig != self._sig:
            with torch.no_grad():
                self._val = self._builder()
            self._sig = sig
        return self._val


def _w(lin):
    return lin.weight.detach().to(BF16).contiguous()


def _b(lin):
    return lin.bias.detach().float().contiguous() if lin.bias is not None else None


def _ln(norm):
    return norm.weight.detach().float().contiguous(), norm.bias.detach().float().contiguous()


HEAD_DIMS = (64, 96)   # head widths the sm_100a attention kernels are built for


def head_dim_of(n_heads, d_model):
    """d_model // n_heads when it is a head width the attention kernels support, else NotImplementedError."""
    if n_heads < 1 or d_model % n_heads or d_model // n_heads not in HEAD_DIMS:
        raise NotImplementedError(f'the sm_100a attention kernels support d_k = d_model / n_heads in {HEAD_DIMS}; '
                                  f'got d_model {d_model}, n_heads {n_heads}')
    return d_model // n_heads


def _no_train(module):
    if module.training and torch.is_grad_enabled():
        raise NotImplementedError('module-level forward is the inference path: call under model.eval() / torch.no_grad(); '
                                  'training runs through SpeechToText.forward (opentransformer_b200.train)')


# ------------------------------------------------------------------------------------------------
# front end
# ------------------------------------------------------------------------------------------------
class Conv2dLayer(nn.Module):
    """Parameter holder with the reference's key names (frontend/conv.py:15-48)."""

    def __init__(self, input_size, in_channel, out_channel, kernel_size, stride, dropout=0.1, batch_norm=False,
                 residual=False, act_func_type='relu'):
        super().__init__()
        ks = kernel_size if isinstance(kernel_size, (list, tuple)) else [kernel_size, kernel_size]
        if list(ks) != [3, 3] or stride != 2 or batch_norm or residual or act_func_type != 'relu':
            raise NotImplementedError('B200 ConvFrontEnd supports the shipped configuration only: '
                                      '3x3 kernels, stride 2, relu, no batch_norm / residual')
        self.conv_layer = nn.Conv2d(in_channel, out_channel, (3, 3), stride=2, padding=(0, 1))
        self.output_size = (input_size + 2 - 3) // 2 + 1
        self.out_channel = out_channel


class ConvFrontEnd(nn.Module):
    """forward(x f32 [B,T,F], mask bool [B,T]) -> (f32 [B,T',D], bool [B,T'])   (frontend/conv.py:131-153)."""

    def __init__(self, input_size, output_size, in_channel=1, mid_channel=32, out_channel=128,
                 kernel_size=[[3, 3], [3, 3]], stride=[2, 2], dropout=0.0, act_func_type='relu',
                 front_end_layer_norm=False):
        super().__init__()
        assert isinstance(kernel_size, list) and len(kernel_size) == 2
        assert isinstance(stride, list) and len(stride) == 2
        if in_channel != 1:
            raise NotImplementedError('in_channel must be 1 (log-fbank input)')
        if dropout:
            raise NotImplementedError('frontend dropout > 0 is a training feature (round 2)')
        self.input_size, self.output_size = input_size, output_size
        self.front_end_layer_norm = front_end_layer_norm
        self.conv1 = Conv2dLayer(input_size, in_channel, mid_channel, kernel_size[0], stride[0], dropout)
        self.conv2 = Conv2dLayer(self.conv1.output_size, mid_channel, out_channel, kernel_size[1], stride[1], dropout)
        self.conv_output_size = self.conv2.output_size * out_channel
        self.output_layer = nn.Linear(self.conv_output_size, output_size)
        if front_end_layer_norm:
            self.layer_norm = nn.LayerNorm(output_size)
        self._pack = _Packed(self, self._build_pack)

    def _build_pack(self):
        c1 = self.conv1.conv_layer
        c2 = self.conv2.conv_layer
        C1, C2 = c1.out_channels, c2.out_channels
        F2 = self.conv2.output_size
        C1p = (C1 + 63) // 64 * 64          # one 128-byte tap per k-block needs 64-channel multiples
        w1 = torch.zeros(C1p, 1, 3, 3, device=c1.weight.device)
        w1[:C1] = c1.weight.detach().float()
        b1 = torch.zeros(C1p, device=c1.weight.device)
        b1[:C1] = c1.bias.detach().float()
        w2 = torch.zeros(C2, 3, 3, C1p, device=c1.weight.device)
        w2[..., :C1] = c2.weight.detach().float().permute(0, 2, 3, 1)   # [C2,kh,kw,C1]: k = (kh*3+kw)*C1 + c
        # reference feature index is c*F2 + f (conv.py:145); conv2 kernel emits f*C2 + c -> permute columns once
        wo = self.output_layer.weight.detach().float().view(self.output_size, C2, F2).permute(0, 2, 1)
        pk = {'w1': w1.contiguous(), 'b1': b1.contiguous(), 'C1p': C1p,
              'w2': w2.reshape(C2, 9 * C1p).to(BF16).contiguous(), 'b2': c2.bias.detach().float().contiguous(),
              'wo': wo.reshape(self.output_size, F2 * C2).to(BF16).contiguous(), 'bo': _b(self.output_layer)}
        if self.front_end_layer_norm:
            pk['ln'] = _ln(self.layer_norm)
        return pk

    def output_mask(self, mask):
        # Conv2dLayer.return_output_mask twice (frontend/conv.py:78-83): mask[:, 1::2][:, :t]
        _, _, t2, _ = ops.conv_geometry(mask.shape[1], self.input_size)
        t1 = (mask.shape[1] - 3) // 2 + 1
        m = mask[:, 1::2][:, :t1]
        return m[:, 1::2][:, :t2]

    def forward_bf16(self, x, posenc_scale=None, posenc_table=None):
        """x f32 [B,T,F] -> bf16 [B*T', D].  When posenc_* are given, x*scale+PE is fused into the Linear
        epilogue (pos.py:56) so the encoder can skip its own positional-encoding pass."""
        _no_train(self)
        pk = self._pack.get()
        B, T, F = x.shape
        if F != self.input_size:
            raise ValueError(f'expected {self.input_size} features, got {F}')
        x = x.contiguous().float()
        _, _, T2, F2 = ops.conv_geometry(T, F)
        h1 = ops.conv1_relu(x, pk['w1'], pk['b1'])
        h2 = ops.conv2_relu(h1, pk['w2'], pk['b2'], B, T, F)
        if posenc_table is not None and not self.front_end_layer_norm:
            y = ops.linear(h2, pk['wo'], pk['bo'], EPI_TABLE, alpha=posenc_scale, table=posenc_table, period=T2)
        else:
            y = ops.linear(h2, pk['wo'], pk['bo'], EPI_BIAS)
            if self.front_end_layer_norm:
                y = ops.layernorm(y, *pk['ln'])
            if posenc_table is not None:
                y = ops.scale_add_table(y, posenc_scale, posenc_table, T2)
        return y, T2

    def forward(self, x, mask):
        y, T2 = self.forward_bf16(x)
        return y.float().view(x.shape[0], T2, self.output_size), self.output_mask(mask)

    def inference(self, x, mask, cache):
        y, m = self.forward(x, mask)
        return y, m, cache


# ------------------------------------------------------------------------------------------------
# parameter holders shared by encoder / decoder layers
# ------------------------------------------------------------------------------------------------
class MultiHeadedSelfAttention(nn.Module):
    """Keys: qvk_proj.{weight,bias} [3d,d] (split order Q,K,V -- attention.py:73), output_proj.*"""

    def __init__(self, n_heads, d_model, dropout_rate=0.0, share_qvk_proj=False):
        super().__init__()
        if share_qvk_proj:
            raise NotImplementedError('share_qvk_proj')
        self.head_dim = head_dim_of(n_heads, d_model)
        self.qvk_proj = nn.Linear(d_model, d_model * 3)
        self.output_proj = nn.Linear(d_model, d_model)


class MultiHeadedCrossAttention(nn.Module):
    """Keys: q_proj.*, vk_proj.* [2d,mem] (split order K,V -- attention.py:134), output_proj.*"""

    def __init__(self, n_heads, d_model, memory_dim, dropout_rate=0.0, share_vk_proj=False):
        super().__init__()
        if share_vk_proj:
            raise NotImplementedError('share_vk_proj')
        self.head_dim = head_dim_of(n_heads, d_model)
        self.q_proj = nn.Linear(d_model, d_model)
        self.vk_proj = nn.Linear(memory_dim, d_model * 2)
        self.output_proj = nn.Linear(d_model, d_model)


class PositionwiseFeedForward(nn.Module):
    """Keys: w_1.* [d_ff or 2*d_ff, d], w_2.* [d, d_ff]   (module/ffn.py:24-41)"""

    def __init__(self, d_model, d_ff, dropout, activation='relu'):
        super().__init__()
        assert activation in ['relu', 'gelu', 'glu', 'tanh', 'swish']
        self.activation = activation
        self.w_1 = nn.Linear(d_model, d_ff * 2 if activation == 'glu' else d_ff)
        self.w_2 = nn.Linear(d_ff, d_model)


class PositionalEncoding(nn.Module):
    """module/pos.py:11-28.  Quirk kept (SURVEY.md 8a): callers pass pos_dropout into the
    ``scale_learnable`` slot, so a non-zero pos_dropout creates ``alpha`` and switches to x + alpha*PE."""

    def __init__(self, emb_dim, scale_learnable=False, dropout=0.0):
        super().__init__()
        self.emb_dim = emb_dim
        self.xscale = math.sqrt(emb_dim)
        self.scale_learnable = bool(scale_learnable)
        if self.scale_learnable:
            self.alpha = nn.Parameter(torch.tensor(1.0))

    def scale_and_table(self, n_pos, device):
        table = ops.sinusoid_table(n_pos, self.emb_dim, 0, device)
        if self.scale_learnable:
            return 1.0, table * self.alpha.detach().float()
        return self.xscale, table


def _ffn(x, pk, resid, ln=None, alpha=1.0):
    """w_2(act(w_1(x))) with the residual (and post-LayerNorm) fused into the second GEMM."""
    h = ops.linear(x, pk['w1'], pk['b1'], pk['act'])
    if ln is not None and pk['w2'].shape[0] in (64, 128, 256):
        return ops.linear(h, pk['w2'], pk['b2'], EPI_RESID_LN, resid=resid, gamma=ln[0], beta=ln[1])
    y = ops.linear(h, pk['w2'], pk['b2'], EPI_RESID, resid=resid, alpha=alpha)
    return ops.layernorm(y, *ln) if ln is not None else y


def _proj_resid_ln(ctx, w, b, resid, ln):
    """output_proj + residual (+ post-LayerNorm) in one GEMM when the row fits one tile."""
    if ln is not None and w.shape[0] in (64, 128, 256):
        return ops.linear(ctx, w, b, EPI_RESID_LN, resid=resid, gamma=ln[0], beta=ln[1])
    y = ops.linear(ctx, w, b, EPI_RESID, resid=resid)
    return ops.layernorm(y, *ln) if ln is not None else y


def _ffn_pack(ff):
    return {'w1': _w(ff.w_1), 'b1': _b(ff.w_1), 'w2': _w(ff.w_2), 'b2': _b(ff.w_2),
            'act': ACT_EPILOGUE[ff.activation]}


# ------------------------------------------------------------------------------------------------
# encoder
# ------------------------------------------------------------------------------------------------
class TransformerEncoderLayer(nn.Module):
    def __init__(self, n_heads, d_model, d_ff, slf_attn_dropout, ffn_dropout, residual_dropout,
                 normalize_before=False, concat_after=False, relative_positional=False, activation='relu'):
        super().__init__()
        if concat_after:
            raise NotImplementedError('concat_after is not used by any shipped config')
        self.n_heads = n_heads
        self.normalize_before = normalize_before
        self.relative_positional = relative_positional
        # dropout is a training-time op (encoder/transformer.py:32-33,54,61); inference ignores it, train.py checks it
        self.dropout_rates = {'slf_attn_dropout': slf_attn_dropout, 'ffn_dropout': ffn_dropout,
                              'residual_dropout': residual_dropout}
        if relative_positional:     # encoder/transformer.py:23-24: Transformer-XL style attention, NO output projection (SURVEY 8a quirk)
            self.slf_attn = MultiHeadedSelfAttentionWithRelPos(n_heads, d_model, slf_attn_dropout)
        else:
            self.slf_attn = MultiHeadedSelfAttention(n_heads, d_model, slf_attn_dropout)
        self.feed_forward = PositionwiseFeedForward(d_model, d_ff, ffn_dropout, activation)
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)

    def pack(self):
        a = self.slf_attn
        pk = {'ffn': _ffn_pack(self.feed_forward), 'ln1': _ln(self.norm1), 'ln2': _ln(self.norm2)}
        if self.relative_positional:
            pk['rel'] = a.pack()
        else:
            pk.update({'wqkv': _w(a.qvk_proj), 'bqkv': _b(a.qvk_proj), 'wo': _w(a.output_proj), 'bo': _b(a.output_proj)})
        return pk

    def run(self, x, pk, B, T, lengths, causal=False, pos_bf16=None):
        """x bf16 [B*T, d] -> bf16 [B*T, d]   (encoder/transformer.py:41-65); causal=True is the tril mask the
        Transformer LM feeds to the same layer (model/lm.py:14-18,148-151)."""
        d, H = x.shape[1], self.n_heads
        if self.normalize_before:
            x = ops.layernorm(x, *pk['ln1'])          # residual is taken AFTER the norm (transformer.py:42-44)
        if self.relative_positional:
            if causal:
                raise NotImplementedError('causal rel-pos attention')
            x = self.slf_attn.run(x, x, pk['rel'], B, T, lengths, pos_bf16)       # x + attention (no output projection)
            if not self.normalize_before:
                x = ops.layernorm(x, *pk['ln1'])
            if self.normalize_before:
                x = ops.layernorm(x, *pk['ln2'])
            return _ffn(x, pk['ffn'], x, None if self.normalize_before else pk['ln2'])
        qkv = ops.linear(x, pk['wqkv'], pk['bqkv'])
        ctx = ops.attention(qkv, qkv, qkv, B, H, T, T, kv_len=lengths, causal=causal, q_col0=0, k_col0=d,
                            v_col0=2 * d, head_dim=self.slf_attn.head_dim)
        x = _proj_resid_ln(ctx, pk['wo'], pk['bo'], x, None if self.normalize_before else pk['ln1'])
        if self.normalize_before:
            x = ops.layernorm(x, *pk['ln2'])
        return _ffn(x, pk['ffn'], x, None if self.normalize_before else pk['ln2'])


class TransformerEncoder(nn.Module):
    """forward(inputs f32 [B,T,D], mask bool [B,T]) -> (f32 [B,T,D], mask, attn_weights)

    ``attn_weights`` maps 'enc_block_i' -> {'slf_attn_weights': None}: the reference materialises and
    returns [B,h,T,T] weights that no caller reads (SURVEY.md 8a row 5); the fused kernel never forms them.
    """

    def __init__(self, d_model=256, n_heads=4, d_ff=2048, n_blocks=6, pos_dropout=0.0, slf_attn_dropout=0.0,
                 ffn_dropout=0.0, residual_dropout=0.1, normalize_before=False, concat_after=False,
                 relative_positional=False, activation='relu'):
        super().__init__()
        self.d_model = d_model
        self.normalize_before = normalize_before
        self.relative_positional = relative_positional
        self.pos_emb = PositionalEncoding(d_model, pos_dropout)
        self.blocks = nn.ModuleList([
            TransformerEncoderLayer(n_heads, d_model, d_ff, slf_attn_dropout, ffn_dropout, residual_dropout,
                                    normalize_before, concat_after, relative_positional, activation)
            for _ in range(n_blocks)])
        if normalize_before:
            self.norm = nn.LayerNorm(d_model)
        self._pack = _Packed(self, lambda: {'blocks': [b.pack() for b in self.blocks],
                                            'norm': _ln(self.norm) if normalize_before else None})
        self._pos_cache = {}

    def _rel_pos(self, T, device):
        key = (T, device.index)
        p = self._pos_cache.get(key)
        if p is None:   # PE[-(T-1) .. T-1] (encoder/transformer.py:117-119), bf16 GEMM operand of pos_proj
            p = ops.scale_add_table(ops.sinusoid_table(2 * T - 1, self.d_model, -(T - 1), device))
            self._pos_cache[key] = p
        return p

    def forward_bf16(self, x, B, T, lengths):
        """x bf16 [B*T, d] with the positional encoding already applied (abs-pos) / the raw front-end output (rel-pos)."""
        _no_train(self)
        pk = self._pack.get()
        pos = self._rel_pos(T, x.device) if self.relative_positional else None
        for blk, bpk in zip(self.blocks, pk['blocks']):
            x = blk.run(x, bpk, B, T, lengths, pos_bf16=pos)
        if self.normalize_before:
            x = ops.layernorm(x, *pk['norm'])
        return x

    def fuse_abs_posenc(self):
        """True when x*sqrt(d)+PE may be fused into the front end's Linear epilogue."""
        return not self.relative_positional

    def apply_posenc_bf16(self, x, B, T):
        if self.relative_positional:       # enc_output = inputs (encoder/transformer.py:116): no x*sqrt(d)+PE
            return x if x.dtype == BF16 else ops.scale_add_table(x)
        scale, table = self.pos_emb.scale_and_table(T, x.device)
        return ops.scale_add_table(x, scale, table, T)

    def forward(self, inputs, mask):
        B, T, D = inputs.shape
        x = self.apply_posenc_bf16(inputs.contiguous().view(B * T, D), B, T)
        y = self.forward_bf16(x, B, T, _lengths(mask))
        attn = {'enc_block_%d' % i: {'slf_attn_weights': None} for i in range(len(self.blocks))}
        return y.float().view(B, T, D), mask, attn


# ------------------------------------------------------------------------------------------------
# Conformer encoder  (otrans/encoder/conformer.py, otrans/module/conformer.py, attention.py:176-257)
# ------------------------------------------------------------------------------------------------
class MultiHeadedSelfAttentionWithRelPos(nn.Module):
    """Keys: qvk_proj.*, pos_proj.weight, posu, posv  (attention.py:176-194).  Quirk kept (SURVEY.md 8a): the
    reference passes dropout_rate into the enable_output_proj slot, so with the shipped slf_attn_dropout 0.0
    there is NO output projection; a non-zero rate makes the reference itself crash."""

    def __init__(self, n_heads, d_model, dropout_rate=0.0, skip_term_b=False, share_qvk_proj=False):
        super().__init__()
        if dropout_rate or skip_term_b or share_qvk_proj:
            raise NotImplementedError('rel-pos attention: dropout / skip_term_b / share_qvk_proj')
        self.head_dim = head_dim_of(n_heads, d_model)
        self.nheads, self.d_model = n_heads, d_model
        self.qvk_proj = nn.Linear(d_model, d_model * 3)
        self.pos_proj = nn.Linear(d_model, d_model, bias=False)
        self.posu = nn.Parameter(torch.Tensor(1, 1, n_heads, d_model // n_heads))
        self.posv = nn.Parameter(torch.Tensor(1, 1, n_heads, d_model // n_heads))
        torch.nn.init.xavier_normal_(self.posu)
        torch.nn.init.xavier_normal_(self.posv)

    def pack(self):
        d = self.d_model
        w, b = self.qvk_proj.weight.detach().float(), self.qvk_proj.bias.detach().float()
        u, v = self.posu.detach().float().reshape(d), self.posv.detach().float().reshape(d)
        # one projection producing [q+u | q+v | k | v]: (q+u) = x Wq^T + (bq + u)
        w_ext = torch.cat([w[:d], w[:d], w[d:2 * d], w[2 * d:]], 0)
        b_ext = torch.cat([b[:d] + u, b[:d] + v, b[d:2 * d], b[2 * d:]], 0)
        return {'wext': w_ext.to(BF16).contiguous(), 'bext': b_ext.contiguous(), 'wpos': _w(self.pos_proj)}

    def run(self, y, x_resid, pk, B, T, lengths, pos_bf16):
        """y = LN(x) bf16 [B*T,d]; returns x_resid + attention (no output projection)."""
        d, H, dk = self.d_model, self.nheads, self.head_dim
        ext = ops.linear(y, pk['wext'], pk['bext'])                       # [M, 4d]
        pproj = ops.linear(pos_bf16, pk['wpos'])                          # [2T-1, d]  pos_proj(PE[-(T-1)..T-1])
        ld = (2 * T - 1 + 3) // 4 * 4
        bd = torch.empty(H, B * T, ld, dtype=torch.float32, device=y.device)
        for h in range(H):  # BD_full[h] = (q+v)_h P_h^T ; the attention kernel reads the j-i+T-1 diagonal band
            # K = dk column views: the GEMM's TMA maps are bounded by K, so a 64-column k-block past the head zero-fills
            ops.linear(ext[:, d + dk * h: d + dk * (h + 1)], pproj[:, dk * h: dk * (h + 1)], out=bd[h])
        return ops.attention(ext, ext, ext, B, H, T, T, kv_len=lengths, q_col0=0, k_col0=2 * d, v_col0=3 * d,
                             bd=bd, resid=x_resid, head_dim=dk)


class ConformerConvolutionModule(nn.Module):
    """Keys: pointwise_conv1.*, depthwise_conv.*, batch_norm.*, pointwise_conv2.*  (module/conformer.py:12-34)."""

    def __init__(self, channels, kernel_size, bias=True, dropout=0.0):
        super().__init__()
        assert kernel_size % 2 == 1
        self.pointwise_conv1 = nn.Linear(channels, 2 * channels, bias=bias)
        self.depthwise_conv = nn.Conv1d(channels, channels, kernel_size, stride=1, padding=(kernel_size - 1) // 2,
                                        groups=channels, bias=bias)
        self.batch_norm = nn.BatchNorm1d(channels)
        self.pointwise_conv2 = nn.Linear(channels, channels, bias=bias)

    def pack(self):
        bn, dw = self.batch_norm, self.depthwise_conv
        s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
        w = dw.weight.detach().float()[:, 0, :] * s[:, None]                       # [C,k] BN scale folded in
        b0 = dw.bias.detach().float() if dw.bias is not None else torch.zeros_like(s)
        b = (b0 - bn.running_mean.detach().float()) * s + bn.bias.detach().float()
        return {'w1': _w(self.pointwise_conv1), 'b1': _b(self.pointwise_conv1),
                'wd': w.t().contiguous(), 'bd': b.contiguous(),                     # tap-major [k,C]
                'w2': _w(self.pointwise_conv2), 'b2': _b(self.pointwise_conv2)}

    def run(self, y, x_resid, pk, B, T, lengths):
        """x_resid + conv_module(y); padded frames are zeroed after the GLU and after the last Linear
        (module/conformer.py:46,55) through the GEMM's row mask."""
        g = ops.linear(y, pk['w1'], pk['b1'], EPI_GLU, row_len=lengths, row_period=T)
        c = ops.dwconv_swish(g, pk['wd'], pk['bd'], B, T)
        return ops.linear(c, pk['w2'], pk['b2'], EPI_RESID, resid=x_resid, row_len=lengths, row_period=T)


class ConformerEncoderBlock(nn.Module):
    def __init__(self, d_model, d_ff, cov_kernel_size, n_heads, slf_attn_dropout=0.0, ffn_dropout=0.0,
                 residual_dropout=0.1, conv_dropout=0.0, macaron_style=True, conv_first=False, ffn_scale=0.5,
                 conv_bias=True, relative_positional=True, activation='glu'):
        super().__init__()
        self.conv_first, self.macaron_style, self.ffn_scale = conv_first, macaron_style, ffn_scale
        self.relative_positional, self.n_heads = relative_positional, n_heads
        if macaron_style:
            self.pre_ffn = PositionwiseFeedForward(d_model, d_ff, ffn_dropout, activation=activation)
            self.macaron_ffn_norm = nn.LayerNorm(d_model)
        if relative_positional:
            self.mha = MultiHeadedSelfAttentionWithRelPos(n_heads, d_model, slf_attn_dropout)
        else:
            self.mha = MultiHeadedSelfAttention(n_heads, d_model, slf_attn_dropout)
        self.mha_norm = nn.LayerNorm(d_model)
        self.conv = ConformerConvolutionModule(d_model, cov_kernel_size, conv_bias, conv_dropout)
        self.conv_norm = nn.LayerNorm(d_model)
        # kept for state_dict parity; the reference never applies post_ffn, only post_ffn_norm (conformer.py:87)
        self.post_ffn = PositionwiseFeedForward(d_model, d_ff, ffn_dropout, activation=activation)
        self.post_ffn_norm = nn.LayerNorm(d_model)
        self.final_norm = nn.LayerNorm(d_model)

    def pack(self):
        pk = {'mha_ln': _ln(self.mha_norm), 'conv_ln': _ln(self.conv_norm), 'post_ln': _ln(self.post_ffn_norm),
              'final_ln': _ln(self.final_norm), 'conv': self.conv.pack()}
        if self.macaron_style:
            pk['pre_ffn'] = _ffn_pack(self.pre_ffn)
            pk['mac_ln'] = _ln(self.macaron_ffn_norm)
        if self.relative_positional:
            pk['mha'] = self.mha.pack()
        else:
            a = self.mha
            pk['mha'] = {'wqkv': _w(a.qvk_proj), 'bqkv': _b(a.qvk_proj), 'wo': _w(a.output_proj), 'bo': _b(a.output_proj)}
        return pk

    def _attn(self, x, pk, B, T, lengths, pos_bf16):
        y = ops.layernorm(x, *pk['mha_ln'])
        if self.relative_positional:
            return self.mha.run(y, x, pk['mha'], B, T, lengths, pos_bf16)
        d, H, m = x.shape[1], self.n_heads, pk['mha']
        qkv = ops.linear(y, m['wqkv'], m['bqkv'])
        ctx = ops.attention(qkv, qkv, qkv, B, H, T, T, kv_len=lengths, q_col0=0, k_col0=d, v_col0=2 * d,
                            head_dim=self.mha.head_dim)
        return ops.linear(ctx, m['wo'], m['bo'], EPI_RESID, resid=x)

    def _conv(self, x, pk, B, T, lengths):
        return self.conv.run(ops.layernorm(x, *pk['conv_ln']), x, pk['conv'], B, T, lengths)

    def run(self, x, pk, B, T, lengths, pos_bf16):
        """ConformerEncoderBlock.forward (encoder/conformer.py:75-89) with the residual dropout disabled."""
        if self.macaron_style:
            y = ops.layernorm(x, *pk['mac_ln'])
            f = pk['pre_ffn']
            h = ops.linear(y, f['w1'], f['b1'], f['act'])
            x = ops.linear(h, f['w2'], f['b2'], EPI_RESID, resid=x, alpha=self.ffn_scale)
        if self.conv_first:
            x = self._attn(self._conv(x, pk, B, T, lengths), pk, B, T, lengths, pos_bf16)
        else:
            x = self._conv(self._attn(x, pk, B, T, lengths, pos_bf16), pk, B, T, lengths)
        return ops.layernorm(x, *pk['post_ln'], *pk['final_ln'])   # post_ffn_norm then final_norm, one kernel


class ConformerEncoder(nn.Module):
    """forward(inputs f32 [B,T,D], mask bool [B,T]) -> (f32 [B,T,D], mask, attn_weights)   (encoder/conformer.py:117-164)

    The reference applies F.dropout(p=residual_dropout) with training=True even in eval() (conformer.py:53,58,63,72),
    i.e. its inference is stochastic for residual_dropout > 0 (SURVEY.md 8a).  This implementation is the
    deterministic network (no dropout at inference); parity is defined against residual_dropout = 0.0."""

    def __init__(self, d_model, d_ff, cov_kernel_size, n_heads, nblocks=12, pos_dropout=0.0, slf_attn_dropout=0.0,
                 ffn_dropout=0.0, residual_dropout=0.1, conv_dropout=0.0, macaron_style=True, ffn_scale=0.5,
                 conv_bias=True, positional_encoding=True, relative_positional=True, conv_first=False,
                 activation='glu'):
        super().__init__()
        self.positional_encoding = positional_encoding
        self.relative_positional = relative_positional
        self.output_size = self.d_model = d_model
        if positional_encoding:
            self.pos_emb = PositionalEncoding(d_model, pos_dropout)
        self.blocks = nn.ModuleList([
            ConformerEncoderBlock(d_model, d_ff, cov_kernel_size, n_heads, slf_attn_dropout, ffn_dropout,
                                  residual_dropout, conv_dropout, macaron_style, conv_first, ffn_scale, conv_bias,
                                  relative_positional, activation) for _ in range(nblocks)])
        self._pack = _Packed(self, lambda: [b.pack() for b in self.blocks])
        self._pos_cache = {}

    def fuse_abs_posenc(self):
        return self.positional_encoding and not self.relative_positional

    def apply_posenc_bf16(self, x, B, T):
        if self.positional_encoding and not self.relative_positional:
            scale, table = self.pos_emb.scale_and_table(T, x.device)
            return ops.scale_add_table(x, scale, table, T)
        return x if x.dtype == BF16 else ops.scale_add_table(x)

    def _rel_pos(self, T, device):
        key = (T, device.index)
        p = self._pos_cache.get(key)
        if p is None:   # PE[-(T-1) .. T-1] (encoder/conformer.py:140-143), bf16 GEMM operand
            p = ops.scale_add_table(ops.sinusoid_table(2 * T - 1, self.d_model, -(T - 1), device))
            self._pos_cache[key] = p
        return p

    def forward_bf16(self, x, B, T, lengths):
        _no_train(self)
        pks = self._pack.get()
        pos = self._rel_pos(T, x.device) if (self.positional_encoding and self.relative_positional) else None
        for blk, pk in zip(self.blocks, pks):
            x = blk.run(x, pk, B, T, lengths, pos)
        return x

    def forward(self, inputs, mask):
        B, T, D = inputs.shape
        x = self.apply_posenc_bf16(inputs.contiguous().view(B * T, D), B, T)
        y = self.forward_bf16(x, B, T, _lengths(mask))
        attn = {'enc_block_%d' % i: {'slf_attn_weights': None} for i in range(len(self.blocks))}
        return y.float().view(B, T, D), mask, attn


# ------------------------------------------------------------------------------------------------
# decoder
# ------------------------------------------------------------------------------------------------
class DecoderCache:
    """The decoder cache the reference stubbed out (decoder/transformer.py:92-126,188-203; README TODO), as the opaque
    `cache` object of ``TransformerDecoder.inference(preds, memory, memory_mask, cache)``:

      * cross-attention K/V of the memory, projected ONCE (the reference re-runs vk_proj on the beam-tiled memory at every
        step, attention.py:129).  When the memory rows are the beam-tiled copies of `batch` utterances
        (recognize/speech2text.py:51-52) pass ``beam`` so that each utterance is projected once and shared by its beams;
      * self-attention K/V of every decoded position [layer, position, row, d]; beam pruning never moves K/V rows, it
        rewrites a 4-byte ancestry entry per (row, position) -- ``reorder(parent_rows)`` is what `decode_step` calls where
        the reference intended reselect_hidden* (recognize/speech2text.py:195-218).

    Build it with ``TransformerDecoder.init_cache``.  One `inference` call consumes exactly one new token per row."""

    def __init__(self, decoder, memory, memory_mask, max_len, beam=1):
        n, T, D = memory.shape
        if n % beam:
            raise ValueError('DecoderCache: memory rows must be a multiple of beam')
        dev = memory.device
        self.N, self.T, self.beam, self.Lmax, self.step = n, T, beam, max_len, 0
        self.batch = n // beam
        nl, d = len(decoder.blocks), decoder.d_model
        pk = decoder.packed()
        self._pk = pk            # the cache is tied to this weight pack (K/V were projected with it)
        mem = memory.contiguous().view(self.batch, beam, T, D)[:, 0]                 # one copy per utterance
        msk = memory_mask.contiguous().view(self.batch, beam, T)[:, 0]
        mem_bf16 = ops.scale_add_table(mem.contiguous().view(self.batch * T, D).float())
        self.mem_len = _lengths(msk)
        self.kvx = torch.empty(nl, self.batch * T, 2 * d, dtype=BF16, device=dev)
        for l, p in enumerate(pk['blocks']):
            ops.linear(mem_bf16, p['wkv'], p['bkv'], out=self.kvx[l])
        self.kc = torch.zeros(nl, max_len, n, d, dtype=BF16, device=dev)
        self.vc = torch.zeros(nl, max_len, n, d, dtype=BF16, device=dev)
        self.anc = torch.zeros(2, n, max_len, dtype=torch.int32, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.table = ops.sinusoid_table(max_len + 1, d, 0, dev)

    def reorder(self, parent_rows):
        """Row n of the next step continues row parent_rows[n] (i64/i32 [N], global row indices)."""
        if self.step == 0:
            raise RuntimeError('DecoderCache.reorder before the first inference step')
        s = self.step - 1                     # the position that was just decoded
        cur, nxt = s & 1, (s & 1) ^ 1
        par = parent_rows.view(-1).long()
        self.anc[nxt] = self.anc[cur].index_select(0, par)
        self.anc[nxt, :, s] = par.to(torch.int32)

    def advance_without_reorder(self):
        """Greedy / teacher-forced use (no pruning): every row continues itself."""
        self.reorder(torch.arange(self.N, device=self.anc.device))


class TransformerDecoderLayer(nn.Module):
    def __init__(self, n_heads, d_model, d_ff, memory_dim, slf_attn_dropout=0.0, src_attn_dropout=0.0,
                 ffn_dropout=0.0, residual_dropout=0.1, normalize_before=False, concat_after=False,
                 relative_positional=False, activation='relu'):
        super().__init__()
        if concat_after or relative_positional:
            raise NotImplementedError('concat_after / relative_positional decoder')
        self.n_heads = n_heads
        self.normalize_before = normalize_before
        self.dropout_rates = {'slf_attn_dropout': slf_attn_dropout, 'src_attn_dropout': src_attn_dropout,
                              'ffn_dropout': ffn_dropout, 'residual_dropout': residual_dropout}
        self.slf_attn = MultiHeadedSelfAttention(n_heads, d_model, slf_attn_dropout)
        self.src_attn = MultiHeadedCrossAttention(n_heads, d_model, memory_dim, src_attn_dropout)
        self.feed_forward = PositionwiseFeedForward(d_model, d_ff, ffn_dropout, activation)
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)
        self.norm3 = nn.LayerNorm(d_model)

    def pack(self):
        a, c = self.slf_attn, self.src_attn
        return {'wqkv': _w(a.qvk_proj), 'bqkv': _b(a.qvk_proj), 'wo': _w(a.output_proj), 'bo': _b(a.output_proj),
                'wq': _w(c.q_proj), 'bq': _b(c.q_proj), 'wkv': _w(c.vk_proj), 'bkv': _b(c.vk_proj),
                'wo2': _w(c.output_proj), 'bo2': _b(c.output_proj), 'ffn': _ffn_pack(self.feed_forward),
                'ln1': _ln(self.norm1), 'ln2': _ln(self.norm2), 'ln3': _ln(self.norm3)}


class TransformerDecoder(nn.Module):
    """forward(targets i64 [B,L], memory f32 [B,T,D], memory_mask bool [B,T]) -> (logits f32 [B,L,V], attn)
    inference(preds i64 [N,l], memory, memory_mask, cache) -> (log_probs f32 [N,V], cache, attn)
    (decoder/transformer.py:161-208).  `cache` is passed through untouched exactly like the reference;
    the KV-cached incremental path lives in recognize.BeamDecoder."""

    def __init__(self, vocab_size, d_model=256, n_heads=4, d_ff=2048, memory_dim=256, n_blocks=6, pos_dropout=0.0,
                 slf_attn_dropout=0.0, src_attn_dropout=0.0, ffn_dropout=0.0, residual_dropout=0.1,
                 activation='relu', normalize_before=True, concat_after=False, share_embedding=False):
        super().__init__()
        self.decoder_type = 'transformer'
        self.normalize_before = normalize_before
        self.relative_positional = False
        self.d_model, self.n_heads, self.vocab_size = d_model, n_heads, vocab_size
        self.head_dim = head_dim_of(n_heads, d_model)
        self.embedding = nn.Embedding(vocab_size, d_model)
        self.pos_emb = PositionalEncoding(d_model, pos_dropout)
        self.blocks = nn.ModuleList([
            TransformerDecoderLayer(n_heads, d_model, d_ff, memory_dim, slf_attn_dropout, src_attn_dropout,
                                    ffn_dropout, residual_dropout, normalize_before, concat_after, False, activation)
            for _ in range(n_blocks)])
        if normalize_before:
            self.after_norm = nn.LayerNorm(d_model)
        self.output_layer = nn.Linear(d_model, vocab_size)
        if share_embedding:
            assert self.embedding.weight.size() == self.output_layer.weight.size()
            self.output_layer.weight = self.embedding.weight   # tied (decoder/transformer.py:156-158)
        self._pack = _Packed(self, self._build_pack)

    def _build_pack(self):
        emb = self.embedding.weight.detach().to(BF16).contiguous()
        tied = self.output_layer.weight is self.embedding.weight
        return {'emb': emb, 'wout': emb if tied else _w(self.output_layer), 'bout': _b(self.output_layer),
                'blocks': [b.pack() for b in self.blocks],
                'after': _ln(self.after_norm) if self.normalize_before else None}

    def packed(self):
        return self._pack.get()

    @property
    def ld_logits(self):
        return (self.vocab_size + 7) // 8 * 8

    def forward_bf16(self, targets, memory_bf16, mem_len, B, L, T):
        """targets i64 [B,L]; memory bf16 [B*T, D] -> logits f32 [B*L, ld_logits] (first V columns valid)."""
        _no_train(self)
        pk = self._pack.get()
        d, H = self.d_model, self.n_heads
        scale, table = self.pos_emb.scale_and_table(L, memory_bf16.device)
        if self.pos_emb.scale_learnable:
            raise NotImplementedError('decoder with learnable positional scale')
        x = ops.embed_posenc(targets.contiguous(), pk['emb'], table, B * L, d, period=L)
        for blk, p in zip(self.blocks, pk['blocks']):
            nb = blk.normalize_before
            if nb:
                x = ops.layernorm(x, *p['ln1'])
            qkv = ops.linear(x, p['wqkv'], p['bqkv'])
            ctx = ops.attention(qkv, qkv, qkv, B, H, L, L, causal=True, q_col0=0, k_col0=d, v_col0=2 * d, head_dim=self.head_dim)
            x = _proj_resid_ln(ctx, p['wo'], p['bo'], x, None if nb else p['ln1'])
            if nb:
                x = ops.layernorm(x, *p['ln2'])
            q = ops.linear(x, p['wq'], p['bq'])
            kv = ops.linear(memory_bf16, p['wkv'], p['bkv'])
            ctx = ops.attention(q, kv, kv, B, H, L, T, kv_len=mem_len, k_col0=0, v_col0=d, head_dim=self.head_dim)
            x = _proj_resid_ln(ctx, p['wo2'], p['bo2'], x, None if nb else p['ln2'])
            if nb:
                x = ops.layernorm(x, *p['ln3'])
            x = _ffn(x, p['ffn'], x, None if nb else p['ln3'])
        if self.normalize_before:
            x = ops.layernorm(x, *pk['after'])
        return ops.linear(x, pk['wout'], pk['bout'], EPI_BIAS, out_f32=True, n_out=self.ld_logits)

    def forward(self, targets, memory, memory_mask):
        B, L = targets.shape
        T, D = memory.shape[1], memory.shape[2]
        mem = ops.scale_add_table(memory.contiguous().view(B * T, D))   # f32 -> bf16
        logits = self.forward_bf16(targets, mem, _lengths(memory_mask), B, L, T)
        attn = {'dec_block_%d' % i: {'slf_attn_weights': None, 'src_attn_weights': None}
                for i in range(len(self.blocks))}
        return logits.view(B, L, -1)[:, :, :self.vocab_size], attn

    def init_cache(self, memory, memory_mask, max_len, beam=1):
        """KV cache for `inference` (see DecoderCache).  memory f32 [N,T,D] (beam-tiled or not), memory_mask bool [N,T]."""
        _no_train(self)
        return DecoderCache(self, memory, memory_mask, max_len, beam)

    def inference(self, preds, memory, memory_mask=None, cache=None):
        """decoder/transformer.py:185-208.  cache None (the reference's only working mode): the whole prefix is recomputed.
        cache = DecoderCache (``init_cache``): only the newest token preds[:, -1] is run through the layers against the cached
        keys / values -- O(l) instead of O(l^2) per step -- and the same object is returned; the caller reorders it after
        pruning (SpeechToTextRecognizer.decode_step does)."""
        assert preds.dim() == 2
        if isinstance(cache, DecoderCache):
            return self._inference_cached(preds, cache)
        logits, attn = self.forward(preds, memory, memory_mask)       # full recompute, as transformer.py:204
        last = logits[:, -1, :].contiguous()
        return ops.log_softmax(last, self.vocab_size), cache, attn

    def _inference_cached(self, preds, c):
        _no_train(self)
        pk = self._pack.get()
        if pk is not c._pk:
            raise RuntimeError('DecoderCache was built with different decoder weights (parameters changed since init_cache)')
        if preds.shape[0] != c.N or preds.shape[1] != c.step + 1:
            raise ValueError(f'cached inference expects preds [N={c.N}, {c.step + 1}] (one new token per call), got {tuple(preds.shape)}')
        if c.step >= c.Lmax:
            raise ValueError('DecoderCache is full (max_len reached)')
        if self.pos_emb.scale_learnable:
            raise NotImplementedError('decoder with learnable positional scale')
        d, H, N = self.d_model, self.n_heads, c.N
        c.step_dev.fill_(c.step)
        tok = preds[:, -1].contiguous()
        x = ops.embed_posenc(tok, pk['emb'], c.table, N, d, step_ptr=c.step_dev)
        for l, (blk, p) in enumerate(zip(self.blocks, pk['blocks'])):
            nb = blk.normalize_before
            if nb:
                x = ops.layernorm(x, *p['ln1'])
            qkv = ops.linear(x, p['wqkv'], p['bqkv'])
            ctx = ops.decode_self_attn(qkv, c.kc[l], c.vc[l], c.anc, c.step_dev, N, H, c.Lmax, head_dim=self.head_dim)
            x = _proj_resid_ln(ctx, p['wo'], p['bo'], x, None if nb else p['ln1'])
            if nb:
                x = ops.layernorm(x, *p['ln2'])
            q = ops.linear(x, p['wq'], p['bq'])
            ctx = ops.attention(q, c.kvx[l], c.kvx[l], c.batch, H, c.beam, c.T, kv_len=c.mem_len, k_col0=0, v_col0=d,
                                head_dim=self.head_dim)
            x = _proj_resid_ln(ctx, p['wo2'], p['bo2'], x, None if nb else p['ln2'])
            if nb:
                x = ops.layernorm(x, *p['ln3'])
            x = _ffn(x, p['ffn'], x, None if nb else p['ln3'])
        if self.normalize_before:
            x = ops.layernorm(x, *pk['after'])
        logits = ops.linear(x, pk['wout'], pk['bout'], EPI_BIAS, out_f32=True, n_out=self.ld_logits)
        c.step += 1
        attn = {'dec_block_%d' % i: {'slf_attn_weights': None, 'src_attn_weights': None} for i in range(len(self.blocks))}
        return ops.log_softmax(logits, self.vocab_size), c, attn
