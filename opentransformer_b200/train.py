"""Training step of the speech transformer on the B200 path (SURVEY.md 8a rows 16-17, 8e).

Mirror of the inner step of otrans/train/trainer.py:206-234 for `SpeechToText` (model/speech2text.py:39-64):

    loss, _ = model(inputs, targets); loss.backward(); clip_grad_norm_(params, 5); scheduler.step(); optimizer.step()

The reference differentiates its forward through torch autograd.  Here the backward is written by hand as a reverse
walk over a tape of saved bf16 activations, so that every contraction runs on the tcgen05 kernels (dgrad = otb_linear
with the transposed weight, residual gradients fused into its epilogue; wgrad = otb_linear_wgrad; attention backward =
otb_attention_bwd) and everything else on the HBM-bound backward kernels (csrc/backward.cu).  The only torch autograd
node is `_SpeechToTextLoss`, which makes `model(inputs, targets)[0].backward()` populate `.grad` of the fp32 master
parameters exactly like the reference module.

Scope: the shipped Speech-Transformer configuration -- conv front end, post-norm Transformer encoder / decoder with GLU
feed-forward, tied or untied output layer, `residual_dropout` as shipped (0.1: counter-based masks in the residual GEMM's
epilogue, replayed in the backward; csrc/dropout.cuh); the other dropout rates must be 0 (as shipped) and raise
otherwise.  Conformer / pre-norm training is not built yet and raises.
"""
import math

import torch

from . import ops
from . import modules
from .dp import allreduce_mean_
from .modules import TransformerDecoder, TransformerEncoder, ConvFrontEnd, _lengths
from .ops import BF16, EPI_BIAS, EPI_RESID, EPI_TABLE, EPI_RELU


def _bf(t):
    return t.detach().to(BF16).contiguous()


def _f(t):
    return t.detach().float().contiguous()


class TrainPack:
    """bf16 operands of one training step: W [N,K] for the forward / wgrad, W^T [K,N] for the dgrad GEMMs.
    `bf16_of(param)` (optional) returns a bf16 copy of a parameter without a per-tensor cast kernel (FusedTrainer casts
    its flat fp32 master buffer once per step and hands out views)."""

    def __init__(self, model, bf16_of=None):
        self._bf16_of = bf16_of
        fe, enc, dec = model.frontend, model.encoder, model.decoder
        if not isinstance(fe, ConvFrontEnd) or not isinstance(enc, TransformerEncoder) or not isinstance(dec, TransformerDecoder):
            raise NotImplementedError('training path: conv front end + Transformer encoder / decoder only (round 1)')
        if enc.relative_positional:
            raise NotImplementedError('training path: absolute positions only')
        for blk in list(enc.blocks) + list(dec.blocks):
            if blk.slf_attn.head_dim != 64:
                # the attention backward kernel (otb_attention_bwd) is built for 64-wide heads only
                raise NotImplementedError(f'training path: the attention backward supports d_k = 64 only, '
                                          f'got d_k = {blk.slf_attn.head_dim}')
        if fe.front_end_layer_norm or enc.pos_emb.scale_learnable or dec.pos_emb.scale_learnable:
            raise NotImplementedError('training path: front_end_layer_norm / learnable positional scale')
        for blk in list(enc.blocks) + list(dec.blocks):
            if blk.feed_forward.activation not in ('glu', 'relu'):
                raise NotImplementedError('training path: GLU or ReLU feed-forward only')
            rates = getattr(blk, 'dropout_rates', {})
            other = {k: v for k, v in rates.items() if k != 'residual_dropout' and float(v) > 0.0}
            if other:
                # the reference applies these in train mode (attention.py:45, ffn.py:40); training WITHOUT them would be a
                # different network, so refuse instead of silently dropping the regulariser.  residual_dropout -- the only
                # non-zero rate of the shipped configs -- IS implemented (otb_linear_dropout_resid / otb_dropout_bwd).
                raise NotImplementedError(f'training path: only residual_dropout is implemented, got {other}; set them to 0.0')
            if not (0.0 <= float(rates.get('residual_dropout', 0.0)) < 1.0):
                raise ValueError('residual_dropout must be in [0, 1)')
        self.fe = self._frontend(fe)
        self.enc = [self._enc_layer(b) for b in enc.blocks]
        self.dec = [self._dec_layer(b) for b in dec.blocks]
        # pre-norm stacks end with one more LayerNorm (encoder/transformer.py:96-97,131-132; decoder/transformer.py:151-152,178-179)
        self.enc_pre, self.dec_pre = bool(enc.normalize_before), bool(dec.normalize_before)
        self.enc_norm = self._ln(enc.norm) if self.enc_pre else None
        self.dec_norm = self._ln(dec.after_norm) if self.dec_pre else None
        V, d = dec.vocab_size, dec.d_model
        self.ld_logits = dec.ld_logits
        emb = self._w(dec.embedding.weight)
        self.tied = dec.output_layer.weight is dec.embedding.weight
        wout = emb if self.tied else self._w(dec.output_layer.weight)
        wout_t = torch.zeros(d, self.ld_logits, dtype=BF16, device=emb.device)      # [d, V padded]: dgrad of the logits GEMM
        wout_t[:, :V] = wout.t()
        self.out = {'emb': emb, 'wout': wout, 'wout_t': wout_t, 'bout': _f(dec.output_layer.bias)}

    def _w(self, param):
        return self._bf16_of(param) if self._bf16_of is not None else _bf(param)

    def _lin(self, lin):
        w = self._w(lin.weight)
        return w, w.t().contiguous(), _f(lin.bias)

    @staticmethod
    def _ln(norm):
        return _f(norm.weight), _f(norm.bias)

    def _frontend(self, fe):
        pk = dict(fe._build_pack())
        pk['w2_t'] = pk['w2'].t().contiguous()           # [9*C1p, C2]
        pk['wo_t'] = pk['wo'].t().contiguous()           # [F2*C2, D]
        return pk

    def _enc_layer(self, b):
        a, f = b.slf_attn, b.feed_forward
        return {'qkv': self._lin(a.qvk_proj), 'o': self._lin(a.output_proj), 'w1': self._lin(f.w_1), 'w2': self._lin(f.w_2),
                'ln1': self._ln(b.norm1), 'ln2': self._ln(b.norm2), 'act': f.activation}

    def _dec_layer(self, b):
        a, c, f = b.slf_attn, b.src_attn, b.feed_forward
        return {'qkv': self._lin(a.qvk_proj), 'o': self._lin(a.output_proj), 'q': self._lin(c.q_proj),
                'kv': self._lin(c.vk_proj), 'o2': self._lin(c.output_proj), 'w1': self._lin(f.w_1), 'w2': self._lin(f.w_2),
                'ln1': self._ln(b.norm1), 'ln2': self._ln(b.norm2), 'ln3': self._ln(b.norm3), 'act': f.activation}


class _Grads(dict):
    """name -> fp32 gradient.  With `sink` (name -> fp32 view of the optimizer's flat gradient buffer) the kernels ADD
    their result straight into the sink (otb_linear_wgrad / otb_colsum / otb_layernorm_bwd accumulate flags) -- what
    autograd's AccumulateGrad does, without one torch add per parameter."""

    def __init__(self, sink=None):
        super().__init__()
        self.sink = sink

    def out(self, name):
        return self.sink[name] if self.sink is not None else None

    def put(self, name, value):
        """For gradients produced by code that cannot accumulate in place."""
        if self.sink is not None:
            self.sink[name].add_(value.reshape(self.sink[name].shape))
            self[name] = self.sink[name]
        else:
            self[name] = value.contiguous()


def _ln_bwd(dy, z, gamma, grads, wname, bname):
    acc = grads.sink is not None
    dz, dg, db = ops.layernorm_bwd(dy, z, gamma, dgamma=grads.out(wname), dbeta=grads.out(bname), accumulate=acc)
    grads[wname], grads[bname] = dg, db
    return dz


def _linear_bwd(dy, x, wt, grads, wname, bname, resid=None):
    """Gradients of y = x W^T + b: parameter grads into `grads`, returns dx (+ resid) as bf16."""
    acc = grads.sink is not None
    grads[wname] = ops.linear_wgrad(dy, x, out=grads.out(wname), accumulate=acc)
    grads[bname] = ops.colsum(dy, out=grads.out(bname), accumulate=acc)
    if wt is None:
        return None
    if resid is not None:
        return ops.linear(dy, wt, None, EPI_RESID, resid=resid)
    return ops.linear(dy, wt)


ENC_SITE, DEC_SITE = 0, 1000      # dropout site ids: encoder layer i -> 2 i + {0, 1}; decoder layer i -> 1000 + 3 i + {0, 1, 2}


def _ffn_fwd(p, x):
    """First half of the position-wise feed-forward (ffn.py:38-41): returns (pre-activation u or None, hidden h)."""
    if p['act'] == 'glu':
        u = ops.linear(x, p['w1'][0], p['w1'][2])
        return u, ops.glu_fwd(u)
    return None, ops.linear(x, p['w1'][0], p['w1'][2], EPI_RELU)      # ReLU fused into the GEMM; its backward needs only h


def _ffn_act_bwd(p, dh, u, h):
    return ops.glu_bwd(dh, u) if p['act'] == 'glu' else ops.relu_bwd(dh, h)


def dropout_sites(model):
    """[(site id, 'encoder' | 'decoder', rate)] of every residual-dropout site (what a parity test must replay)."""
    out = []
    for i, b in enumerate(model.encoder.blocks):
        out += [(ENC_SITE + 2 * i + k, 'encoder', float(b.dropout_rates['residual_dropout'])) for k in range(2)]
    for i, b in enumerate(model.decoder.blocks):
        out += [(DEC_SITE + 3 * i + k, 'decoder', float(b.dropout_rates['residual_dropout'])) for k in range(3)]
    return out


def _resid(ctx, w, b, x, rate, seed, site):
    """x + dropout(ctx W^T + b): the residual connection of a sub-layer in training mode (transformer.py:54,61)."""
    if rate > 0.0:
        return ops.linear_dropout_resid(ctx, w, b, x, rate, seed, site)
    return ops.linear(ctx, w, b, EPI_RESID, resid=x)


def _drop_bwd(dz, rate, seed, site):
    return ops.dropout_bwd(dz, rate, seed, site) if rate > 0.0 else dz


def forward_backward(model, inputs, mask, truth, smoothing=None, want_grads=True, grad_sink=None, grad_scale=1.0,
                     bf16_of=None, drop_seed=None, truth_length=None, return_ctc=False):
    """One forward (+ backward) pass.  inputs f32 [B,T,F], mask bool [B,T], truth i64 [B,L+1] (BOS ... EOS PAD*).
    Returns (loss 0-d f32 tensor, {parameter name -> fp32 gradient}) with names as in model.named_parameters().
    grad_sink: name -> fp32 tensor the gradients (x grad_scale) are ADDED into (gradient accumulation buffer).
    drop_seed: int32 device tensor [1], the dropout seed of THIS pass (read on the device); required when any
    residual_dropout rate is non-zero.  truth_length: i32/i64 [B] label counts incl. <S/E> (targets['targets_length'],
    data/loader.py:94) -- required when model.ctc_weight > 0: the loss is then (1 - w) * attention + w * CTC
    (model/speech2text.py:60-62) and the CTC head's gradients flow into the encoder through the memory."""
    fe, enc, dec = model.frontend, model.encoder, model.decoder
    ctc_w = float(getattr(model, 'ctc_weight', 0.0) or 0.0)
    if ctc_w > 0.0 and truth_length is None:
        raise ValueError('forward_backward: ctc_weight > 0 needs truth_length')
    pk = TrainPack(model, bf16_of)
    dev = inputs.device
    e_rates = [float(b.dropout_rates['residual_dropout']) for b in enc.blocks]
    d_rates = [float(b.dropout_rates['residual_dropout']) for b in dec.blocks]
    if drop_seed is None and any(r > 0.0 for r in e_rates + d_rates):
        raise ValueError('forward_backward: residual_dropout > 0 needs a drop_seed tensor')
    B, T, F = inputs.shape
    H, d = enc.blocks[0].n_heads, enc.d_model
    x_in = inputs.contiguous().float()
    _, _, T2, F2 = ops.conv_geometry(T, F)
    T1, F1 = (T - 3) // 2 + 1, (F - 1) // 2 + 1
    lengths = _lengths(fe.output_mask(mask))
    fpk = pk.fe
    C1p, C2 = fpk['C1p'], fpk['w2'].shape[0]

    # ------------------------------------------------------------------ forward
    h1 = ops.conv1_relu(x_in, fpk['w1'], fpk['b1'])
    h2 = ops.conv2_relu(h1, fpk['w2'], fpk['b2'], B, T, F)                       # [B*T2, F2*C2]
    scale, table = enc.pos_emb.scale_and_table(T2, dev)
    x = ops.linear(h2, fpk['wo'], fpk['bo'], EPI_TABLE, alpha=scale, table=table, period=T2)
    enc_tape = []
    for i, p in enumerate(pk.enc):
        if pk.enc_pre:
            # pre-norm as the reference writes it (encoder/transformer.py:41-63): the residual is taken AFTER the norm,
            # x = n + sublayer(n) with n = norm(x); the stack ends with one more LayerNorm
            xn = ops.layernorm(x, *p['ln1'])
            qkv = ops.linear(xn, p['qkv'][0], p['qkv'][2])
            ctx, lse = ops.attention_train(qkv, qkv, qkv, B, H, T2, T2, kv_len=lengths, q_col0=0, k_col0=d, v_col0=2 * d)
            z1 = _resid(ctx, p['o'][0], p['o'][2], xn, e_rates[i], drop_seed, ENC_SITE + 2 * i)
            x1 = ops.layernorm(z1, *p['ln2'])
            u, h = _ffn_fwd(p, x1)
            z2 = _resid(h, p['w2'][0], p['w2'][2], x1, e_rates[i], drop_seed, ENC_SITE + 2 * i + 1)
            enc_tape.append((x, qkv, ctx, lse, z1, x1, u, h, xn))
            x = z2
            continue
        qkv = ops.linear(x, p['qkv'][0], p['qkv'][2])
        ctx, lse = ops.attention_train(qkv, qkv, qkv, B, H, T2, T2, kv_len=lengths, q_col0=0, k_col0=d, v_col0=2 * d)
        z1 = _resid(ctx, p['o'][0], p['o'][2], x, e_rates[i], drop_seed, ENC_SITE + 2 * i)
        x1 = ops.layernorm(z1, *p['ln1'])
        u, h = _ffn_fwd(p, x1)
        z2 = _resid(h, p['w2'][0], p['w2'][2], x1, e_rates[i], drop_seed, ENC_SITE + 2 * i + 1)
        enc_tape.append((x, qkv, ctx, lse, z1, x1, u, h, z2))
        x = ops.layernorm(z2, *p['ln2'])
    enc_last = x
    mem = ops.layernorm(x, *pk.enc_norm) if pk.enc_pre else x

    tgt_in = truth[:, :-1].contiguous()
    tgt_out = truth[:, 1:].contiguous()
    L = tgt_in.shape[1]
    Hd = dec.n_heads
    _, dtable = dec.pos_emb.scale_and_table(L, dev)
    y = ops.embed_posenc(tgt_in, pk.out['emb'], dtable, B * L, d, period=L)
    dec_tape = []
    for i, p in enumerate(pk.dec):
        if pk.dec_pre:      # decoder/transformer.py:54-90 with normalize_before: y = n + sublayer(n), n = norm(y), three times
            yn = ops.layernorm(y, *p['ln1'])
            qkv = ops.linear(yn, p['qkv'][0], p['qkv'][2])
            ctx, lse = ops.attention_train(qkv, qkv, qkv, B, Hd, L, L, causal=True, q_col0=0, k_col0=d, v_col0=2 * d)
            z1 = _resid(ctx, p['o'][0], p['o'][2], yn, d_rates[i], drop_seed, DEC_SITE + 3 * i)
            y1 = ops.layernorm(z1, *p['ln2'])
            q = ops.linear(y1, p['q'][0], p['q'][2])
            kv = ops.linear(mem, p['kv'][0], p['kv'][2])
            ctx2, lse2 = ops.attention_train(q, kv, kv, B, Hd, L, T2, kv_len=lengths, k_col0=0, v_col0=d)
            z2 = _resid(ctx2, p['o2'][0], p['o2'][2], y1, d_rates[i], drop_seed, DEC_SITE + 3 * i + 1)
            y2 = ops.layernorm(z2, *p['ln3'])
            u, h = _ffn_fwd(p, y2)
            z3 = _resid(h, p['w2'][0], p['w2'][2], y2, d_rates[i], drop_seed, DEC_SITE + 3 * i + 2)
            dec_tape.append((y, qkv, ctx, lse, z1, y1, q, kv, ctx2, lse2, z2, y2, u, h, yn))
            y = z3
            continue
        qkv = ops.linear(y, p['qkv'][0], p['qkv'][2])
        ctx, lse = ops.attention_train(qkv, qkv, qkv, B, Hd, L, L, causal=True, q_col0=0, k_col0=d, v_col0=2 * d)
        z1 = _resid(ctx, p['o'][0], p['o'][2], y, d_rates[i], drop_seed, DEC_SITE + 3 * i)
        y1 = ops.layernorm(z1, *p['ln1'])
        q = ops.linear(y1, p['q'][0], p['q'][2])
        kv = ops.linear(mem, p['kv'][0], p['kv'][2])
        ctx2, lse2 = ops.attention_train(q, kv, kv, B, Hd, L, T2, kv_len=lengths, k_col0=0, v_col0=d)
        z2 = _resid(ctx2, p['o2'][0], p['o2'][2], y1, d_rates[i], drop_seed, DEC_SITE + 3 * i + 1)
        y2 = ops.layernorm(z2, *p['ln2'])
        u, h = _ffn_fwd(p, y2)
        z3 = _resid(h, p['w2'][0], p['w2'][2], y2, d_rates[i], drop_seed, DEC_SITE + 3 * i + 2)
        dec_tape.append((y, qkv, ctx, lse, z1, y1, q, kv, ctx2, lse2, z2, y2, u, h, z3))
        y = ops.layernorm(z3, *p['ln3'])
    V = dec.vocab_size
    dec_last = y
    if pk.dec_pre:
        y = ops.layernorm(y, *pk.dec_norm)
    logits = ops.linear(y, pk.out['wout'], pk.out['bout'], EPI_BIAS, out_f32=True, n_out=pk.ld_logits)
    sm = model.smoothing if smoothing is None else smoothing
    loss_ctc, dctc = None, None
    if ctc_w > 0.0:     # CTCAssistor on the encoder states (model/ctc.py:33-52)
        wc = pk._w(model.assistor.output_layer.weight)
        ctc_logits = ops.linear(mem, wc, _f(model.assistor.output_layer.bias), EPI_BIAS, out_f32=True, n_out=model.assistor.ld_logits)
        loss_ctc, _, dctc = ops.ctc_loss(ctc_logits, B, T2, V, lengths, tgt_out, truth_length.to(torch.int32).to(dev).contiguous(),
                                         model.assistor.blank, want_grad=want_grads, grad_scale=ctc_w * grad_scale)
    if not want_grads:
        loss, _ = ops.ls_cross_entropy(logits, tgt_out, V, sm)
        if ctc_w > 0.0:
            loss = (1.0 - ctc_w) * loss + ctc_w * loss_ctc
        return (loss, None, loss_ctc) if return_ctc else (loss, None)
    loss, dlogits = ops.ls_cross_entropy_train(logits, tgt_out, V, sm)
    att_scale = grad_scale * (1.0 - ctc_w)
    if att_scale != 1.0:
        dlogits = ops.scale_add_table(dlogits, att_scale)                        # loss / accum_steps (trainer.py:216), x (1 - w)
    if ctc_w > 0.0:
        loss = (1.0 - ctc_w) * loss + ctc_w * loss_ctc

    # ------------------------------------------------------------------ backward
    g = _Grads(grad_sink)
    acc = grad_sink is not None
    wname = 'decoder.embedding.weight' if pk.tied else 'decoder.output_layer.weight'
    # dlogits[:, :V] as a strided view: the TMA map stops at column V, so the result has exactly V rows
    dwout = ops.linear_wgrad(dlogits[:, :V], y, out=g.out(wname), accumulate=acc)          # [V, d]
    g.put('decoder.output_layer.bias', ops.colsum(dlogits)[:V])
    dy = ops.linear(dlogits, pk.out['wout_t'])                                   # [B*L, d]
    dmem = None
    if pk.dec_pre:
        dy = _ln_bwd(dy, dec_last, pk.dec_norm[0], g, 'decoder.after_norm.weight', 'decoder.after_norm.bias')
    for i in reversed(range(len(pk.dec))):
        p, pre = pk.dec[i], f'decoder.blocks.{i}.'
        rt, st0 = d_rates[i], DEC_SITE + 3 * i
        if pk.dec_pre:
            (y0, qkv, ctx, lse, z1, y1, q, kv, ctx2, lse2, z2, y2, u, h, yn) = dec_tape[i]
            # z3 = y2 + drop(ffn(y2)), y2 = norm3(z2): dy is the gradient of z3
            dh = _linear_bwd(_drop_bwd(dy, rt, drop_seed, st0 + 2), h, p['w2'][1], g, pre + 'feed_forward.w_2.weight', pre + 'feed_forward.w_2.bias')
            du = _ffn_act_bwd(p, dh, u, h)
            dy2 = _linear_bwd(du, y2, p['w1'][1], g, pre + 'feed_forward.w_1.weight', pre + 'feed_forward.w_1.bias', resid=dy)
            dz2 = _ln_bwd(dy2, z2, p['ln3'][0], g, pre + 'norm3.weight', pre + 'norm3.bias')
            dctx2 = _linear_bwd(_drop_bwd(dz2, rt, drop_seed, st0 + 1), ctx2, p['o2'][1], g, pre + 'src_attn.output_proj.weight', pre + 'src_attn.output_proj.bias')
            dq = torch.empty_like(q)
            dkv = torch.empty_like(kv)
            ops.attention_bwd(q, kv, kv, ctx2, dctx2, lse2, B, Hd, L, T2, dq, dkv, dkv, kv_len=lengths, k_col0=0, v_col0=d,
                              dq_col0=0, dk_col0=0, dv_col0=d)
            dmem = _linear_bwd(dkv, mem, p['kv'][1], g, pre + 'src_attn.vk_proj.weight', pre + 'src_attn.vk_proj.bias', resid=dmem)
            dy1 = _linear_bwd(dq, y1, p['q'][1], g, pre + 'src_attn.q_proj.weight', pre + 'src_attn.q_proj.bias', resid=dz2)
            dz1 = _ln_bwd(dy1, z1, p['ln2'][0], g, pre + 'norm2.weight', pre + 'norm2.bias')
            dctx = _linear_bwd(_drop_bwd(dz1, rt, drop_seed, st0), ctx, p['o'][1], g, pre + 'slf_attn.output_proj.weight', pre + 'slf_attn.output_proj.bias')
            dqkv = torch.empty_like(qkv)
            ops.attention_bwd(qkv, qkv, qkv, ctx, dctx, lse, B, Hd, L, L, dqkv, dqkv, dqkv, causal=True, q_col0=0, k_col0=d,
                              v_col0=2 * d, dq_col0=0, dk_col0=d, dv_col0=2 * d)
            dyn = _linear_bwd(dqkv, yn, p['qkv'][1], g, pre + 'slf_attn.qvk_proj.weight', pre + 'slf_attn.qvk_proj.bias', resid=dz1)
            dy = _ln_bwd(dyn, y0, p['ln1'][0], g, pre + 'norm1.weight', pre + 'norm1.bias')
            continue
        (y0, qkv, ctx, lse, z1, y1, q, kv, ctx2, lse2, z2, y2, u, h, z3) = dec_tape[i]
        dz3 = _ln_bwd(dy, z3, p['ln3'][0], g, pre + 'norm3.weight', pre + 'norm3.bias')
        # the sub-layer branch sees the replayed dropout mask, the residual branch (resid= below) the plain gradient
        dh = _linear_bwd(_drop_bwd(dz3, rt, drop_seed, st0 + 2), h, p['w2'][1], g, pre + 'feed_forward.w_2.weight', pre + 'feed_forward.w_2.bias')
        du = _ffn_act_bwd(p, dh, u, h)
        dy2 = _linear_bwd(du, y2, p['w1'][1], g, pre + 'feed_forward.w_1.weight', pre + 'feed_forward.w_1.bias', resid=dz3)
        dz2 = _ln_bwd(dy2, z2, p['ln2'][0], g, pre + 'norm2.weight', pre + 'norm2.bias')
        dctx2 = _linear_bwd(_drop_bwd(dz2, rt, drop_seed, st0 + 1), ctx2, p['o2'][1], g, pre + 'src_attn.output_proj.weight', pre + 'src_attn.output_proj.bias')
        dq = torch.empty_like(q)
        dkv = torch.empty_like(kv)
        ops.attention_bwd(q, kv, kv, ctx2, dctx2, lse2, B, Hd, L, T2, dq, dkv, dkv, kv_len=lengths, k_col0=0, v_col0=d,
                          dq_col0=0, dk_col0=0, dv_col0=d)
        dmem = _linear_bwd(dkv, mem, p['kv'][1], g, pre + 'src_attn.vk_proj.weight', pre + 'src_attn.vk_proj.bias', resid=dmem)
        dy1 = _linear_bwd(dq, y1, p['q'][1], g, pre + 'src_attn.q_proj.weight', pre + 'src_attn.q_proj.bias', resid=dz2)
        dz1 = _ln_bwd(dy1, z1, p['ln1'][0], g, pre + 'norm1.weight', pre + 'norm1.bias')
        dctx = _linear_bwd(_drop_bwd(dz1, rt, drop_seed, st0), ctx, p['o'][1], g, pre + 'slf_attn.output_proj.weight', pre + 'slf_attn.output_proj.bias')
        dqkv = torch.empty_like(qkv)
        ops.attention_bwd(qkv, qkv, qkv, ctx, dctx, lse, B, Hd, L, L, dqkv, dqkv, dqkv, causal=True, q_col0=0, k_col0=d,
                          v_col0=2 * d, dq_col0=0, dk_col0=d, dv_col0=2 * d)
        dy = _linear_bwd(dqkv, y0, p['qkv'][1], g, pre + 'slf_attn.qvk_proj.weight', pre + 'slf_attn.qvk_proj.bias', resid=dz1)
    # embedding (decoder/transformer.py:163,169); with tied weights the output-layer gradient lands in the same tensor
    if pk.tied:
        ops.embed_bwd(tgt_in, dy, dwout, math.sqrt(d))          # atomics on top of the output-layer gradient
        g['decoder.embedding.weight'] = dwout
    else:
        g['decoder.output_layer.weight'] = dwout
        demb = g.out('decoder.embedding.weight')
        if demb is None:
            demb = torch.zeros(V, d, dtype=torch.float32, device=dev)
        ops.embed_bwd(tgt_in, dy, demb, math.sqrt(d))
        g['decoder.embedding.weight'] = demb

    dx = dmem
    if ctc_w > 0.0:     # CTC head: parameter gradients, and its gradient with respect to the memory joins the decoder's
        wname_c = 'assistor.output_layer.weight'
        g[wname_c] = ops.linear_wgrad(dctc[:, :V], mem, out=g.out(wname_c), accumulate=acc)
        g.put('assistor.output_layer.bias', ops.colsum(dctc)[:V])
        wc_t = torch.zeros(d, dctc.shape[1], dtype=BF16, device=dev)
        wc_t[:, :V] = wc.t()
        dx = ops.linear(dctc, wc_t, None, EPI_RESID, resid=dmem)
    if pk.enc_pre:
        dx = _ln_bwd(dx, enc_last, pk.enc_norm[0], g, 'encoder.norm.weight', 'encoder.norm.bias')
    for i in reversed(range(len(pk.enc))):
        p, pre = pk.enc[i], f'encoder.blocks.{i}.'
        rt, st0 = e_rates[i], ENC_SITE + 2 * i
        if pk.enc_pre:
            (x0, qkv, ctx, lse, z1, x1, u, h, xn) = enc_tape[i]
            dh = _linear_bwd(_drop_bwd(dx, rt, drop_seed, st0 + 1), h, p['w2'][1], g, pre + 'feed_forward.w_2.weight', pre + 'feed_forward.w_2.bias')
            du = _ffn_act_bwd(p, dh, u, h)
            dx1 = _linear_bwd(du, x1, p['w1'][1], g, pre + 'feed_forward.w_1.weight', pre + 'feed_forward.w_1.bias', resid=dx)
            dz1 = _ln_bwd(dx1, z1, p['ln2'][0], g, pre + 'norm2.weight', pre + 'norm2.bias')
            dctx = _linear_bwd(_drop_bwd(dz1, rt, drop_seed, st0), ctx, p['o'][1], g, pre + 'slf_attn.output_proj.weight', pre + 'slf_attn.output_proj.bias')
            dqkv = torch.empty_like(qkv)
            ops.attention_bwd(qkv, qkv, qkv, ctx, dctx, lse, B, H, T2, T2, dqkv, dqkv, dqkv, kv_len=lengths, q_col0=0, k_col0=d,
                              v_col0=2 * d, dq_col0=0, dk_col0=d, dv_col0=2 * d)
            dxn = _linear_bwd(dqkv, xn, p['qkv'][1], g, pre + 'slf_attn.qvk_proj.weight', pre + 'slf_attn.qvk_proj.bias', resid=dz1)
            dx = _ln_bwd(dxn, x0, p['ln1'][0], g, pre + 'norm1.weight', pre + 'norm1.bias')
            continue
        (x0, qkv, ctx, lse, z1, x1, u, h, z2) = enc_tape[i]
        dz2 = _ln_bwd(dx, z2, p['ln2'][0], g, pre + 'norm2.weight', pre + 'norm2.bias')
        dh = _linear_bwd(_drop_bwd(dz2, rt, drop_seed, st0 + 1), h, p['w2'][1], g, pre + 'feed_forward.w_2.weight', pre + 'feed_forward.w_2.bias')
        du = _ffn_act_bwd(p, dh, u, h)
        dx1 = _linear_bwd(du, x1, p['w1'][1], g, pre + 'feed_forward.w_1.weight', pre + 'feed_forward.w_1.bias', resid=dz2)
        dz1 = _ln_bwd(dx1, z1, p['ln1'][0], g, pre + 'norm1.weight', pre + 'norm1.bias')
        dctx = _linear_bwd(_drop_bwd(dz1, rt, drop_seed, st0), ctx, p['o'][1], g, pre + 'slf_attn.output_proj.weight', pre + 'slf_attn.output_proj.bias')
        dqkv = torch.empty_like(qkv)
        ops.attention_bwd(qkv, qkv, qkv, ctx, dctx, lse, B, H, T2, T2, dqkv, dqkv, dqkv, kv_len=lengths, q_col0=0, k_col0=d,
                          v_col0=2 * d, dq_col0=0, dk_col0=d, dv_col0=2 * d)
        dx = _linear_bwd(dqkv, x0, p['qkv'][1], g, pre + 'slf_attn.qvk_proj.weight', pre + 'slf_attn.qvk_proj.bias', resid=dz1)

    # front end: x = (h2 Wo^T + bo) * sqrt(d) + PE  ->  conv2 (implicit-GEMM forward, im2col GEMMs backward) -> conv1
    dyl = ops.scale_add_table(dx, scale)                                          # d(h2 Wo^T + bo) = sqrt(d) * dx
    D_out = fe.output_size
    dwo = ops.linear_wgrad(dyl, h2)                                               # [D, F2*C2], feature index f*C2 + c
    g.put('frontend.output_layer.weight', dwo.view(D_out, F2, C2).permute(0, 2, 1).reshape(D_out, C2 * F2))
    g['frontend.output_layer.bias'] = ops.colsum(dyl, out=g.out('frontend.output_layer.bias'), accumulate=acc)
    dh2 = ops.linear(dyl, fpk['wo_t'])                                            # [B*T2, F2*C2]
    dpre2 = ops.relu_bwd(dh2, h2).view(B * T2 * F2, C2)
    col = ops.conv_im2col(h1, B, T, F, C1p)
    C1 = fe.conv1.conv_layer.out_channels
    dw2 = ops.linear_wgrad(dpre2, col)                                            # [C2, 9*C1p], k = (kh*3+kw)*C1p + c
    g.put('frontend.conv2.conv_layer.weight', dw2.view(C2, 3, 3, C1p)[..., :C1].permute(0, 3, 1, 2))
    g['frontend.conv2.conv_layer.bias'] = ops.colsum(dpre2, out=g.out('frontend.conv2.conv_layer.bias'), accumulate=acc)
    dcol = ops.linear(dpre2, fpk['w2_t'])                                         # [B*T2*F2, 9*C1p]
    del col
    dpre1 = ops.conv_col2im_relu(dcol, h1, B, T, F, C1p)
    g1 = ops.conv1_wgrad(dpre1, x_in, B, T, F, C1p)                               # [C1p, 9 taps + bias]
    g.put('frontend.conv1.conv_layer.weight', g1[:C1, :9].reshape(C1, 1, 3, 3))
    g.put('frontend.conv1.conv_layer.bias', g1[:C1, 9])
    return (loss, g, loss_ctc) if return_ctc else (loss, g)


class _SpeechToTextLoss(torch.autograd.Function):
    """loss = SpeechToText.forward(...) as ONE autograd node over the fp32 master parameters."""

    @staticmethod
    def forward(ctx, model, inputs, mask, truth, tlen, names, *params):
        with torch.no_grad():
            seed = getattr(model, '_drop_seed', None)
            if seed is None or seed.device != inputs.device:      # a fresh dropout mask per training forward
                seed = torch.randint(0, 2 ** 31 - 1, (1,), dtype=torch.int32).to(inputs.device)
                model._drop_seed = seed
            seed.add_(1)
            loss, grads, ctc = forward_backward(model, inputs, mask, truth, drop_seed=seed, truth_length=tlen, return_ctc=True)
        ctx.grads = [grads.get(n) for n in names]
        ctx.shapes = [p.shape for p in params]
        model._last_ctc_loss = ctc
        return loss.clone()

    @staticmethod
    def backward(ctx, gloss):
        out = []
        for gr, shp in zip(ctx.grads, ctx.shapes):
            out.append(None if gr is None else (gr.view(shp) * gloss))
        return (None, None, None, None, None, None) + tuple(out)


def loss_with_grad(model, inputs, mask, truth, truth_length=None):
    """Training-mode SpeechToText.forward: (loss tensor whose .backward() fills `.grad` of every parameter, CTC loss or None)."""
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    names = [n for n, _ in named]
    loss = _SpeechToTextLoss.apply(model, inputs, mask, truth, truth_length, names, *[p for _, p in named])
    return loss, getattr(model, '_last_ctc_loss', None)


def transformer_lr(step, model_size, warmup_steps, factor=1.0):
    """TransformerScheduler.get_step_lr (otrans/train/scheduler.py:137-138)."""
    return factor * model_size ** (-0.5) * min(step ** (-0.5), step * warmup_steps ** (-1.5))


class FusedTrainer:
    """The inner step of Trainer.train_one_epoch (trainer.py:206-234) on flat fp32 buffers:
    forward + hand-written backward -> (data-parallel) gradient all-reduce over NCCL -> global-norm clip + Adam in two
    kernels, no host synchronisation.  Parameters become views into one flat buffer (state_dict keys / shapes unchanged)."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.98), eps=1e-9, weight_decay=1e-6, clip_grad=5.0, model_size=256,
                 warmup_steps=12000, factor=1.0, accum_steps=1, process_group=None, use_graph=True):
        self.model = model
        self.params = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
        dev = self.params[0][1].device
        total = sum(p.numel() for _, p in self.params)
        self.flat_p = torch.empty(total, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(total, dtype=torch.float32, device=dev)
        self.m = torch.zeros(total, dtype=torch.float32, device=dev)
        self.v = torch.zeros(total, dtype=torch.float32, device=dev)
        self.sumsq = torch.zeros(1, dtype=torch.float32, device=dev)
        self.flat_bf16 = torch.empty(total, dtype=BF16, device=dev)      # ONE cast of the master weights per micro-step
        self.offsets = {}
        o = 0
        with torch.no_grad():
            for n, p in self.params:
                k = p.numel()
                self.flat_p[o:o + k].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[o:o + k].view_as(p)            # parameters now alias the flat buffer
                self.offsets[n] = (o, k)
                o += k
        self.sink = {n: self.flat_g[o:o + k].view_as(p) for (n, p), (o, k) in zip(self.params, [self.offsets[n] for n, _ in self.params])}
        self._by_ptr = {p.data_ptr(): (self.offsets[n], p.shape) for n, p in self.params}
        self.betas, self.eps, self.wd, self.clip = betas, eps, weight_decay, clip_grad
        self.base_lr, self.model_size, self.warmup, self.factor = lr, model_size, warmup_steps, factor
        self.accum_steps = accum_steps
        self.group = process_group
        # BaseScheduler starts at global_step 1 and its constructor already calls step() once (scheduler.py:22,42-46);
        # the trainer steps it again before every optimizer.step() (trainer.py:232): the first update uses lr(3)
        # The counts live on the DEVICE ({optimizer steps, scheduler global_step, skipped}): the fused Adam launch advances them
        # only when the gradient norm is finite, as the reference skips scheduler.step() together with optimizer.step()
        # (trainer.py:229-233) -- no host sync, and a skipped step cannot desynchronise the LR schedule / bias correction.
        self.counters = torch.tensor([0, 2, 0], dtype=torch.int32, device=dev)
        self.hyper = torch.zeros(4, dtype=torch.float32, device=dev)
        self.micro = 0
        # dropout seed of the current micro-step, on the device: incremented inside the (captured) micro-step, so every
        # CUDA-graph replay draws fresh masks (a seed passed by value would be frozen into the graph)
        self.drop_seed = torch.randint(0, 2 ** 31 - 1, (1,), dtype=torch.int32).to(dev)
        self.use_graph = use_graph
        self.graph_after = 2          # capture a CUDA graph for an input geometry once it has been seen this many times
        self.max_graphs = 8           # LRU bound: every graph owns a private pool with the whole activation tape
        self._graphs = {}             # key -> (graph, inputs, mask, truth, loss, launches), most recently used last
        self._seen = {}

    @property
    def opt_steps(self):
        return int(self.counters[0].item())

    @property
    def global_step(self):
        return int(self.counters[1].item())

    @property
    def skipped_steps(self):
        return int(self.counters[2].item())

    def lr(self):
        if self.warmup:
            return transformer_lr(self.global_step, self.model_size, self.warmup, self.factor)
        return self.base_lr

    def _bf16_of(self, param):
        (o, k), shape = self._by_ptr[param.data_ptr()]
        return self.flat_bf16[o:o + k].view(shape)

    def _micro(self, inputs, mask, truth, tlen=None):
        """forward + backward of one micro-batch; gradients / accum_steps are ADDED into the flat buffer by the backward
        kernels themselves (no per-parameter add)."""
        self.flat_bf16.copy_(self.flat_p)
        self.drop_seed.add_(1)
        loss, _ = forward_backward(self.model, inputs, mask, truth, grad_sink=self.sink, grad_scale=1.0 / self.accum_steps,
                                   bf16_of=self._bf16_of, drop_seed=self.drop_seed, truth_length=tlen)
        return loss

    def _graph_for(self, inputs, mask, truth, tlen=None):
        """The ~870 launches of one micro-batch captured once per input geometry and replayed: launched one by one from
        Python the step is host-bound (14.6 ms against 10.2 ms of kernel time, profiles/r1_launches_train_v0.csv).
        Real ASR batches have a new (T, L) almost every step, so a geometry runs EAGERLY until it has recurred
        `graph_after` times, and at most `max_graphs` graphs are kept (least recently used first out): use_graph pays off
        with bucketed / padded batches (otrans/data/bucket.py), it must not grow memory without bound otherwise.
        Returns None when this call should run eagerly."""
        key = (tuple(inputs.shape), tuple(truth.shape), inputs.device.index)
        ent = self._graphs.pop(key, None)
        if ent is None:
            n = self._seen.get(key, 0) + 1
            if len(self._seen) > 4096:
                self._seen.clear()
            self._seen[key] = n
            if n < self.graph_after:
                return None
            while len(self._graphs) >= self.max_graphs:
                self._graphs.pop(next(iter(self._graphs)))        # drops the graph and its memory pool
            sx, sm, st = inputs.clone(), mask.clone(), truth.clone()
            stl = tlen.to(torch.int32).to(inputs.device).clone() if tlen is not None else None
            snap = self.flat_g.clone()
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):          # warm-up outside capture: lazy kernel attributes, cached tables
                self._micro(sx, sm, st, stl)
            cur.wait_stream(side)
            self.flat_g.copy_(snap)
            graph = torch.cuda.CUDAGraph()
            n0 = ops.COUNTERS['launches']
            with torch.cuda.graph(graph):
                loss = self._micro(sx, sm, st, stl)
            launches = ops.COUNTERS['launches'] - n0
            ops.COUNTERS['launches'] = n0           # capture records, it does not launch
            ent = (graph, sx, sm, st, loss, launches, stl)
        self._graphs[key] = ent       # (re-)insert as most recently used
        return ent

    def step(self, inputs, mask, truth, truth_length=None):
        """One micro-batch; every `accum_steps` calls an optimizer step.  Returns the (un-scaled) loss tensor.
        truth_length (targets['targets_length']) is needed by joint-CTC models only."""
        with torch.no_grad():
            ent = self._graph_for(inputs, mask, truth, truth_length) if self.use_graph else None
            if ent is not None:
                graph, sx, sm, st, loss, launches, stl = ent
                sx.copy_(inputs)
                sm.copy_(mask)
                st.copy_(truth)
                if stl is not None:
                    stl.copy_(truth_length)
                graph.replay()
                ops.COUNTERS['launches'] += launches
            else:
                loss = self._micro(inputs, mask, truth, truth_length)
            self.micro += 1
            if self.micro % self.accum_steps == 0:
                # the one exchange step of data-parallel training (SURVEY.md 8e): mean of the flat gradient over ranks,
                # ONE NCCL all-reduce per optimizer step (the reference's DDP reduces on every micro-batch)
                allreduce_mean_(self.flat_g, self.group)
                ops.sumsq(self.flat_g, self.sumsq)
                ops.adam_step_sched(self.flat_p, self.flat_g, self.m, self.v, self.sumsq, self.clip, self.base_lr, self.model_size,
                                    self.warmup, self.factor, self.betas, self.eps, self.wd, self.counters, self.hyper)
                self.flat_g.zero_()
                modules.bump_param_generation()     # bf16 shadow copies (modules._Packed) must be rebuilt
        return loss
