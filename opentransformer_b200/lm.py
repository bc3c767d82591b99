"""Transformer language model for shallow fusion on the B200 path.

Mirror of otrans/model/lm.py:93-171 (TransformerLanguageModel): embedding + sinusoidal positions +
``num_blocks`` post-norm TransformerEncoderLayers (GLU FFN) under a causal mask + tied output projection.
Same constructor (``params`` dict of the YAML ``model:`` section), ``state_dict`` keys and ``predict``
signature; the layers are the same sm_100a kernels as the acoustic encoder (causal flag on the attention
kernel).  The recogniser adds ``lm_weight * log_probs`` inside the fused log-softmax/top-k kernel
(recognize/speech2text.py:102-105 -> otb_logsoftmax_topk).  Inference only.
"""
import torch
import torch.nn as nn

from . import ops
from .modules import BF16, PositionalEncoding, TransformerEncoderLayer, _Packed, _b, _no_train, _w


class TransformerLanguageModel(nn.Module):
    def __init__(self, params):
        super().__init__()
        self.params = params
        self.model_type = 'transformer_lm'
        self.normalize_before = False
        self.smoothing = params.get('smoothing', 0.0)
        self.vocab_size = params['vocab_size']
        self.num_blocks = params['num_blocks']
        self.d_model = params['d_model']
        if self.d_model != params['n_heads'] * 64:
            # the layers would run at d_k = 96 too, but that LM path has no parity test yet
            raise NotImplementedError('TransformerLanguageModel: d_k = d_model / n_heads must be 64')
        self.embedding = nn.Embedding(self.vocab_size, self.d_model)
        self.pos_embedding = PositionalEncoding(self.d_model, 0.0)
        self.blocks = nn.ModuleList([
            TransformerEncoderLayer(params['n_heads'], self.d_model, params['d_ff'], slf_attn_dropout=0.0,
                                    ffn_dropout=0.0, residual_dropout=params.get('residual_dropout', 0.0),
                                    normalize_before=False, concat_after=False, activation='glu')
            for _ in range(self.num_blocks)])
        self.output_project = nn.Linear(self.d_model, self.vocab_size)
        if params.get('share_embedding', False):
            self.output_project.weight = self.embedding.weight
        self._pack = _Packed(self, self._build_pack)

    def _build_pack(self):
        emb = self.embedding.weight.detach().to(BF16).contiguous()
        tied = self.output_project.weight is self.embedding.weight
        return {'emb': emb, 'wout': emb if tied else _w(self.output_project), 'bout': _b(self.output_project),
                'blocks': [b.pack() for b in self.blocks]}

    @property
    def ld_logits(self):
        return (self.vocab_size + 7) // 8 * 8

    def logits_bf16(self, targets):
        """targets i64 [N,L] -> logits f32 [N*L, ld_logits] (full prefix, as the reference recomputes it)."""
        _no_train(self)
        pk = self._pack.get()
        N, L = targets.shape
        scale, table = self.pos_embedding.scale_and_table(L, targets.device)
        x = ops.embed_posenc(targets.contiguous(), pk['emb'], table, N * L, self.d_model, period=L)
        for blk, p in zip(self.blocks, pk['blocks']):
            x = blk.run(x, p, N, L, None, causal=True)
        return ops.linear(x, pk['wout'], pk['bout'], ops.EPI_BIAS, out_f32=True, n_out=self.ld_logits)

    def predict(self, targets, last_frame=True):
        """model/lm.py:143-163: log-probs [N,1,V] of the last position, or [N,L,V] of all positions."""
        N, L = targets.shape
        with torch.no_grad():
            logits = self.logits_bf16(targets).view(N, L, -1)
            if last_frame:
                last = logits[:, -1, :].contiguous()
                return ops.log_softmax(last, self.vocab_size).unsqueeze(1)
            flat = logits.reshape(N * L, -1)
            return ops.log_softmax(flat, self.vocab_size).view(N, L, self.vocab_size)

    def forward(self, inputs, targets):
        """model/lm.py:126-141, forward only: label-smoothed CE of the next-token prediction."""
        with torch.no_grad():
            logits = self.logits_bf16(inputs['inputs'])
            loss, _ = ops.ls_cross_entropy(logits, targets['targets'].contiguous(), self.vocab_size, self.smoothing)
        return loss, None

    def save_checkpoint(self, params, name):
        torch.save({'params': params, 'model': self.state_dict()}, name)


LanguageModel = {'transformer_lm': TransformerLanguageModel}
