"""Batched beam-search recogniser on the B200 hot path.

Mirror of otrans/recognize/speech2text.py (SpeechToTextRecognizer) and the bits of
otrans/recognize/base.py it needs.  Same constructor, same ``recognize`` / ``encode`` / ``decode`` /
``decode_step`` seams and return types.  What changes underneath:

  * encode: conv front end + encoder run as hand-written sm_100a kernels (bf16 tensor cores);
  * decode: the reference re-runs the whole decoder over the whole prefix -- and the cross-attention
    K/V projection of the beam-tiled memory -- at every step (decoder/transformer.py:204,
    attention.py:129).  Here cross K/V are projected ONCE per utterance (shared by the beams), self-attention
    K/V live in a per-hypothesis cache addressed through a 4-byte ancestry table, and one step is
    a fixed sequence of kernels captured in a CUDA graph and replayed;
  * beam step: one kernel per step (top-k, finished masking, pruning, back-pointers), no host sync
    inside the loop except a 4-byte "all ended" poll every few steps.
"""
import torch

from . import ops
from .modules import _lengths, _ffn, _proj_resid_ln

PAD, BOS, EOS = 0, 1, 1   # otrans/data/__init__.py:7-10


class Recognizer:
    """otrans/recognize/base.py:5-24,91-119 (model holder + id -> string translation)."""

    def __init__(self, model, idx2unit=None, lm=None, lm_weight=None, ngpu=1):
        self.ngpu = ngpu
        self.model = model
        self.model.eval()
        if self.ngpu > 0:
            self.model.cuda()
        self.lm = lm
        if self.lm is not None:
            self.lm.eval()
            if self.ngpu > 0:
                self.lm.cuda()
        self.idx2unit = idx2unit
        self.lm_weight = lm_weight

    def lm_decode(self, preds, hidden=None):
        """recognize/base.py:26-37 (Transformer LM branch)."""
        return self.lm.predict(preds, last_frame=True), hidden

    def translate(self, seqs):
        results = []
        for seq in seqs:
            pred = []
            for i in seq:
                if int(i) == EOS:
                    break
                if int(i) == PAD:
                    continue
                pred.append(self.idx2unit[int(i)])
            results.append(' '.join(pred))
        return results

    def nbest_translate(self, nbest_preds):
        assert nbest_preds.dim() == 3
        if self.idx2unit is None:          # ids requested (tests / benchmarks): keep the tensor
            return nbest_preds
        rows = nbest_preds.cpu().tolist()
        results = []
        for per_utt in rows:
            nbest_list = []
            for seq in per_utt:
                pred = []
                for token in seq:
                    if token == EOS:
                        break
                    pred.append(self.idx2unit[token])
                nbest_list.append(' '.join(pred))
            results.append(nbest_list)
        return results


class BeamDecoder:
    """KV-cached incremental decoder + device-side beam search for one (batch, beam, T, max_len) shape.

    Buffers are allocated once; one decode step (decoder on the newest token -> log-softmax -> beam
    kernel) is captured into a CUDA graph on first use and replayed for every step.
    """

    def __init__(self, decoder, batch, beam, T, max_len, device, use_graph=True, persistent=False, keep_logp=None):
        self.dec = decoder
        self.B, self.beam, self.T, self.Lmax = batch, beam, T, max_len
        self.N = batch * beam
        self.device = device
        d, nl = decoder.d_model, len(decoder.blocks)
        self.state = ops.BeamState(batch, beam, max_len, device)
        self.kc = torch.zeros(nl, max_len, self.N, d, dtype=ops.BF16, device=device)
        self.vc = torch.zeros(nl, max_len, self.N, d, dtype=ops.BF16, device=device)
        self.kvx = torch.zeros(nl, batch * T, 2 * d, dtype=ops.BF16, device=device)  # cross K|V per utterance
        self.mem_len = torch.zeros(batch, dtype=torch.int32, device=device)
        self.table = ops.sinusoid_table(max_len + 1, d, 0, device)
        self.logits = torch.zeros(self.N, decoder.ld_logits, dtype=torch.float32, device=device)
        self.logp = torch.zeros(self.N, decoder.vocab_size, dtype=torch.float32, device=device)
        self.topk_val = torch.zeros(self.N, beam, dtype=torch.float32, device=device)
        self.topk_idx = torch.zeros(self.N, beam, dtype=torch.int32, device=device)
        # eager (test / debug) mode also materialises the full log-probs; keep_logp=True does so on the graph path (parity traces)
        self.keep_logp = (not use_graph) if keep_logp is None else bool(keep_logp)
        self.use_graph = use_graph
        self.graph = None
        self._graph_pk = None      # the bf16 weight pack whose device pointers the captured graph bakes in (kept alive with it)
        self.lm_logp = None
        self.lm_weight = 0.0
        if decoder.pos_emb.scale_learnable:
            raise NotImplementedError('decoder with learnable positional scale')
        # persistent path: the whole loop in ONE launch (csrc/decode_group.cu: row groups of <= 128 hypotheses x 16 CTAs,
        # tcgen05 GEMMs, group-local barriers) when the configuration is the shipped one (post-norm GLU decoder, d_model 256,
        # 4 heads, d_ff 2048, <= 256 memory frames); anything else takes the per-step graph.
        self.persistent = bool(persistent) and self.mega_supported()
        self._mega_model = None
        self._mega_sig = None
        self._ws = None

    def mega_supported(self):
        dec = self.dec
        groups = -(-self.B // max(1, 128 // self.beam))
        ok = (dec.d_model == 256 and dec.n_heads == 4 and not dec.normalize_before and 1 <= len(dec.blocks) <= 8
              and self.beam <= 16 and self.Lmax <= 128 and dec.vocab_size >= 16 and self.T <= 256
              and groups * 16 <= ops.num_sms())
        for blk in dec.blocks:
            ff = blk.feed_forward
            ok = ok and ff.activation == 'glu' and ff.w_2.in_features == 2048 and not blk.normalize_before
            ok = ok and all(m.bias is not None for m in (blk.slf_attn.qvk_proj, blk.slf_attn.output_proj, blk.src_attn.q_proj,
                                                         blk.src_attn.output_proj, ff.w_1, ff.w_2))
        return bool(ok)

    def _mega(self):
        """otb_mega_model over the packed bf16 weights (rebuilt when the pack changes)."""
        pk = self.dec.packed()
        if self._mega_model is None or self._mega_sig is not pk:
            from ._lib import MegaModelC
            m = MegaModelC()
            m.n_layers, m.d_model, m.n_heads = len(self.dec.blocks), self.dec.d_model, self.dec.n_heads
            m.d_ff, m.vocab = self.dec.blocks[0].feed_forward.w_2.in_features, self.dec.vocab_size
            m.emb, m.wout = pk['emb'].data_ptr(), pk['wout'].data_ptr()
            m.bout = pk['bout'].data_ptr() if pk['bout'] is not None else None
            m.pe = self.table.data_ptr()
            m.ln_eps = 1e-5
            for l, p in enumerate(pk['blocks']):
                ly = m.layers[l]
                f = p['ffn']
                for name, t in (('wqkv', p['wqkv']), ('wo', p['wo']), ('wq', p['wq']), ('wo2', p['wo2']), ('w1', f['w1']),
                                ('w2', f['w2']), ('bqkv', p['bqkv']), ('bo', p['bo']), ('bq', p['bq']), ('bo2', p['bo2']),
                                ('b1', f['b1']), ('b2', f['b2']), ('g1', p['ln1'][0]), ('be1', p['ln1'][1]),
                                ('g2', p['ln2'][0]), ('be2', p['ln2'][1]), ('g3', p['ln3'][0]), ('be3', p['ln3'][1])):
                    setattr(ly, name, t.data_ptr())
            self._mega_model, self._mega_sig = m, pk
        return self._mega_model

    def run_persistent(self, max_steps, dbg_logp=None, dbg_scores=None):
        """All steps in ONE launch; no host round trip (ctrl[0] = executed steps is read by the caller)."""
        if self._ws is None:
            self._ws = ops.decode_persistent_workspace(self.N, len(self.dec.blocks), self.Lmax, self.B, self.beam,
                                                       self.dec.vocab_size, self.device)
        ops.decode_persistent(self._mega(), self.kvx, self.mem_len, self.kc, self.vc, self.state, self.B, self.T, max_steps,
                              self._ws, dbg_logp, dbg_scores)

    def setup(self, memory_bf16, mem_len):
        """Project cross-attention K/V once per utterance and reset the search state."""
        pk = self.dec.packed()
        self.mem_len.copy_(mem_len)
        for l, p in enumerate(pk['blocks']):
            ops.linear(memory_bf16, p['wkv'], p['bkv'], out=self.kvx[l])
        self.state.init()

    def _step_kernels(self):
        dec, st = self.dec, self.state
        pk = dec.packed()
        d, H, N = dec.d_model, dec.n_heads, self.N
        x = ops.embed_posenc(st.last_tok, pk['emb'], self.table, N, d, step_ptr=st.step_ptr)
        for l, (blk, p) in enumerate(zip(dec.blocks, pk['blocks'])):
            nb = blk.normalize_before
            if nb:
                x = ops.layernorm(x, *p['ln1'])
            qkv = ops.linear(x, p['wqkv'], p['bqkv'])
            ctx = ops.decode_self_attn(qkv, self.kc[l], self.vc[l], st.anc, st.step_ptr, N, H, self.Lmax, head_dim=dec.head_dim)
            x = _proj_resid_ln(ctx, p['wo'], p['bo'], x, None if nb else p['ln1'])
            if nb:
                x = ops.layernorm(x, *p['ln2'])
            q = ops.linear(x, p['wq'], p['bq'])
            # the `beam` hypotheses of utterance b are the query rows [b*beam, (b+1)*beam) of one attention problem
            # (a SIMT kernel specialised for <= 16 query rows was measured at 14.9 us against 10.0 us for this tcgen05 kernel
            # padded to 128 rows and was dropped: profiles/r1_bench_history.md)
            ctx = ops.attention(q, self.kvx[l], self.kvx[l], self.B, H, self.beam, self.T, kv_len=self.mem_len,
                                k_col0=0, v_col0=d, head_dim=dec.head_dim)
            x = _proj_resid_ln(ctx, p['wo2'], p['bo2'], x, None if nb else p['ln2'])
            if nb:
                x = ops.layernorm(x, *p['ln3'])
            x = _ffn(x, p['ffn'], x, None if nb else p['ln3'])
        if dec.normalize_before:
            x = ops.layernorm(x, *pk['after'])
        ops.linear(x, pk['wout'], pk['bout'], out=self.logits)
        ops.logsoftmax_topk(self.logits, dec.vocab_size, self.beam, self.lm_logp, self.lm_weight,
                            out_val=self.topk_val, out_idx=self.topk_idx,
                            out_logp=self.logp if self.keep_logp else None)
        st.step_topk(self.topk_val, self.topk_idx)

    def step(self):
        if not self.use_graph:
            return self._step_kernels()
        if self.graph is not None and self._graph_pk is not self.dec.packed():
            # parameters changed (load_state_dict / optimizer step): the pack was rebuilt at new addresses, the captured
            # kernels would read the old (stale or recycled) weights -- drop the graph and capture again
            self.graph = None
        if self.graph is None:
            self._graph_pk = self.dec.packed()
            # warm-up outside capture (lazy func attributes, caches), then restore the state it advanced
            snap = [t.clone() for t in (self.state.tok_hist, self.state.par_hist, self.state.last_tok,
                                        self.state.scores, self.state.flag, self.state.anc, self.state.ctrl)]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._step_kernels()
            torch.cuda.current_stream().wait_stream(s)
            for t, c in zip((self.state.tok_hist, self.state.par_hist, self.state.last_tok, self.state.scores,
                             self.state.flag, self.state.anc, self.state.ctrl), snap):
                t.copy_(c)
            self.graph = torch.cuda.CUDAGraph()
            n0 = ops.COUNTERS['launches']
            with torch.cuda.graph(self.graph):
                self._step_kernels()
            self.launches_per_step = ops.COUNTERS['launches'] - n0
            ops.COUNTERS['launches'] = n0                      # capture records, it does not launch
            for t, c in zip((self.state.tok_hist, self.state.par_hist, self.state.last_tok, self.state.scores,
                             self.state.flag, self.state.anc, self.state.ctrl), snap):
                t.copy_(c)
        self.graph.replay()
        ops.COUNTERS['launches'] += self.launches_per_step

    def run_with_lm(self, max_steps, lm, lm_weight):
        """Shallow fusion (speech2text.py:102-105, base.py:26-37): every step the LM re-scores the full prefixes
        (as the reference's TransformerLanguageModel.predict does) and lm_weight * log-probs are added inside the
        fused log-softmax/top-k kernel.  Eager mode: the prefix length is host-side state."""
        assert not self.use_graph, 'LM fusion runs the decode loop eagerly'
        self.lm_weight = float(lm_weight)
        for i in range(max_steps):
            preds = self.state.reconstruct(i)                       # [N, i+1], column 0 = BOS
            self.lm_logp = lm.predict(preds, last_frame=True).squeeze(1).contiguous()
            self._step_kernels()
            if int(self._read_ctrl()[1]):
                break
        self.lm_logp = None
        return int(self._read_ctrl()[0])

    def _read_ctrl(self):
        """{step, done, ...} of the search state on the host.  The copy lands in pinned memory and the thread SLEEPS on a
        blocking-sync event instead of spinning in cudaStreamSynchronize (`.item()`): a server keeps many of these loops
        alive on few cores (16 lanes x 8 ranks on one host in bench.py)."""
        if getattr(self, '_ctrl_pin', None) is None:
            self._ctrl_pin = torch.zeros(4, dtype=torch.int32).pin_memory()
            self._ctrl_ev = torch.cuda.Event(blocking=True)
        self._ctrl_pin.copy_(self.state.ctrl, non_blocking=True)
        self._ctrl_ev.record()
        self._ctrl_ev.synchronize()
        return self._ctrl_pin

    def run(self, max_steps, poll_every=8):
        """Run up to max_steps decode steps; stops early once the device reports every hypothesis ended
        (speech2text.py:66-67).  Steps launched after the end are no-ops on the search state.
        (A sync-free variant -- the flag copied asynchronously to pinned memory and inspected one poll later -- shortened a
        lone decode by 0.5 ms but cost 8 concurrent lanes 18 % of their throughput: free-running lanes fall into lockstep
        and queue for the same SMs, whereas this 4-byte poll staggers them.  profiles/r1_bench_history.md)"""
        if self.persistent and self.lm_logp is None:
            self.run_persistent(max_steps)
            return int(self._read_ctrl()[0])
        for i in range(max_steps):
            self.step()
            if (i + 1) % poll_every == 0 and i + 1 < max_steps:
                if int(self._read_ctrl()[1]):
                    break
        return int(self._read_ctrl()[0])


class SpeechToTextRecognizer(Recognizer):
    """otrans/recognize/speech2text.py:6-93 on the B200 path."""

    def __init__(self, model, lm=None, lm_weight=0.1, ctc_weight=0.0, beam_width=5, nbest=1, max_len=50,
                 idx2unit=None, penalty=0, lamda=5, ngpu=1, apply_cache=False, use_graph=True, persistent=None):
        super().__init__(model, idx2unit, lm, lm_weight, ngpu)
        if lm is not None and getattr(lm, 'model_type', None) != 'transformer_lm':
            raise NotImplementedError('shallow fusion is implemented for the Transformer LM (opentransformer_b200.lm); '
                                      'the RNN LM is out of scope')
        self.beam_width, self.max_len, self.nbest = beam_width, max_len, nbest
        self.penalty, self.lamda = penalty, lamda
        self.ctc_weight, self.lm_weight = ctc_weight, lm_weight
        self.attn_weights = {}
        self.apply_cache = False
        self.use_graph = use_graph
        # None = automatic: the persistent decode kernel (one launch per batch, csrc/decode_group.cu) whenever the decoder,
        # the batch geometry and the options (no LM fusion) fit it; False forces the per-step CUDA-graph path
        self.persistent = True if persistent is None else bool(persistent)
        self._decoders = {}

    # ---- reference-facing seams -------------------------------------------------------------
    def encode(self, inputs, inputs_mask, cache=None):
        mem, mem_len, B, T2 = self._encode_bf16(inputs, inputs_mask)
        memory = mem.float().view(B, T2, -1)
        return memory, self.model.frontend.output_mask(inputs_mask), {'frontend': None}, {}

    def decode(self, preds, memory, memory_mask, cache=None):
        return self.model.decoder.inference(preds, memory, memory_mask, cache)

    def decode_step(self, preds, memory, memory_mask, cache, scores, flag):
        """One reference-style step on caller-owned tensors (speech2text.py:95-153): decoder.inference + the CUDA beam
        kernel.  With cache['decoder'] = model.decoder.init_cache(memory, mask, max_len, beam) the decoder runs KV-cached
        (one token per call) and the cache is reordered by the surviving hypotheses' parents -- the feature the reference
        left as a stub (decoder/transformer.py:188-203, reselect_hidden* :195-218); with None it recomputes the full prefix
        like the reference.  The fast path used by recognize() is BeamDecoder."""
        from .modules import DecoderCache
        n = scores.size(0)
        batch = n // self.beam_width
        dcache = cache.get('decoder') if isinstance(cache, dict) else None
        log_probs, dcache, _ = self.decode(preds, memory, memory_mask, dcache)
        st = ops.BeamState(batch, self.beam_width, 1, scores.device)
        st.init()
        st.scores.copy_(scores.view(-1))
        st.flag.copy_(flag.view(-1).to(torch.uint8))
        lm_logp, lm_w = None, 0.0
        if self.lm is not None and self.lm_weight:
            lm_logp = self.lm.predict(preds, last_frame=True).squeeze(1).contiguous()
            lm_w = float(self.lm_weight)
        st.step(log_probs.contiguous(), log_probs.shape[-1], lm_logp, lm_w)
        parent = st.par_hist[0].long()
        tok = st.tok_hist[0].long()
        if isinstance(dcache, DecoderCache):
            dcache.reorder(parent)
        preds_symbol = torch.cat((preds.index_select(0, parent), tok.view(-1, 1)), dim=1)
        return preds_symbol, cache, st.scores.view(-1, 1).clone(), (tok == EOS).view(-1, 1)

    # ---- fast path ------------------------------------------------------------------------------
    def _encode_bf16(self, inputs, inputs_mask):
        fe, enc = self.model.frontend, self.model.encoder
        B, T, _ = inputs.shape
        _, _, T2, _ = ops.conv_geometry(T, fe.input_size)
        lengths = _lengths(fe.output_mask(inputs_mask))
        fused = getattr(enc, 'fuse_abs_posenc', None)
        if fused is not None and fused():
            scale, table = enc.pos_emb.scale_and_table(T2, inputs.device)
            x, _ = fe.forward_bf16(inputs, scale, table)
        else:
            x, _ = fe.forward_bf16(inputs)
            x = enc.apply_posenc_bf16(x, B, T2)
        mem = enc.forward_bf16(x, B, T2, lengths)
        return mem, lengths, B, T2

    def _decoder_for(self, B, T2, device):
        key = (B, self.beam_width, T2, self.max_len, device.index)
        bd = self._decoders.get(key)
        if bd is None:
            bd = BeamDecoder(self.model.decoder, B, self.beam_width, T2, self.max_len, device,
                             self.use_graph and self.lm is None, persistent=self.persistent and self.lm is None)
            self._decoders[key] = bd
        return bd

    def recognize_ids(self, inputs, inputs_mask):
        """-> (nbest ids i64 [B,nbest,steps], scores f32 [B,nbest], steps)"""
        with torch.no_grad():
            mem, mem_len, B, T2 = self._encode_bf16(inputs, inputs_mask)
            bd = self._decoder_for(B, T2, inputs.device)
            bd.setup(mem, mem_len)
            if self.lm is not None:
                steps = bd.run_with_lm(self.max_len, self.lm, self.lm_weight)
            else:
                steps = bd.run(self.max_len)
            preds, scores = bd.state.finalize(self.penalty, self.lamda, self.nbest)
        return preds[:, :, :steps], scores, steps

    def recognize(self, inputs, inputs_mask):
        preds, scores, _ = self.recognize_ids(inputs, inputs_mask)
        return self.nbest_translate(preds), scores


def build_recognizer(model_type, model, lm, args, idx2unit):
    """otrans/recognize/__init__.py:5-16 (speech2text only; CTC is out of scope, SURVEY.md 2)."""
    if model_type == 'speech2text':
        return SpeechToTextRecognizer(
            model=model, lm=lm, lm_weight=args.lm_weight, ctc_weight=args.ctc_weight, beam_width=args.beam_width,
            nbest=args.nbest, max_len=args.max_len, idx2unit=idx2unit, penalty=args.penalty, lamda=args.lamda,
            ngpu=args.ngpu)
    raise NotImplementedError(model_type)
