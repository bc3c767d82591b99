"""GPU parity of the shipped Conformer recipe (conformer_baseline.yaml: d_model 384, 4 heads of width 96, d_ff 768 GLU,
rel-pos Conformer encoder, post-norm Transformer decoder, V = 4234) against the fp32 oracle:
  * 2 encoder + 2 decoder blocks: encoder states, teacher-forced decoder logits, the per-step graph decoder in lock-step
    with the oracle's beam_step (beam 4 and 10), recognize() (never the persistent kernel at d = 384) and the
    decode_step / DecoderCache seam;
  * full depth (12 encoder / 6 decoder blocks), 4 utterances x 1000 frames: encoder states and a 60-step lock-step search;
  * training a 96-wide model is refused (the attention backward is 64-wide).
Run with -m gpu on a B200."""
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from opentransformer_b200 import train
    from opentransformer_b200.model import SpeechToText
    from opentransformer_b200.recognize import SpeechToTextRecognizer, BeamDecoder
    DEV = torch.device('cuda:0')

from oracle import beam_search as obs
from oracle import speech_model as om
from tests.test_conformer_baseline_ref import conformer_baseline_params
from tests.test_gpu_model import _batch, _rel, _valid, REL_L2_STATES, REL_L2_LOGITS, MAX_ABS_FRAC


def _build(params, seed=1234):
    torch.manual_seed(seed)
    model = SpeechToText(params).eval()
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if 'norm' in n:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
            elif n.endswith('.bias'):
                p.add_(0.05 * torch.randn(p.shape, generator=g))
        for n, b in model.named_buffers():             # non-trivial BatchNorm running statistics
            if n.endswith('running_mean'):
                b.copy_(0.3 * torch.randn(b.shape, generator=g))
            if n.endswith('running_var'):
                b.copy_(1.0 + 0.5 * torch.rand(b.shape, generator=g))
        model.decoder.output_layer.bias[1] = -1e4          # <S/E> never wins: every step runs
    sd = {}
    for part in ('frontend', 'encoder', 'decoder'):
        for k, v in getattr(model, part).state_dict().items():
            sd[f'{part}.{k}'] = v.detach().clone().float() if v.dtype.is_floating_point else v.clone()
    return model.to(DEV), sd


@pytest.fixture(scope='module')
def small():
    params = conformer_baseline_params(n_enc=2, n_dec=2)
    model, sd = _build(params)
    x, mask = _batch(3, 400, 80, [400, 301, 233])
    return params, model, sd, x, mask


def test_conformer_baseline_encoder_states(small):
    params, model, sd, x, mask = small
    mem_ref, mmask = om.encode(x, mask, sd, params)
    with torch.no_grad():
        mem, lens, B, T2 = model.encode_bf16(x.to(DEV), mask.to(DEV))
        api, _, _ = model.encoder(*model.frontend(x.to(DEV), mask.to(DEV)))
    r = _rel(_valid(mem.float().view(B, T2, -1).cpu(), mmask), _valid(mem_ref, mmask))
    r_api = _rel(_valid(api.cpu(), mmask), _valid(mem_ref, mmask))
    print(f'conformer_baseline 2-block encoder states: rel_l2 fused={r:.3e} module-API={r_api:.3e}')
    assert lens.cpu().tolist() == mmask.sum(1).tolist()
    assert r < REL_L2_STATES and r_api < REL_L2_STATES


def test_conformer_baseline_decoder_logits_teacher_forced(small):
    params, model, sd, x, mask = small
    mem_ref, mmask = om.encode(x, mask, sd, params)
    g = torch.Generator().manual_seed(5)
    tgt = torch.randint(3, 4234, (3, 31), generator=g)
    tgt[:, 0] = 1
    kw = om.decoder_kwargs(params)
    logits_ref = om.transformer_decoder(tgt[:, :-1], mem_ref, mmask, sd, 'decoder.', **kw)
    with torch.no_grad():
        logits, _ = model.decoder(tgt[:, :-1].to(DEV), mem_ref.to(DEV), mmask.to(DEV))
        lp, _, _ = model.decoder.inference(tgt[:, :7].to(DEV), mem_ref.to(DEV), mmask.to(DEV), None)
    keep = [i for i in range(4234) if i != 1]
    lp_ref = om.decoder_inference(tgt[:, :7], mem_ref, mmask, sd, 'decoder.', **kw)
    r = _rel(logits.cpu()[..., keep], logits_ref[..., keep])
    r_lp = _rel(lp.cpu()[:, keep], lp_ref[:, keep])
    d_lp = float((lp.cpu()[:, keep] - lp_ref[:, keep]).abs().max())
    lim = MAX_ABS_FRAC * float(lp_ref[:, keep].abs().max())
    print(f'conformer_baseline decoder logits rel_l2={r:.3e}; inference log-probs rel_l2={r_lp:.3e} max_abs={d_lp:.3e} '
          f'(limit {lim:.3e})')
    assert r < REL_L2_LOGITS and r_lp < REL_L2_LOGITS and d_lp < lim


def _lockstep(bd, sd, params, mem, lens, B, beam, max_len, T2, check_every=1):
    """Feed the oracle's beam_step the CUDA decoder's log-probs after every graph step: ids, parents, score bit patterns
    and finished flags must be identical at every step."""
    memory = mem.float().view(B, T2, -1).cpu()
    mmask = torch.arange(T2)[None] < lens.cpu()[:, None]
    bm = memory.unsqueeze(1).repeat(1, beam, 1, 1).view(B * beam, T2, -1)
    bmask = mmask.unsqueeze(1).repeat(1, beam, 1).view(B * beam, T2)
    preds = torch.full((B * beam, 1), 1, dtype=torch.long)
    scores = torch.tensor([0.0] + [float('-inf')] * (beam - 1)).repeat(B).unsqueeze(1)
    flag = torch.zeros_like(scores, dtype=torch.bool)
    kw = om.decoder_kwargs(params)
    worst_rel = 0.0
    for s in range(max_len):
        bd.step()
        lp_gpu = bd.logp.cpu()
        alive = ~flag.view(-1)
        if s % check_every == 0:
            lp_ref = om.decoder_inference(preds, bm, bmask, sd, 'decoder.', **kw)
            worst_rel = max(worst_rel, _rel(lp_gpu[alive][:, 2:], lp_ref[alive][:, 2:]))
        preds, scores, flag = obs.beam_step(lp_gpu, preds, scores, flag, beam)
        assert torch.equal(bd.state.reconstruct(s + 1).cpu(), preds), f'token / parent ids differ at step {s}'
        assert torch.equal(bd.state.scores.cpu().view(torch.int32), scores.view(-1).view(torch.int32)), f'scores differ at step {s}'
        assert torch.equal(bd.state.flag.cpu().bool(), flag.view(-1)), f'finished flags differ at step {s}'
    return preds, scores, worst_rel


@pytest.mark.parametrize('beam', [4, 10])
def test_conformer_baseline_graph_path_lockstep(small, beam):
    params, model, sd, x, mask = small
    B, max_len = 3, 8
    with torch.no_grad():
        mem, lens, _, T2 = model.encode_bf16(x.to(DEV), mask.to(DEV))
        bd = BeamDecoder(model.decoder, B, beam, T2, max_len, DEV, use_graph=True, keep_logp=True)
        assert not bd.mega_supported() and not bd.persistent
        bd.setup(mem, lens)
        preds, scores, worst_rel = _lockstep(bd, sd, params, mem, lens, B, beam, max_len, T2)
        assert bd.graph is not None
    print(f'conformer_baseline graph path beam {beam}: {max_len} steps identical; log-probs rel_l2<={worst_rel:.3e}')
    assert worst_rel < REL_L2_LOGITS
    nb, ns = obs.beam_finalize(preds, scores, beam, 1, 0.6, 5)
    gp, gs = bd.state.finalize(0.6, 5, 1)
    assert torch.equal(gp[:, :, :max_len].cpu(), nb)
    torch.testing.assert_close(gs.cpu(), ns, rtol=1e-5, atol=1e-5)


def test_conformer_baseline_recognize_takes_graph_path_and_matches_bf16_oracle(small):
    params, model, sd, x, mask = small
    beam, max_len = 4, 8
    rec = SpeechToTextRecognizer(model, beam_width=beam, nbest=1, max_len=max_len, penalty=0.6, lamda=5, ngpu=1)
    ids, sc, n = rec.recognize_ids(x.to(DEV), mask.to(DEV))
    assert n == max_len
    assert not any(bd.persistent for bd in rec._decoders.values()), 'd_model 384 must take the per-step graph decoder'
    out, scores = rec.recognize(x.to(DEV), mask.to(DEV))
    assert torch.equal(out, ids)
    nb_ref, ns_ref, _, _ = obs.recognize(x, mask, sd, params, beam=beam, nbest=1, max_len=max_len, penalty=0.6, lamda=5,
                                         policy='bf16')
    print(f'conformer_baseline recognize(): 1-best {ids[:, 0].tolist()} vs bf16 oracle {nb_ref[:, 0].tolist()}; '
          f'scores {sc.view(-1).tolist()} vs {ns_ref.view(-1).tolist()}')
    assert torch.equal(ids[:, 0].cpu(), nb_ref[:, 0])
    torch.testing.assert_close(sc.cpu(), ns_ref, rtol=3e-2, atol=0.3)


def test_conformer_baseline_decoder_cache_seam(small):
    """decoder.inference(preds, memory, mask, cache) with a DecoderCache and decode_step's reordering, against the
    full-prefix recompute of the same seam and the oracle in lock-step."""
    params, model, sd, x, mask = small
    B, beam, max_len = 3, 4, 6
    rec = SpeechToTextRecognizer(model, beam_width=beam, nbest=1, max_len=max_len, penalty=0.6, lamda=5, ngpu=1)
    memory, mmask, _, _ = rec.encode(x.to(DEV), mask.to(DEV))
    T2 = memory.shape[1]
    bm = memory.unsqueeze(1).repeat(1, beam, 1, 1).view(B * beam, T2, -1)
    bmask = mmask.unsqueeze(1).repeat(1, beam, 1).view(B * beam, T2)

    def loop(cache):
        preds = torch.ones(B * beam, 1, dtype=torch.long, device=DEV)
        scores = torch.tensor([0.0] + [float('-inf')] * (beam - 1), device=DEV).repeat(B).unsqueeze(1)
        flag = torch.zeros_like(scores, dtype=torch.bool)
        with torch.no_grad():
            for _ in range(max_len):
                preds, cache, scores, flag = rec.decode_step(preds, bm, bmask, cache, scores, flag)
        return preds, scores

    with torch.no_grad():
        dc = model.decoder.init_cache(bm, bmask, max_len, beam=beam)
    p_c, s_c = loop({'decoder': dc})
    p_f, s_f = loop({'decoder': None})
    assert dc.step == max_len
    torch.testing.assert_close(s_c, s_f, rtol=3e-2, atol=0.3)
    assert torch.equal(p_c.view(B, beam, -1)[:, 0], p_f.view(B, beam, -1)[:, 0])
    kw = om.decoder_kwargs(params)
    with torch.no_grad():
        dc = model.decoder.init_cache(bm, bmask, max_len, beam=beam)
        preds = torch.ones(B * beam, 1, dtype=torch.long, device=DEV)
        o_preds = preds.cpu()
        o_scores = torch.tensor([0.0] + [float('-inf')] * (beam - 1)).repeat(B).unsqueeze(1)
        o_flag = torch.zeros_like(o_scores, dtype=torch.bool)
        for s in range(max_len):
            lp, dc, _ = model.decoder.inference(preds, bm, bmask, dc)
            lp_ref = om.decoder_inference(o_preds, bm.cpu(), bmask.cpu(), sd, 'decoder.', **kw)
            alive = ~o_flag.view(-1)
            assert _rel(lp.cpu()[alive][:, 2:], lp_ref[alive][:, 2:]) < REL_L2_LOGITS
            tr = []
            o_preds, o_scores, o_flag = obs.beam_step(lp.cpu(), o_preds, o_scores, o_flag, beam, trace=tr)
            dc.reorder(tr[0]['parent'].to(DEV))
            preds = o_preds.to(DEV)


def test_conformer_baseline_full_depth_1000_frames():
    """12 Conformer blocks / 6 decoder blocks, 4 x 1000 frames (T' = 249): encoder states and 60 lock-step graph steps."""
    params = conformer_baseline_params()
    model, sd = _build(params)
    lens_in = [1000, 873, 640, 999]
    x, mask = _batch(4, 1000, 80, lens_in)
    mem_ref, mmask = om.encode(x, mask, sd, params)
    B, beam, max_len = 4, 10, 60
    with torch.no_grad():
        mem, lens, _, T2 = model.encode_bf16(x.to(DEV), mask.to(DEV))
        got = mem.float().view(B, T2, -1).cpu()
        r = _rel(_valid(got, mmask), _valid(mem_ref, mmask))
        worst = max(_rel(got[b][mmask[b]], mem_ref[b][mmask[b]]) for b in range(B))
        print(f'conformer_baseline 12-block encoder, 4 x 1000 frames: rel_l2={r:.3e}, worst utterance {worst:.3e}')
        assert T2 == 249 and r < REL_L2_STATES and worst < REL_L2_STATES
        bd = BeamDecoder(model.decoder, B, beam, T2, max_len, DEV, use_graph=True, keep_logp=True)
        assert not bd.persistent
        bd.setup(mem, lens)
        _, _, worst_rel = _lockstep(bd, sd, params, mem, lens, B, beam, max_len, T2, check_every=6)
    print(f'conformer_baseline full depth: {max_len} graph steps identical; log-probs rel_l2<={worst_rel:.3e}')
    assert worst_rel < REL_L2_LOGITS


def test_training_refuses_96_wide_heads():
    """A d_model 384 / 4-head Transformer is constructible for inference; its training step must refuse rather than run
    the 64-wide attention backward on 96-wide heads."""
    from tests.test_gpu_model import _params
    params = _params(n_enc=1, n_dec=1)
    for part in ('encoder', 'decoder'):
        params[part].update(d_model=384, d_ff=768, residual_dropout=0.0)
    params['decoder']['memory_dim'] = 384
    params['frontend']['output_size'] = 384
    model = SpeechToText(params).to(DEV)
    x, mask = _batch(2, 120, 80, [120, 97])
    tgt = torch.tensor([[1, 5, 6, 1], [1, 7, 1, 0]])
    with pytest.raises(NotImplementedError, match='d_k = 64'):
        train.forward_backward(model.train(), x.to(DEV), mask.to(DEV), tgt.to(DEV))
