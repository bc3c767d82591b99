"""The oracle port at the geometry of the shipped Conformer recipe (conformer_baseline.yaml: d_model 384, 4 heads of
width 96), pinned to what the reference's own modules computed on a seeded 2 + 2 block model.  The reference outputs are
stored in tests/golden/conformer_baseline_checks.pt (tests/golden/make_conformer_baseline_checks.py records them from
oracle/_ref).  Also checks that the B200 model builds from the same params with the reference's state_dict layout, and
the head-width guards of the modules and of the C ABI (no GPU needed)."""
import ctypes
import os

import pytest
import torch

from oracle import beam_search as obs
from oracle import speech_model as om
from tests.test_oracle_ref import random_weights

GOLDEN_FILE = 'conformer_baseline_checks.pt'


def conformer_baseline_params(n_enc=12, n_dec=6):
    """The `model:` section of conformer_baseline.yaml with residual_dropout 0.0 (the reference applies the Conformer
    residual dropout even in eval(), so only the dropout-free network is deterministic)."""
    return {'type': 'speech2text', 'frontend_type': 'conv', 'encoder_type': 'conformer', 'decoder_type': 'transformer',
            'frontend': dict(input_size=80, output_size=384, in_channel=1, mid_channel=256, out_channel=256,
                             kernel_size=[[3, 3], [3, 3]], stride=[2, 2], dropout=0.0, act_func_type='relu',
                             front_end_layer_norm=False),
            'encoder': dict(d_model=384, d_ff=768, cov_kernel_size=5, n_heads=4, nblocks=n_enc, pos_dropout=0.0,
                            slf_attn_dropout=0.0, ffn_dropout=0.0, residual_dropout=0.0, conv_dropout=0.0,
                            macaron_style=True, ffn_scale=0.5, conv_bias=True, activation='glu',
                            positional_encoding=True, relative_positional=True),
            'decoder': dict(vocab_size=4234, d_model=384, n_heads=4, d_ff=768, memory_dim=384, n_blocks=n_dec,
                            pos_dropout=0.0, slf_attn_dropout=0.0, src_attn_dropout=0.0, ffn_dropout=0.0,
                            residual_dropout=0.0, activation='glu', normalize_before=False, concat_after=False,
                            share_embedding=True),
            'ctc_weight': 0.0, 'smoothing': 0.1}


def case():
    """(params, weight seed, <S/E> bias, (x, mask), search settings) recorded by make_conformer_baseline_checks.py."""
    g = torch.Generator().manual_seed(21)
    lens = torch.tensor([120, 97, 61])
    mask = torch.arange(120)[None] < lens[:, None]
    x = torch.randn(3, 120, 80, generator=g) * mask.unsqueeze(2)
    return (conformer_baseline_params(n_enc=2, n_dec=2), 384, 1.5, (x, mask),
            dict(beam=4, nbest=4, max_len=8, penalty=0.6, lamda=5))


@pytest.fixture(scope='module')
def reference(golden_dir):
    return torch.load(os.path.join(golden_dir, GOLDEN_FILE), weights_only=False)


def test_oracle_equals_reference_at_conformer_baseline_geometry(reference):
    """Encoder states on valid frames to 1e-4, recognize() hypotheses bit-exact and scores to 1e-4 (beam 4)."""
    params, seed, eos_bias, (x, mask), s = case()
    sd = random_weights(reference['shapes'], seed, eos_bias)
    with torch.no_grad():
        mem, mm = om.encode(x, mask, sd, params)
        assert torch.equal(mm, reference['memory_mask'])
        torch.testing.assert_close(mem[mm], reference['memory'], rtol=1e-4, atol=1e-4)
        nb, ns, _, _ = obs.recognize(x, mask, sd, params, **s)
    for b in range(x.shape[0]):
        for r in range(s['nbest']):
            port = [int(t) for t in nb[b, r].tolist()]
            port = port[:port.index(1)] if 1 in port else port
            assert port == reference['hyps'][b][r], (b, r)
    torch.testing.assert_close(ns, reference['scores'], rtol=1e-4, atol=1e-4)


def test_b200_model_has_the_reference_state_dict_layout(reference):
    from opentransformer_b200.model import SpeechToText
    params = case()[0]
    model = SpeechToText(params)
    ours = [(k, tuple(v.shape)) for k, v in model.state_dict().items() if k.split('.')[0] in ('frontend', 'encoder', 'decoder')]
    assert sorted(ours) == sorted(reference['shapes'])
    assert model.decoder.head_dim == 96 and all(b.mha.head_dim == 96 for b in model.encoder.blocks)


def test_modules_accept_64_and_96_wide_heads_only():
    from opentransformer_b200 import modules as m
    for d, h in ((256, 4), (384, 4), (192, 2), (96, 1)):
        assert m.MultiHeadedSelfAttention(h, d).head_dim == d // h
        assert m.MultiHeadedCrossAttention(h, d, d).head_dim == d // h
        assert m.MultiHeadedSelfAttentionWithRelPos(h, d).head_dim == d // h
    for d, h in ((320, 4), (512, 4), (384, 8), (100, 3)):
        for make in (lambda: m.MultiHeadedSelfAttention(h, d), lambda: m.MultiHeadedCrossAttention(h, d, d),
                     lambda: m.MultiHeadedSelfAttentionWithRelPos(h, d)):
            with pytest.raises(NotImplementedError, match='d_k'):
                make()


def test_language_model_keeps_64_wide_heads():
    from opentransformer_b200.lm import TransformerLanguageModel
    p = dict(vocab_size=50, d_model=384, n_heads=4, d_ff=768, num_blocks=1)
    with pytest.raises(NotImplementedError, match='d_k'):
        TransformerLanguageModel(p)
    TransformerLanguageModel(dict(p, d_model=256))


def test_c_abi_rejects_other_head_widths_without_launching():
    from opentransformer_b200 import _lib, build
    build.build()
    lib = _lib.lib()
    one = ctypes.c_void_p(16)          # never dereferenced: the head width is checked first
    for hd in (32, 80, 128, 0):
        assert lib.otb_attention_hd(one, 384, 1, one, 384, 1, one, 384, one, 384, 1, 4, hd, 1, 1, None, 0, 0, 0, 0,
                                    None, 0, None, 0, None) != 0
        assert b'head_dim must be 64 or 96' in lib.otb_last_error()
        assert lib.otb_attention_lse_hd(one, 384, 1, one, 384, 1, one, 384, one, 384, 1, 4, hd, 1, 1, None, 0, 0, 0, 0,
                                        None, 0, None, 0, one, None) != 0
        assert b'head_dim must be 64 or 96' in lib.otb_last_error()
        assert lib.otb_decode_self_attn_hd(one, one, one, one, one, one, 4, 4, hd, 8, None) != 0
        assert b'head_dim must be 64 or 96' in lib.otb_last_error()
