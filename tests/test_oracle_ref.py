"""The oracle port against the reference's own modules on fresh random models: encoder states, the whole recognize() and the
training loss / gradients.  Weights and inputs are drawn from seeds here; what the reference computed for them is stored in
tests/golden/reference_checks.pt (tests/golden/make_reference_checks.py runs the reference on exactly these cases).
Complements tests/test_oracle_golden.py, whose fixtures pin the reference's configurations with its own initialisation."""
import math
import os

import pytest
import torch

from oracle import beam_search as obs
from oracle import speech_model as om

GOLDEN_FILE = 'reference_checks.pt'
GRAD_SAMPLES = 32           # gradient entries stored per parameter tensor, with its L2 norm and GRAD_PROJECTIONS projections
GRAD_PROJECTIONS = 4


def _params(normalize_before, activation):
    return {'type': 'speech2text', 'frontend_type': 'conv', 'encoder_type': 'transformer', 'decoder_type': 'transformer',
            'frontend': dict(input_size=20, output_size=32, in_channel=1, mid_channel=4, out_channel=8,
                             kernel_size=[[3, 3], [3, 3]], stride=[2, 2], dropout=0.0, act_func_type='relu',
                             front_end_layer_norm=False),
            'encoder': dict(d_model=32, n_heads=4, d_ff=48, n_blocks=2, pos_dropout=0.0, slf_attn_dropout=0.0,
                            ffn_dropout=0.0, residual_dropout=0.0, normalize_before=normalize_before, concat_after=False,
                            activation=activation, relative_positional=False),
            'decoder': dict(vocab_size=40, d_model=32, n_heads=4, d_ff=48, memory_dim=32, n_blocks=2, pos_dropout=0.0,
                            slf_attn_dropout=0.0, src_attn_dropout=0.0, ffn_dropout=0.0, residual_dropout=0.0,
                            activation=activation, normalize_before=normalize_before, concat_after=False,
                            share_embedding=True),
            'ctc_weight': 0.0, 'smoothing': 0.1}


def grad_projections(flat, i):
    """Seeded Gaussian projections of the flattened gradient of the i-th parameter: a deviation in any of its entries moves
    them to first order, so together with the sampled entries and the norm they stand in for the full tensor."""
    return torch.randn(GRAD_PROJECTIONS, flat.numel(), generator=torch.Generator().manual_seed(i)) @ flat


def _batch(lens, T, g):
    lens = torch.tensor(lens)
    mask = torch.arange(T)[None] < lens[:, None]
    return torch.randn(len(lens), T, 20, generator=g) * mask.unsqueeze(2), mask


def random_weights(shapes, seed, eos_bias=None):
    """Seeded weights for the state_dict layout `shapes` [(key, shape)]: linear / conv weights with the spread of nn.Linear's
    default init, LayerNorm / BatchNorm parameters and running statistics away from their identity values, the shared
    embedding scaled down.  `eos_bias` raises the output bias of <S/E> (id 1) so that hypotheses end at different steps."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shape in shapes:
        if k == 'decoder.output_layer.weight':         # share_embedding=True
            sd[k] = sd['decoder.embedding.weight']
        elif k.endswith('num_batches_tracked'):
            sd[k] = torch.tensor(0)
        elif k.endswith('running_mean'):
            sd[k] = 0.3 * torch.randn(shape, generator=g)
        elif k.endswith('running_var'):
            sd[k] = 1.0 + 0.5 * torch.rand(shape, generator=g)
        elif 'norm' in k:
            sd[k] = (1.0 if k.endswith('weight') else 0.0) + 0.2 * torch.randn(shape, generator=g)
        elif k == 'decoder.embedding.weight':
            sd[k] = 0.15 * torch.randn(shape, generator=g)
        elif k.endswith('.bias'):
            sd[k] = 0.1 * torch.randn(shape, generator=g)
        else:
            sd[k] = torch.randn(shape, generator=g) / math.sqrt(3 * math.prod(shape[1:]))
    if eos_bias is not None:
        sd['decoder.output_layer.bias'][1] = eos_bias
    return sd


# Each case: (params, weight seed, <S/E> bias, inputs, search settings); make_reference_checks.py records the reference on them.
def recognize_case(normalize_before, activation):
    x, mask = _batch([64, 50, 37], 64, torch.Generator().manual_seed(5))
    return _params(normalize_before, activation), 4321, 1.5, (x, mask), dict(beam=3, nbest=3, max_len=9, penalty=0.6, lamda=5)


def gradient_case(normalize_before, activation):
    g = torch.Generator().manual_seed(7)
    x, mask = _batch([70, 55, 41], 70, g)
    B, L = 3, 8
    tgt = torch.randint(3, 40, (B, L), generator=g)
    tgt[:, 0] = 1
    tgt[0, L - 2:] = torch.tensor([1, 0])
    tgt[1, L - 1] = 1
    tgt[2, 4:] = torch.tensor([1, 0, 0, 0])
    return _params(normalize_before, activation), 99, None, (x, mask, tgt), None


def relpos_encoder_case(kind):
    params = _params(False, 'glu')
    if kind == 'conformer':
        params['encoder_type'] = 'conformer'
        params['encoder'] = dict(d_model=32, d_ff=24, cov_kernel_size=5, n_heads=4, nblocks=2, pos_dropout=0.0, slf_attn_dropout=0.0,
                                 ffn_dropout=0.0, residual_dropout=0.0, conv_dropout=0.0, macaron_style=True, ffn_scale=0.5,
                                 conv_bias=True, activation='glu', positional_encoding=True, relative_positional=True)
    else:
        params['encoder']['relative_positional'] = True
    x, mask = _batch([72, 60, 33], 72, torch.Generator().manual_seed(11))
    return params, 77, 1.5, (x, mask), dict(beam=3, nbest=1, max_len=7, penalty=0.6, lamda=5)


RECOGNIZE = [(False, 'glu'), (True, 'relu')]
GRADIENTS = [(False, 'glu'), (True, 'glu'), (False, 'relu'), (True, 'relu')]
ENCODERS = ['conformer', 'relpos_transformer']


def _name(family, *args):
    return family + '/' + '-'.join(str(a) for a in args)


def cases():
    """(golden key, 'recognize' | 'gradients', case) of every test below."""
    return ([(_name('recognize', *a), 'recognize', recognize_case(*a)) for a in RECOGNIZE]
            + [(_name('gradients', *a), 'gradients', gradient_case(*a)) for a in GRADIENTS]
            + [(_name('encoder', k), 'recognize', relpos_encoder_case(k)) for k in ENCODERS])


@pytest.fixture(scope='module')
def reference(golden_dir):
    return torch.load(os.path.join(golden_dir, GOLDEN_FILE), weights_only=False)


def _setup(reference, name, case):
    params, seed, eos_bias, inputs, search = case
    ref = reference[name]
    return ref, params, random_weights(ref['shapes'], seed, eos_bias), inputs, search


def _check_encoder(ref, x, mask, sd, params):
    mem, mm = om.encode(x, mask, sd, params)
    assert torch.equal(mm, ref['memory_mask'])
    torch.testing.assert_close(mem[mm], ref['memory'], rtol=1e-4, atol=2e-5)


def _port_hyps(nb, b, r):
    port = [int(t) for t in nb[b, r].tolist()]
    return port[:port.index(1)] if 1 in port else port


@pytest.mark.parametrize('normalize_before,activation', RECOGNIZE)
def test_port_equals_live_reference(reference, normalize_before, activation):
    """Encoder states and the whole recognize(): ids bit-exact, scores to fp32 tolerance."""
    ref, params, sd, (x, mask), s = _setup(reference, _name('recognize', normalize_before, activation),
                                           recognize_case(normalize_before, activation))
    with torch.no_grad():
        _check_encoder(ref, x, mask, sd, params)
        nb, ns, _, _ = obs.recognize(x, mask, sd, params, **s)
    for b in range(x.shape[0]):
        for r in range(s['beam']):
            assert _port_hyps(nb, b, r) == ref['hyps'][b][r], (b, r)
    torch.testing.assert_close(ns, ref['scores'], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('normalize_before,activation', GRADIENTS)
def test_port_gradients_equal_live_reference_autograd(reference, normalize_before, activation):
    """model.train(); loss, _ = model(inputs, targets); loss.backward() through the reference's own modules (trainer.py:206-217)
    vs oracle/train_step.loss_and_grads: the loss, and for every parameter gradient its L2 norm and a seeded sample of its
    entries -- in particular for the pre-norm and ReLU stacks whose hand-written CUDA backward is tested against this port
    (tests/test_gpu_train.py)."""
    from oracle import train_step as ot
    ref, params, sd, (x, mask, tgt), _ = _setup(reference, _name('gradients', normalize_before, activation),
                                                gradient_case(normalize_before, activation))
    loss, grads = ot.loss_and_grads(x, mask, tgt, sd, params)
    torch.testing.assert_close(loss, ref['loss'], rtol=1e-5, atol=1e-5)
    assert set(grads) == set(ref['grad_names']), set(grads) ^ set(ref['grad_names'])
    for i, n in enumerate(ref['grad_names']):
        got = grads[n].reshape(-1)
        torch.testing.assert_close(got[ref['grad_index'][i].long()], ref['grad_sample'][i], rtol=2e-4, atol=2e-6,
                                   msg=lambda m, n=n: f'{n}: {m}')
        torch.testing.assert_close(got.norm(), ref['grad_norm'][i], rtol=2e-4, atol=2e-6, msg=lambda m, n=n: f'{n} (L2 norm): {m}')
        # entrywise errors within rtol / atol move a projection by about their L2 norm
        tol = 4 * (2e-4 * float(ref['grad_norm'][i]) + 2e-6 * math.sqrt(got.numel()))
        diff = float((grad_projections(got, i) - ref['grad_proj'][i]).abs().max())
        assert diff <= tol, f'{n}: random projections differ by {diff:.3e} > {tol:.3e}'


@pytest.mark.parametrize('kind', ENCODERS)
def test_port_encoder_states_equal_live_reference_for_relpos_encoders(reference, kind):
    """Conformer (macaron FFN, rel-pos attention without output projection, conv module with BatchNorm running statistics,
    only post_ffn_norm applied: SURVEY.md 8a quirks) and the rel-pos Transformer encoder: valid-frame states of the port vs
    the reference modules, recognize() ids bit-exact."""
    ref, params, sd, (x, mask), s = _setup(reference, _name('encoder', kind), relpos_encoder_case(kind))
    with torch.no_grad():
        _check_encoder(ref, x, mask, sd, params)
        nb, _, _, _ = obs.recognize(x, mask, sd, params, **s)
    for b in range(x.shape[0]):
        assert _port_hyps(nb, b, 0) == ref['hyps'][b][0], b
