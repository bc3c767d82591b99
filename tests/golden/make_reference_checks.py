"""Record the reference's own outputs for the cases of tests/test_oracle_ref.py into tests/golden/reference_checks.pt.

    python oracle/build_ref.py && python tests/golden/make_reference_checks.py [out.pt]

The reference is imported from its byte-compiled modules under oracle/_ref (oracle/build_ref.py).  Weights and inputs are
the seeded cases of tests/test_oracle_ref.py, so only what the reference computed is stored: the state_dict layout, encoder
states on valid frames, recognize() hypotheses and scores, and the training loss with, for every parameter gradient, its
L2 norm, GRAD_SAMPLES entries at seeded positions and GRAD_PROJECTIONS seeded projections (the full gradients would not keep
the fixture small).
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import build_ref                  # noqa: E402
from tests import test_oracle_ref as cases    # noqa: E402


def _reference_model(params, seed, eos_bias):
    from otrans.model import End2EndModel
    ref = End2EndModel['speech2text'](params)
    # interned names are pickled once for the whole file
    shapes = [(sys.intern(k), tuple(v.shape)) for k, v in ref.state_dict().items() if k.split('.')[0] in ('frontend', 'encoder', 'decoder')]
    missing, unexpected = ref.load_state_dict(cases.random_weights(shapes, seed, eos_bias), strict=False)
    assert not unexpected and all(k.split('.')[0] not in ('frontend', 'encoder', 'decoder') for k in missing), (missing, unexpected)
    return ref, shapes


def record_recognize(params, seed, eos_bias, inputs, search):
    from otrans.recognize.speech2text import SpeechToTextRecognizer
    x, mask = inputs
    ref, shapes = _reference_model(params, seed, eos_bias)
    ref.eval()
    vocab = params['decoder']['vocab_size']
    with torch.no_grad():
        fx, fm = ref.frontend(x, mask)
        mem, mm, _ = ref.encoder(fx, fm)
        rec = SpeechToTextRecognizer(ref, beam_width=search['beam'], nbest=search['nbest'], max_len=search['max_len'],
                                     idx2unit={i: str(i) for i in range(vocab)}, penalty=search['penalty'],
                                     lamda=search['lamda'], ngpu=0)
        hyps, scores = rec.recognize(x, mask)
    hyps = [[[int(t) for t in h.split()] if h else [] for h in row] for row in hyps]
    return {'shapes': shapes, 'memory_mask': mm.clone(), 'memory': mem[mm].clone(), 'hyps': hyps, 'scores': scores.float().clone()}


def record_gradients(params, seed, eos_bias, inputs, _):
    x, mask, tgt = inputs
    ref, shapes = _reference_model(params, seed, eos_bias)
    ref.train()
    loss, _ = ref({'inputs': x, 'mask': mask}, {'targets': tgt, 'targets_length': None})
    loss.backward()
    names, index, sample, norm, proj = [], [], [], [], []
    with torch.no_grad():
        for n, p in ref.named_parameters():
            if p.grad is None:
                continue
            i, flat = len(names), p.grad.reshape(-1)
            idx = torch.randint(flat.numel(), (cases.GRAD_SAMPLES,), generator=torch.Generator().manual_seed(i))
            names.append(sys.intern(n))
            index.append(idx.to(torch.int16))
            sample.append(flat[idx])
            norm.append(flat.norm())
            proj.append(cases.grad_projections(flat, i))
    return {'shapes': shapes, 'loss': loss.detach().clone(), 'grad_names': names, 'grad_index': torch.stack(index),
            'grad_sample': torch.stack(sample), 'grad_norm': torch.stack(norm), 'grad_proj': torch.stack(proj)}


def main(out):
    if build_ref.load() is None:
        raise SystemExit('oracle/_ref is missing: run oracle/build_ref.py first')
    record = {'recognize': record_recognize, 'gradients': record_gradients}
    golden = {name: record[kind](*case) for name, kind, case in cases.cases()}
    torch.save(golden, out)
    for name, g in golden.items():
        print(name, {k: len(v) if isinstance(v, list) else tuple(getattr(v, 'shape', ())) for k, v in g.items() if k != 'shapes'})
    print(f'wrote {out} ({os.path.getsize(out)} bytes)')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'tests', 'golden', cases.GOLDEN_FILE))
