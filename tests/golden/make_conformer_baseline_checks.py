"""Record the reference's own outputs for the conformer_baseline.yaml case of tests/test_conformer_baseline_ref.py into
tests/golden/conformer_baseline_checks.pt.

    python oracle/build_ref.py && python tests/golden/make_conformer_baseline_checks.py [out.pt]

The reference is imported from its byte-compiled modules under oracle/_ref (oracle/build_ref.py).  Weights and inputs are
the seeded case of the test module, so only what the reference computed is stored: the state_dict layout, encoder states
on valid frames and recognize() hypotheses and scores.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import build_ref                                # noqa: E402
from tests import test_conformer_baseline_ref as cases      # noqa: E402
from tests.golden.make_reference_checks import record_recognize   # noqa: E402


def main(out):
    if build_ref.load() is None:
        raise SystemExit('oracle/_ref is missing: run oracle/build_ref.py first')
    golden = record_recognize(*cases.case())
    torch.save(golden, out)
    print({k: len(v) if isinstance(v, list) else tuple(getattr(v, 'shape', ())) for k, v in golden.items() if k != 'shapes'})
    print(f'wrote {out} ({os.path.getsize(out)} bytes)')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'tests', 'golden', cases.GOLDEN_FILE))
