"""Time the shipped Conformer recipe (conformer_baseline.yaml: d_model 384, 4 heads of width 96, 12 Conformer blocks,
6 decoder blocks, V = 4234) on one GPU, 32 utterances x 1000 frames, and print one JSON line.

    python tools/conformer_baseline_bench.py [--passes 20] [--warmup 3]

  * encoder forward (front end + 12 Conformer blocks), per 32-utterance batch;
  * SpeechToTextRecognizer.recognize with beam 10 and 60 steps (<S/E> bias -1e4, as in bench.py, so that every step
    runs; d_model 384 takes the per-step CUDA-graph decoder), per batch, encoder included;
  * the attention kernel alone at T' = 249 (32 x 4 heads, ragged lengths), head width 64 (d_model 256) and 96
    (d_model 384), plain and with the rel-pos band + residual the Conformer uses.

Method: CUDA events around each timed pass after warm-up; medians are reported.  Inputs rotate through 16 distinct
resident batches (16 x 10.2 MB of fbank features; the encoder writes > 0.5 GB of activations per pass), and the attention
timings rotate through enough distinct operand buffers that each pass's working set exceeds the 126 MB L2.
Weights are random (seeded): the timings do not depend on their values, and residual dropout is 0.0 (inference).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from tests.test_conformer_baseline_ref import conformer_baseline_params  # noqa: E402

B, T_IN, BEAM, MAX_LEN = 32, 1000, 10, 60


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.splitlines()[0].split(','))
    return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def median_ms(fn, passes, warmup):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    ts = []
    for i in range(passes):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(i)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def attention_times(ops, dev, passes, warmup):
    """Self-attention at T' = 249 over 32 utterances x 4 heads, head width 64 and 96; rotating operand buffers."""
    H, T = 4, 249
    lens = torch.randint(150, T + 1, (B,), generator=torch.Generator().manual_seed(5))
    lens[0] = T
    kv_len = lens.to(torch.int32).to(dev)
    ld = (2 * T - 1 + 3) // 4 * 4
    out = {}
    for hd in (64, 96):
        d = H * hd
        nbuf = 8            # 8 x 18 MB (hd 96) of qkv per rotation
        qkv = [torch.randn(B * T, 3 * d, device=dev).to(torch.bfloat16) for _ in range(nbuf)]
        bd = [torch.randn(H, B * T, ld, device=dev) for _ in range(2)]            # 2 x 64 MB
        res = torch.randn(B * T, d, device=dev).to(torch.bfloat16)
        with torch.no_grad():
            plain = median_ms(lambda i: ops.attention(qkv[i % nbuf], qkv[i % nbuf], qkv[i % nbuf], B, H, T, T, kv_len=kv_len,
                                                      q_col0=0, k_col0=d, v_col0=2 * d, head_dim=hd), passes, warmup)
            band = median_ms(lambda i: ops.attention(qkv[i % nbuf], qkv[i % nbuf], qkv[i % nbuf], B, H, T, T, kv_len=kv_len,
                                                     q_col0=0, k_col0=d, v_col0=2 * d, bd=bd[i % 2], resid=res, head_dim=hd),
                             passes, warmup)
        out[f'hd{hd}'] = {'self_attn_ms': plain[0], 'relpos_band_resid_ms': band[0],
                          'self_attn_min_max_ms': plain[1:], 'relpos_min_max_ms': band[1:]}
        del qkv, bd, res
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--passes', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('conformer_baseline_bench.py needs a GPU')
    from opentransformer_b200 import ops
    from opentransformer_b200.model import SpeechToText
    from opentransformer_b200.recognize import SpeechToTextRecognizer
    dev = torch.device('cuda:0')
    torch.manual_seed(1234)
    model = SpeechToText(conformer_baseline_params()).eval()
    with torch.no_grad():
        model.decoder.output_layer.bias[1] = -1e4
    model.to(dev)
    ring = [tuple(t.to(dev) for t in bench.synthetic_batch(B, i)) for i in range(16)]
    with torch.no_grad():
        enc = median_ms(lambda i: model.encode_bf16(*ring[i % 16]), args.passes, args.warmup)
        rec = SpeechToTextRecognizer(model, beam_width=BEAM, nbest=1, max_len=MAX_LEN, penalty=0.6, lamda=5, ngpu=1)
        n_passes = max(5, args.passes // 4)
        recog = median_ms(lambda i: rec.recognize(*ring[i % 16]), n_passes, args.warmup)
        persistent = any(bd.persistent for bd in rec._decoders.values())
    attn = attention_times(ops, dev, args.passes * 5, args.warmup)
    line = {'metric': 'conformer_baseline.yaml on one GPU, 32 utt x 1000 frames', 'gpu': gpu_info(),
            'encoder_forward_ms': enc[0], 'encoder_forward_min_max_ms': enc[1:],
            'encoder_utt_per_s': B / (enc[0] * 1e-3),
            'recognize_ms': recog[0], 'recognize_min_max_ms': recog[1:], 'recognize_utt_per_s': B / (recog[0] * 1e-3),
            'recognize': f'beam {BEAM}, {MAX_LEN} steps (<S/E> bias -1e4), encoder included, '
                         f'{"persistent" if persistent else "per-step CUDA-graph"} decoder',
            'attention_T249': attn, 'passes': args.passes, 'recognize_passes': n_passes, 'warmup': args.warmup,
            'timing': 'CUDA events, median of passes after warm-up',
            'l2_policy': '16 rotating input batches; attention operands rotate over 8 qkv / 2 band buffers (> 126 MB)'}
    print(json.dumps(line))


if __name__ == '__main__':
    main()
