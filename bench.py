#!/usr/bin/env python
"""Benchmark of the B200 hot path (BASELINE.json metric): utterances/sec through frontend+encoder
forward and batched beam-search decode, synthetic 80-dim fbank (1000 frames), random-init weights.

    python bench.py [--gpus N --steps K --warmup W] [--dump-outputs DIR]     # this repo's CUDA path
    python bench.py --impl reference [...]                      # the reference algorithm on host cores (oracle port)

One "step" = one full recognize pass (frontend -> 12-layer encoder -> 60-step beam-10 decode ->
n-best) over a batch of 32 utterances per GPU.  N > 1 shards utterance batches across ranks with no
data-path collective (weak scaling; SURVEY.md 8e).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# One hardware work queue per lane: by default a process gets 8 channels to the GPU and streams beyond the 8th share them,
# which serialises the launches of unrelated lanes (false dependencies).  Must be set before the CUDA context exists.
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, T_FRAMES, F_BINS, BEAM, MAX_LEN, PENALTY, LAMDA = 32, 1000, 80, 10, 60, 0.6, 5


def model_params():
    """egs/aishell/conf/transformer_baseline.yaml `model:` with input_size 80 (SURVEY.md 8d config 2/3)."""
    return {'type': 'speech2text', 'frontend_type': 'conv', 'encoder_type': 'transformer',
            'decoder_type': 'transformer',
            'frontend': dict(input_size=F_BINS, output_size=256, in_channel=1, mid_channel=64, out_channel=128,
                             kernel_size=[[3, 3], [3, 3]], stride=[2, 2], dropout=0.0, act_func_type='relu',
                             front_end_layer_norm=False),
            'encoder': dict(d_model=256, n_heads=4, d_ff=2048, n_blocks=12, pos_dropout=0.0, slf_attn_dropout=0.0,
                            ffn_dropout=0.0, residual_dropout=0.1, normalize_before=False, concat_after=False,
                            activation='glu', relative_positional=False),
            'decoder': dict(vocab_size=4234, d_model=256, n_heads=4, d_ff=2048, memory_dim=256, n_blocks=6,
                            pos_dropout=0.0, slf_attn_dropout=0.0, src_attn_dropout=0.0, ffn_dropout=0.0,
                            residual_dropout=0.1, activation='glu', normalize_before=False, concat_after=False,
                            share_embedding=True),
            'ctc_weight': 0.0, 'smoothing': 0.1}


def build_model():
    from opentransformer_b200.model import SpeechToText
    torch.manual_seed(1234)
    model = SpeechToText(model_params()).eval()
    with torch.no_grad():
        model.decoder.output_layer.bias[1] = -1e4      # SURVEY.md 8(d) config 3: all 60 steps execute
    return model


def flat_state_dict(model):
    sd = {}
    for part in ('frontend', 'encoder', 'decoder'):
        for k, v in getattr(model, part).state_dict().items():
            sd[f'{part}.{k}'] = v.detach().float().cpu().clone()
    return sd


def synthetic_batch(batch, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, T_FRAMES, F_BINS, generator=g)
    mask = torch.ones(batch, T_FRAMES, dtype=torch.bool)
    return x, mask


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region (NVML; nvidia-smi as fallback)."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            try:
                return int(vis.split(',')[i])
            except Exception:
                return i
        return i

    def _sample(self):
        if self.nv is not None:
            nv = self.nv
            sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons') \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            bit = lambda name, default: getattr(nv, name, default)
            flags = ['Active' if r & bit('nvmlClocksThrottleReasonHwSlowdown', 0x8) else 'Not Active',
                     'Active' if r & bit('nvmlClocksThrottleReasonHwThermalSlowdown', 0x40) else 'Not Active',
                     'Active' if r & bit('nvmlClocksThrottleReasonSwThermalSlowdown', 0x20) else 'Not Active',
                     'Active' if r & bit('nvmlClocksThrottleReasonSwPowerCap', 0x4) else 'Not Active']
            return [str(sm), str(mx)] + flags
        out = subprocess.run(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                              '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
        return [c.strip() for c in out.strip().split(',')]

    def run(self):
        while not self._halt.is_set():
            try:
                self.rows.append(self._sample())
            except Exception:
                pass
            self._halt.wait(0.02 if self.nv is not None else 0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == 'Active' for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(self.rows), 'source': 'nvml' if self.nv is not None else 'nvidia-smi'}


_REAL_STDOUT = None


def guard_stdout():
    """Rank 0's stdout must carry exactly ONE JSON line, but libraries write there too (NCCL prints its version banner on
    stdout when the communicator is created, whatever NCCL_DEBUG says on this image): from here on file descriptor 1 goes
    to stderr and the JSON line is written to the saved descriptor by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + '\n').encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def nccl_logging():
    """NCCL writes its debug output to STDOUT unless NCCL_DEBUG_FILE is set; rank 0's stdout must carry exactly one JSON
    line.  Round 1 forced NCCL_DEBUG=WARN, which also hid the communicator's rank count from the driver.  Now every rank
    logs INIT-level INFO into a file; rank 0 parses it (ranks of the communicator, NVLS) into the JSON line and echoes the
    init lines to stderr."""
    os.environ['NCCL_DEBUG'] = 'INFO'
    os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT')
    path = '/tmp/otb_nccl_%s_r%s.log' % (os.environ.get('MASTER_PORT', '0'), os.environ.get('RANK', '0'))
    os.environ['NCCL_DEBUG_FILE'] = path
    try:
        os.remove(path)
    except OSError:
        pass
    return path


def nccl_summary(path, world):
    """{'nranks': N seen in the 'Init COMPLETE' line, 'nvls': bool, ...} from rank 0's NCCL INFO log."""
    import re
    out = {'log': path, 'nranks': None, 'nvls': None, 'version': None}
    try:
        txt = open(path, errors='replace').read()
    except OSError:
        return out
    m = re.search(r'nranks (\d+)[^\n]*Init COMPLETE', txt) or re.search(r'nranks (\d+)', txt)
    if m:
        out['nranks'] = int(m.group(1))
    out['nvls'] = bool(re.search(r'NVLS', txt))
    m = re.search(r'NCCL version ([0-9.+a-z]+)', txt)
    if m:
        out['version'] = m.group(1)
    out['nranks_ok'] = (out['nranks'] == world) if out['nranks'] is not None else None
    for ln in txt.splitlines():
        if 'Init COMPLETE' in ln or 'NCCL version' in ln or ('NVLS' in ln and 'comm' in ln):
            sys.stderr.write('[nccl] ' + ln.strip()[:240] + '\n')
    return out


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return p, 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


# ------------------------------------------------------------------------------------------------
def usable_cpus():
    """CPUs this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def pick_cpu_threads():
    """Give the CPU arm its best case: calibrate the intra-op thread count on a micro-workload shaped like
    the decoder hot loop (torch's default of one thread per visible core was 60x slower on the 128-core
    GPU box than 8 threads because the per-op work is small).  Returns (threads, visible_cores)."""
    import torch.nn.functional as F
    cores = usable_cpus()
    a, w = torch.randn(320 * 8, 256), torch.randn(4096, 256)
    xc, wc = torch.randn(2, 64, 499, 40), torch.randn(128, 64, 3, 3)
    best, best_t = 1, float('inf')
    cands = sorted({c for c in (4, 8, 16, 32, 64, 128, cores) if c <= cores} | {min(cores, 4)})
    for c in cands:
        torch.set_num_threads(c)
        F.glu(a @ w.t()); F.conv2d(xc, wc, stride=2, padding=(0, 1))      # warm the pool
        t0 = time.perf_counter()
        for _ in range(5):
            F.glu(a @ w.t())
            torch.softmax((a[:, :64] @ a[:, :64].t()), -1)
        F.conv2d(xc, wc, stride=2, padding=(0, 1))
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        elif dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best, cores


def cpu_reference_pass(sd, params, x, mask):
    """The reference algorithm (oracle port, fp32, all host threads): encode + 60-step beam-10 decode."""
    from oracle import beam_search as obs
    with torch.no_grad():
        return obs.recognize(x, mask, sd, params, beam=BEAM, nbest=1, max_len=MAX_LEN, penalty=PENALTY, lamda=LAMDA)


def reference_recognizer(model):
    """The reference's OWN SpeechToTextRecognizer on the CPU with the weights of `model`, from the byte-compiled package
    under oracle/_ref (oracle/build_ref.py; built by __graft_entry__.build() where /root/reference exists, travels with
    gpurun).  None when oracle/_ref is absent: the caller then times the oracle port instead."""
    try:
        from oracle import build_ref
        if build_ref.load() is None:
            return None
        from otrans.model import End2EndModel
        from otrans.recognize.speech2text import SpeechToTextRecognizer as RefRecognizer
        ref = End2EndModel['speech2text'](model_params()).eval()
        for part in ('frontend', 'encoder', 'decoder'):          # identical state_dict keys (tests/test_capi_symbols.py)
            getattr(ref, part).load_state_dict({k: v.detach().float().cpu() for k, v in getattr(model, part).state_dict().items()})
        idx2unit = {i: str(i) for i in range(model_params()['decoder']['vocab_size'])}
        return RefRecognizer(ref, beam_width=BEAM, nbest=1, max_len=MAX_LEN, idx2unit=idx2unit, penalty=PENALTY, lamda=LAMDA, ngpu=0)
    except Exception as e:      # an unusable _ref must not cost the line: fall back to the port and say so
        sys.stderr.write(f'bench.py: oracle/_ref unusable ({type(e).__name__}: {e}); timing the oracle port\n')
        return None


def reference_ids(rec, x, mask):
    """1-best token ids [B, <= max_len] of the reference recogniser (it returns strings of unit names = the ids here)."""
    with torch.no_grad():
        hyps, _ = rec.recognize(x, mask)
    rows = []
    for h in hyps:
        toks = [int(t) for t in h[0].split()] if h and h[0] else []
        rows.append(toks)
    return rows


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    threads, cores = pick_cpu_threads()
    torch.manual_seed(1234)
    sample = args.ref_sample
    model = build_model()
    sd, params = flat_state_dict(model), model_params()
    x, mask = synthetic_batch(sample, 0)
    rec = reference_recognizer(model)
    kind = 'reference' if rec is not None else 'port'

    def one_pass():
        if rec is not None:
            with torch.no_grad():
                return rec.recognize(x, mask)
        return cpu_reference_pass(sd, params, x, mask)
    for _ in range(max(0, min(args.warmup, 1))):
        one_pass()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass()
    dt = time.perf_counter() - t0
    val = sample * args.steps / dt
    line = {'impl': 'reference', 'metric': 'utterances/sec (encoder-fwd + beam-10 decode, 60 steps)', 'value': val,
            'unit': 'utt/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': min(args.warmup, 1),
            'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args, sample),
            'cpu_baseline': {'value': val, 'unit': 'utt/s', 'cores': threads, 'visible_cores': cores, 'kind': kind,
                             'sample': f'{sample} utterances x {args.steps} passes of the full workload '
                                       + ('(the reference\'s own SpeechToTextRecognizer.recognize, byte-compiled into oracle/_ref '
                                          'by oracle/build_ref.py, fp32 on the host cores)' if kind == 'reference' else
                                          '(oracle/ = torch-CPU fp32 restatement of the reference; oracle/_ref is absent here)')},
            'e2e': {'value': val, 'unit': 'utt/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    emit(line)
    return 0


def time_gemm_shape(tag, dev, reps=200):
    """Average DEVICE duration (ms) of one otb_linear launch of shape `tag` = (epilogue, M, weight rows, K, out_f32): a CUDA
    graph of `reps` launches on synthetic operands, replayed between two CUDA events (round 1 launched them eagerly through
    ctypes, which measured the host's launch rate, VERDICT r1 weak #6)."""
    from opentransformer_b200 import ops
    epi, M, Nw, K, of32 = tag
    g = torch.Generator().manual_seed(3)
    a = torch.randn(M, K, generator=g).to(torch.bfloat16).to(dev)
    w = (torch.randn(Nw, K, generator=g) * 0.05).to(torch.bfloat16).to(dev)
    bias = torch.zeros(Nw, device=dev)
    n_out = Nw // 2 if epi == ops.EPI_GLU else Nw
    kw = {}
    if epi in (ops.EPI_RESID, ops.EPI_RESID_LN):
        kw['resid'] = torch.randn(M, n_out, generator=g).to(torch.bfloat16).to(dev)
    if epi == ops.EPI_RESID_LN:
        kw['gamma'], kw['beta'] = torch.ones(n_out, device=dev), torch.zeros(n_out, device=dev)
    if epi == ops.EPI_TABLE:
        kw['table'], kw['period'] = torch.zeros(M, n_out, device=dev), M
    ld = (n_out + 7) // 8 * 8
    out = torch.empty(M, ld, dtype=torch.float32 if of32 else torch.bfloat16, device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            ops.linear(a, w, bias, epi, out=out, **kw)
    torch.cuda.current_stream().wait_stream(side)
    n0 = ops.COUNTERS['launches']
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(reps):
            ops.linear(a, w, bias, epi, out=out, **kw)
    ops.COUNTERS['launches'] = n0
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def init_dist():
    """(rank, world, local, device, nccl log path): one process per GPU, NCCL over NVLink for N > 1."""
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    log = None
    if world > 1 and not dist.is_initialized():
        log = nccl_logging()
        dist.init_process_group('nccl', device_id=dev)
    return rank, world, local, dev, log


def dist_barrier(world):
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy: floating point as float32, integers as float64 (exact below 2**53)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = torch.as_tensor(a)
        a = a.float().numpy() if a.is_floating_point() else a.numpy().astype(np.float64)
        np.save(os.path.join(path, name + '.npy'), a)


def ids_digest(ids):
    import hashlib
    return hashlib.sha1(ids.detach().to('cpu', torch.int64).contiguous().numpy().tobytes()).hexdigest()


def workload_config(args, batch):
    return {'workload': 'Speech-Transformer 12-enc/6-dec d_model=256 h=4 d_ff=2048(GLU) V=4234; '
                        f'{batch} utt x {T_FRAMES} frames x {F_BINS}-dim fbank per GPU; frontend+encoder forward + '
                        f'batch beam search (beam={BEAM}, max_len={MAX_LEN}, penalty={PENALTY}, lamda={LAMDA}, LM off, '
                        'EOS bias -1e4 so all steps run)',
            'batch_per_gpu': batch, 'frames': T_FRAMES, 'beam': BEAM, 'max_len': MAX_LEN,
            'parallelism': f'dp{args.gpus} (utterance sharding, no data-path collective)',
            'l2_policy': 'no flush; 16 distinct resident input batches rotate (164 MB > 126 MB L2) and each step '
                         'streams ~1 GB of activations'}


# ------------------------------------------------------------------------------------------------
DEC_FLOP = 540.0e9     # SURVEY.md 8(d): KV-cached beam decode, 32 utt x beam 10 x 60 steps
ENC_FLOP = 410.0e9     # frontend + 12-layer encoder forward, 32 x 1000 frames


def decode_step_bytes(model, batch, T2):
    """Algorithmic HBM/L2 bytes of ONE beam step of one utterance batch (SURVEY.md 8d): every decoder weight read once
    (bf16; the cross-attention K/V projection is not part of the step) + the per-utterance cross-attention K/V cache."""
    dec = model.decoder
    w = 0
    for n, p in dec.named_parameters():
        if 'vk_proj' in n or n.startswith('output_layer.weight') and dec.output_layer.weight is dec.embedding.weight:
            continue
        w += p.numel() * 2
    kv = len(dec.blocks) * batch * T2 * 2 * dec.d_model * 2
    return w, kv


def run_b200(args):
    import torch.distributed as dist
    from opentransformer_b200 import ops
    from opentransformer_b200.recognize import SpeechToTextRecognizer, BeamDecoder
    rank, world, local, dev, nccl_log = init_dist()

    def barrier():
        dist_barrier(world)

    model = build_model().to(dev)
    # Distinct resident input batches, rotated by step index, so consecutive steps never re-read the same input
    # and the per-step working set (>= 160 MB of inputs in the ring, ~1 GB of activations) exceeds the 126 MB L2.
    RING = 16
    ring_cpu = [synthetic_batch(B_PER_GPU, 1000 * rank + i) for i in range(RING)]
    ring_pin = [(x.pin_memory(), m.pin_memory()) for x, m in ring_cpu]
    ring_dev = [(x.to(dev), m.to(dev)) for x, m in ring_cpu]

    def make_rec(persistent):
        return SpeechToTextRecognizer(model, beam_width=BEAM, nbest=1, max_len=MAX_LEN, penalty=PENALTY, lamda=LAMDA, ngpu=1,
                                      persistent=persistent)

    # decode path: 'persistent' = the whole 60-step loop in one launch per batch (csrc/decode_group.cu, 48 SMs per batch of
    # 32 utterances x beam 10), 'graph' = one CUDA-graph replay of ~52 kernels per step (round 1).  'auto' takes the
    # persistent kernel only after a probe in a CHILD process produced exactly the graph path's hypotheses on input batch 0:
    # a device-side fault there (a trap poisons the CUDA context) must not cost the benchmark line.
    ops.set_tile_policy('latency')
    persist_ok, probe_note = False, 'not probed'
    if args.decode in ('auto', 'persistent'):
        persist_ok, probe_note = probe_persistent(local)
    use_persist = persist_ok if args.decode == 'auto' else (args.decode == 'persistent')
    if use_persist and not persist_ok:
        raise SystemExit(f'bench.py: --decode persistent, but the probe failed: {probe_note}')
    probe = make_rec(True) if use_persist else None
    L = args.lanes if args.lanes > 0 else (3 if use_persist else 16)
    L = max(1, L)
    # lone-batch diagnostics: one recogniser per decode path (graph path captured under the latency tile policy)
    rec_graph, rec_pers = make_rec(False), probe
    with torch.no_grad():
        for i in range(3):
            rec_graph.recognize_ids(*ring_dev[i])
            if rec_pers is not None:
                rec_pers.recognize_ids(*ring_dev[i])
    torch.cuda.synchronize()
    policy = args.tile_policy if args.tile_policy != 'auto' else ('throughput' if (L > 1 and not use_persist) else 'latency')
    ops.set_tile_policy(policy)
    lanes = [(torch.cuda.Stream(device=dev), make_rec(use_persist)) for _ in range(L)]

    def step_resident(rec, i):
        x, m = ring_dev[i % RING]
        return rec.recognize_ids(x, m)

    out_pin = {}

    def step_e2e(rec, i):
        xp, mp = ring_pin[i % RING]
        xd = xp.to(dev, non_blocking=True)
        md = mp.to(dev, non_blocking=True)
        out, scores = rec.recognize(xd, md)              # public API (ids because idx2unit is None)
        bufs = out_pin.get(id(rec))
        if bufs is None or bufs[0].shape != out.shape:
            bufs = (torch.empty(out.shape, dtype=out.dtype).pin_memory(), torch.empty(scores.shape, dtype=scores.dtype).pin_memory(),
                    torch.cuda.Event(blocking=True))
            out_pin[id(rec)] = bufs
        bufs[0].copy_(out, non_blocking=True)            # results land in pinned host memory; one (sleeping) sync per step
        bufs[1].copy_(scores, non_blocking=True)
        bufs[2].record()
        bufs[2].synchronize()
        return bufs

    last_out = {}

    def timed(fn, steps, n_lanes, recs=None):
        """K steps spread round-robin over n_lanes host threads / CUDA streams; device time by CUDA events.  What step K - 1
        returned is left in last_out['step']."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        errs = []

        def worker(j):
            try:
                torch.cuda.set_device(local)
                st, rec = lanes[j]
                if recs is not None:
                    rec = recs[j]
                st.wait_event(e0)
                with torch.cuda.stream(st):
                    for i in range(j, steps, n_lanes):
                        out = fn(rec, i)
                        if i == steps - 1:
                            last_out['step'] = out
            except Exception as ex:  # surface worker failures in the main thread
                errs.append(ex)

        if n_lanes == 1:
            worker(0)
        else:
            ts = [threading.Thread(target=worker, args=(j,)) for j in range(n_lanes)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        if errs:
            raise errs[0]
        for st, _ in lanes[:n_lanes]:
            torch.cuda.current_stream().wait_stream(st)
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    # warm-up: every lane runs sequentially (graph capture must not overlap other threads' CUDA calls)
    for st, rec in lanes:
        with torch.cuda.stream(st):
            for i in range(max(args.warmup, 3)):
                step_resident(rec, i)
            step_e2e(rec, 0)
        st.synchronize()

    # ---- diagnostics outside the headline region: encoder-only time and lone-batch latency of both decode paths
    def enc_only(rec, i):
        with torch.no_grad():
            return rec._encode_bf16(*ring_dev[i % RING])
    timed(enc_only, 8, 1)                           # untimed: first pass after the graph captures
    ms_enc = timed(enc_only, 16, 1) / 16
    ms_lat_graph = timed(step_resident, 4, 1, [rec_graph]) / 4
    ms_lat_pers = timed(step_resident, 8, 1, [rec_pers]) / 8 if rec_pers is not None else float('nan')
    ms_lat = ms_lat_pers if use_persist else ms_lat_graph
    # device duration of the persistent kernel alone (events on its own stream around the single launch)
    dec_kernel_ms = float('nan')
    if rec_pers is not None:
        with torch.no_grad():
            mem0, len0, B0, T20 = rec_pers._encode_bf16(*ring_dev[0])
            bd0 = rec_pers._decoder_for(B0, T20, dev)
            ts = []
            for _ in range(6):
                bd0.setup(mem0, len0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                bd0.run_persistent(MAX_LEN)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            dec_kernel_ms = sorted(ts)[len(ts) // 2]
    # reference ids of batch 0 for the output check (resident pass on lane 0)
    with torch.no_grad():
        ids0, scores0, steps0 = lanes[0][1].recognize_ids(*ring_dev[0])
        ids0 = ids0.clone()
    torch.cuda.synchronize()

    # K steps over L lanes run in ceil(K/L) rounds; when the last round would be mostly empty (K = 20, L = 16), fewer lanes
    # with full rounds finish sooner (K = 20 -> 2 rounds of 10)
    rounds = -(-args.steps // L)
    L_eff = min(L, -(-args.steps // rounds))
    # group barrier of the persistent kernel: a cluster of 16 CTAs fills a GPC, so clusters cap the GPU at 8 row groups in
    # flight; 3 batches x 3 groups want 9 -> plain CTAs + the software barrier (all 148 SMs) for the multi-lane region, the
    # hardware cluster barrier for the lone-batch latency above (ops.set_decode_barrier, include/otb200.h)
    groups = -(-B_PER_GPU // max(1, 128 // BEAM))
    grp_barrier = args.barrier if args.barrier != 'auto' else ('software' if (use_persist and L_eff * groups > 8) else 'default')
    if use_persist:
        ops.set_decode_barrier(grp_barrier)
    if L > 1:
        timed(step_resident, 2 * L, L)      # untimed multi-lane pass: thread start-up, allocator growth per stream
    # The timed region is exactly `steps` steps between barrier + synchronize, after an untimed pass of the same shape;
    # --min-ms > 0 repeats it until that much device time has been measured and reports the mean.
    probe_ms = timed(step_resident, args.steps, L_eff)
    repeats = int(min(64, max(1, -(-args.min_ms // max(probe_ms, 1e-3)))))
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    n0 = ops.COUNTERS['launches']
    res_ms = [timed(step_resident, args.steps, L_eff) for _ in range(repeats)]
    launches = (ops.COUNTERS['launches'] - n0) // repeats
    last_step = None
    if args.dump_outputs:
        ids_last, scores_last, steps_last = last_out['step']
        last_step = {'ids': ids_last.cpu(), 'scores': scores_last.cpu(), 'steps': steps_last}
    if L > 1:
        timed(step_e2e, 2 * L, L)           # untimed: per-stream allocator pools and pinned result buffers of the e2e path
    e2e_ms = [timed(step_e2e, args.steps, L_eff) for _ in range(repeats)]
    clocks = sampler.stop() if sampler else None
    if last_step is not None and rank == 0:
        dump_outputs(args.dump_outputs, last_step)
    ms_total, ms_e2e = sum(res_ms) / repeats, sum(e2e_ms) / repeats

    t = torch.tensor([ms_total, ms_e2e, ms_enc, ms_lat, ms_lat_graph, dec_kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_enc, ms_lat, ms_lat_graph, dec_kernel_ms = t.tolist()

    line = None
    if rank == 0:
        peaks, src = measured_peaks()
        peak_tf, peak_tf_burst, peak_bw = peaks.get('bf16_tflops_sustained', 1400.0), peaks.get('bf16_tflops', 1590.0), peaks.get('hbm_gbs', 6650.0)
        T2 = ops.conv_geometry(T_FRAMES, F_BINS)[2]
        w_bytes, kv_bytes = decode_step_bytes(model, B_PER_GPU, T2)
        ms_step = ms_total / args.steps
        dec_bytes = MAX_LEN * (w_bytes + kv_bytes)
        enc_bytes = 0.15e9                          # SURVEY.md 8(d): weights + input + 12 x (read + write [M,256] bf16)
        def fr(flop, nbytes, ms, tf_peak):
            return {'tflops': flop / (ms * 1e-3) / 1e12, 'frac_tensor': flop / (ms * 1e-3) / 1e12 / tf_peak,
                    'gbs': nbytes / (ms * 1e-3) / 1e9, 'frac_hbm': nbytes / (ms * 1e-3) / 1e9 / peak_bw}
        traffic = None
        try:    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
            with open(os.path.join(ROOT, 'profiles', 'r2_traffic.json')) as f:
                traffic = json.load(f).get('decode_group_kernel' if use_persist else 'gemm_tc_kernel')
        except Exception:
            pass
        if use_persist:
            # dominant kernel = the persistent decode kernel: one launch per batch, ~90 % of the device time of a pass
            ach = dec_bytes / (dec_kernel_ms * 1e-3) / 1e9
            roofline = {'bound': 'hbm', 'achieved': ach, 'peak': peak_bw, 'unit': 'GB/s', 'frac': ach / peak_bw, 'traffic': traffic,
                        'kernel': f'decode_group_kernel (csrc/decode_group.cu): ONE launch = the whole {MAX_LEN}-step beam-{BEAM} decode of {B_PER_GPU} '
                                  f'utterances on 3 row groups x 16 CTAs; {dec_kernel_ms:.2f} ms per launch (CUDA events on its stream, lone batch, '
                                  f'median of 6); algorithmic bytes per launch = {MAX_LEN} steps x ({w_bytes / 1e6:.1f} MB decoder weights + '
                                  f'{kv_bytes / 1e6:.1f} MB cross-attention K/V) = {dec_bytes / 1e9:.2f} GB (SURVEY.md 8d), {DEC_FLOP / 1e9:.0f} GFLOP; '
                                  'latency-bound: 38 group barriers and ~60 dependent phases per step (profiles/r2_decode_phases_*.txt); the self-attention '
                                  'K/V prefix (<= 133 MB per batch, read through an ancestry table) is not counted in the algorithmic bytes',
                        'alt': fr(DEC_FLOP, dec_bytes, dec_kernel_ms, peak_tf_burst),
                        'peak_source': f'MEASURED_PEAKS.json ({src}); burst bf16 figure for the lone kernel, sustained for whole steps'}
        else:
            roofline = graph_path_roofline(model, lanes, ring_dev, dev, peaks, src, traffic)
        roofline['whole_step'] = dict(fr(ENC_FLOP + DEC_FLOP, enc_bytes + dec_bytes, ms_step, peak_tf),
                                      note=f'(410 + 540) GFLOP and {(enc_bytes + dec_bytes) / 1e9:.2f} GB algorithmic per 32-utterance pass over '
                                           f'ms_per_step = {ms_step:.3f} ms ({L_eff} batches in flight)')
        roofline['lone_batch'] = dict(fr(ENC_FLOP + DEC_FLOP, enc_bytes + dec_bytes, ms_lat, peak_tf), ms=ms_lat)
        roofline['encoder_forward'] = dict(fr(ENC_FLOP, enc_bytes, ms_enc, peak_tf), ms=ms_enc)
        utt = B_PER_GPU * world * args.steps
        value = utt / (ms_total * 1e-3)
        e2e = utt / (ms_e2e * 1e-3)
        cfg = workload_config(args, B_PER_GPU)
        cfg['lanes'] = L_eff
        cfg['decode_path'] = 'persistent (one launch per batch)' if use_persist else 'per-step CUDA graph'
        cfg['persistent_probe'] = probe_note
        cfg['group_barrier'] = ({'default': 'cluster (hardware)', 'cluster': 'cluster (hardware)', 'software': 'software (L2 counter)'}[grp_barrier]
                                if use_persist else None)
        cfg['tile_policy'] = policy
        cfg['repeats'] = repeats
        # output check: digest of the n-best ids of input batch 0 against the committed one (tools/make_bench_digest.py runs
        # the bf16-policy oracle on the same inputs / weights in the build container)
        digest = ids_digest(ids0)
        expected, oracle_agree = None, None
        try:
            with open(os.path.join(ROOT, 'tests', 'golden', 'bench_digest.json')) as f:
                dg = json.load(f)
            expected = dg.get('gpu_persistent' if use_persist else 'gpu_graph')
            if rank == 0 and 'oracle_ids' in dg:       # 1-best of the bf16-policy oracle on the same 32 utterances
                oid = torch.tensor(dg['oracle_ids'], dtype=torch.int64)
                if tuple(oid.shape) == tuple(ids0[:, 0].shape):
                    oracle_agree = int((oid == ids0[:, 0].cpu()).all(dim=1).sum())
        except Exception:
            pass
        line = {
            'metric': 'utterances/sec (encoder-fwd + beam-10 decode, 60 steps)', 'value': value, 'unit': 'utt/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16', 'data': 'synthetic', 'config': cfg,
            'e2e': {'value': e2e, 'unit': 'utt/s', 'h2d_bytes_per_step': ring_cpu[0][0].numel() * 4 + ring_cpu[0][1].numel(),
                    'd2h_bytes_per_step': B_PER_GPU * MAX_LEN * 8 + B_PER_GPU * 4},
            'gpu_launches': launches,
            'breakdown': {'single_lane_step_ms': ms_lat, 'single_lane_utt_per_s': B_PER_GPU * world / (ms_lat * 1e-3),
                          'encoder_fwd_ms': ms_enc, 'encoder_fwd_utt_per_s': B_PER_GPU * world / (ms_enc * 1e-3),
                          'beam_decode_ms': ms_lat - ms_enc,
                          'beam_decode_utt_per_s': B_PER_GPU * world / ((ms_lat - ms_enc) * 1e-3),
                          'persistent_decode_kernel_ms': dec_kernel_ms,
                          'graph_path_single_lane_step_ms': ms_lat_graph,
                          'timed_region_ms': {'mean': ms_total, 'min': min(res_ms), 'max': max(res_ms), 'repeats': repeats}},
            'roofline': roofline,
            'validation': {'ids_sha1': digest, 'expected_sha1': expected, 'match': (digest == expected) if expected else None,
                           'steps_executed': int(steps0), 'one_best_equal_to_bf16_policy_oracle': oracle_agree,
                           'note': 'expected_sha1 = digest of the same decode path recorded on a B200 by tools/gpu_r2_digest.sh '
                                   '(regression check); the oracle count is informational: default-initialised weights give '
                                   'near-ties that bf16 rounding resolves differently'},
            'clocks': clocks,
        }
        if nccl_log:
            line['comm'] = nccl_summary(nccl_log, world)
        if args.cpu_baseline and world == 1:
            threads, cores = pick_cpu_threads()
            sd, params = flat_state_dict(model), model_params()
            xs, ms_ = ring_cpu[0][0][:args.ref_sample], ring_cpu[0][1][:args.ref_sample]
            rec_ref = reference_recognizer(model)
            t0 = time.perf_counter()
            if rec_ref is not None:      # the reference itself (oracle/_ref); the port runs afterwards, untimed, as the cross-check
                ref_rows = reference_ids(rec_ref, xs, ms_)
                dt = time.perf_counter() - t0
                nb_ref, _, _, _ = cpu_reference_pass(sd, params, xs, ms_)
                port_rows = [[int(t) for t in nb_ref[b, 0].tolist() if int(t) != 1] for b in range(args.ref_sample)]
                port_equal = sum(int(ref_rows[b] == port_rows[b]) for b in range(args.ref_sample))
            else:
                nb_ref, _, _, _ = cpu_reference_pass(sd, params, xs, ms_)
                dt = time.perf_counter() - t0
                port_equal = None
            same = sum(int(torch.equal(ids0[b, 0].cpu(), nb_ref[b, 0])) for b in range(args.ref_sample)) \
                if nb_ref.shape[2] == ids0.shape[2] else 0
            kind = 'reference' if rec_ref is not None else 'port'
            line['cpu_baseline'] = {'value': args.ref_sample / dt, 'unit': 'utt/s', 'cores': threads,
                                    'visible_cores': cores, 'kind': kind,
                                    'sample': f'{args.ref_sample} utterances (the first of input batch 0), one full pass '
                                              f'(encoder-fwd + 60-step beam-10 decode) of '
                                              + ('the reference\'s own recogniser (oracle/_ref)' if kind == 'reference' else 'the oracle port')
                                              + f' in {dt:.1f} s'}
            line['validation']['oracle_check'] = {'utterances': args.ref_sample, 'one_best_ids_equal': same,
                                                  'port_equals_reference': port_equal,
                                                  'note': 'fp32 oracle port vs the CUDA path on the same utterances; '
                                                          'port_equals_reference: 1-best of the port vs the reference itself (oracle/_ref)'}
    del lanes, rec_graph, rec_pers, probe
    torch.cuda.empty_cache()
    if args.extras:
        # BASELINE configs 4 and 5 ride along so that the driver's N = 1/2/4/8 runs also cover the Conformer path and the
        # only NCCL collective of the north star (the gradient all-reduce of the training step)
        ex = {}
        for name, fn in (('conformer_cfg4', measure_conformer), ('train_cfg5', measure_train)):
            try:
                r = fn(args, min(args.steps, 12))
                if rank == 0:
                    ex[name] = r
            except Exception as exn:  # an extra must never cost the headline line
                if rank == 0:
                    ex[name] = {'error': repr(exn)[:300]}
        if rank == 0:
            line['extras'] = ex
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def probe_persistent(local):
    """Run `bench.py --probe-persistent` in a child process: (ok, note).  ok = the persistent decode kernel supports the
    benchmark configuration AND returned the same n-best ids / step count as the per-step graph path on input batch 0."""
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT', 'TORCHELASTIC_RUN_ID'):
        env.pop(k, None)
    env['OTB_PROBE_DEVICE'] = str(local)
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), '--probe-persistent'], env=env, capture_output=True, text=True,
                           timeout=300)
    except subprocess.TimeoutExpired:
        return False, 'probe timed out'
    last = (r.stdout.strip().splitlines() or [''])[-1]
    if r.returncode == 0 and last.startswith('PROBE OK'):
        return True, last
    return False, ('rc %d: ' % r.returncode) + (last or r.stderr.strip()[-200:])


def run_probe_persistent():
    """Child process of probe_persistent: the persistent kernel against the per-step graph path on input batch 0.  The two
    are different bf16 pipelines (different rounding points), so lower-ranked hypotheses may legitimately differ; required:
    same executed step count, deterministic output, finite scores within tolerance, 1-best ids equal for >= 90 % of the batch."""
    from opentransformer_b200.recognize import SpeechToTextRecognizer
    dev = torch.device('cuda', int(os.environ.get('OTB_PROBE_DEVICE', '0')))
    torch.cuda.set_device(dev)
    model = build_model().to(dev)
    x, m = synthetic_batch(B_PER_GPU, 0)
    x, m = x.to(dev), m.to(dev)
    kw = dict(beam_width=BEAM, nbest=1, max_len=MAX_LEN, penalty=PENALTY, lamda=LAMDA, ngpu=1)
    rp, rg = SpeechToTextRecognizer(model, persistent=True, **kw), SpeechToTextRecognizer(model, persistent=False, **kw)
    pp, sp, n_p = rp.recognize_ids(x, m)
    if not next(iter(rp._decoders.values())).persistent:
        print('PROBE FAIL persistent kernel does not support this configuration')
        return 1
    pg, sg, n_g = rg.recognize_ids(x, m)
    pp2, _, _ = rp.recognize_ids(x, m)
    torch.cuda.synchronize()
    agree = int((pp[:, 0] == pg[:, 0]).all(dim=1).sum()) if n_p == n_g else 0
    dscore = float((sp - sg).abs().max())
    ok = (n_p == n_g and bool(torch.equal(pp, pp2)) and bool(torch.isfinite(sp).all()) and agree >= 0.9 * B_PER_GPU
          and dscore < 0.3 + 3e-2 * float(sg.abs().max()))
    print(('PROBE OK' if ok else 'PROBE FAIL') + f' steps {n_p}/{n_g}, 1-best ids equal to the graph path for {agree}/{B_PER_GPU} '
          f'utterances, deterministic: {bool(torch.equal(pp, pp2))}, max |score diff| {dscore:.3e}')
    return 0 if ok else 1


def graph_path_roofline(model, lanes, ring_dev, dev, peaks, src, traffic):
    """Per-step CUDA-graph decode path: dominant kernel = the GEMM launch shape with the largest device time per recognize
    pass; launch counts from recorded eager passes, durations from a CUDA graph of 200 launches (device-measured)."""
    from opentransformer_b200 import ops
    from opentransformer_b200.recognize import BeamDecoder
    rec = lanes[0][1]
    ops.PROFILE = []
    with torch.no_grad():
        for i in range(2):
            rec._encode_bf16(*ring_dev[i])
        mem0, len0, B0, T20 = rec._encode_bf16(*ring_dev[0])
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, []
        bd0 = BeamDecoder(model.decoder, B0, BEAM, T20, MAX_LEN, dev, use_graph=False, keep_logp=False)
        bd0.setup(mem0, len0)
        for _ in range(8):
            bd0.step()
        torch.cuda.synchronize()
    prof_dec, ops.PROFILE = ops.PROFILE, None
    epi_names = ['bias', 'relu', 'glu', 'posenc-table', 'residual', 'residual+layernorm', 'swish', 'gelu', 'tanh']
    shapes = {}
    for records, per_pass in ((prof, 1.0 / 3), (prof_dec, MAX_LEN / 8.0)):
        for k, f, a, b, tag in records:
            if k == 'gemm':
                e = shapes.setdefault(tag, {'launches_per_pass': 0.0})
                e['launches_per_pass'] += per_pass
    for tag, e in shapes.items():
        e['avg_ms'] = time_gemm_shape(tag, dev)
        e['ms_per_pass'] = e['avg_ms'] * e['launches_per_pass']
    tag, e = max(shapes.items(), key=lambda kv: kv[1]['ms_per_pass'])
    epi, M_, Nw_, K_, _of32 = tag
    avg_ms = e['avg_ms']
    flops = 2.0 * M_ * Nw_ * K_
    n_out = Nw_ // 2 if epi == 2 else Nw_
    nbytes = 2.0 * (M_ * K_ + Nw_ * K_ + M_ * n_out) + (2.0 * M_ * n_out if epi in (4, 5) else 0.0)
    tf, gbs = flops / (avg_ms * 1e-3) / 1e12, nbytes / (avg_ms * 1e-3) / 1e9
    peak_tf, peak_bw = peaks.get('bf16_tflops', 1590.0), peaks.get('hbm_gbs', 6650.0)
    use_hbm = gbs / peak_bw > tf / peak_tf
    ach, peak = (gbs, peak_bw) if use_hbm else (tf, peak_tf)
    return {'bound': 'hbm' if use_hbm else 'tensor', 'achieved': ach, 'peak': peak, 'unit': 'GB/s' if use_hbm else 'TFLOP/s',
            'frac': ach / peak if peak else None, 'traffic': traffic,
            'kernel': f'gemm_tc_kernel, epilogue {epi_names[epi]}, M={M_} N={Nw_} K={K_}: {e["launches_per_pass"]:.0f} launches and '
                      f'{e["ms_per_pass"]:.2f} ms per recognize pass, avg {avg_ms * 1e3:.1f} us per launch (CUDA graph of 200 launches '
                      f'between events); algorithmic {flops / 1e9:.3f} GFLOP and {nbytes / 1e6:.2f} MB per launch',
            'alt': {'tflops': tf, 'frac_tensor': tf / peak_tf, 'gbs': gbs, 'frac_hbm': gbs / peak_bw},
            'all_gemm_shapes_ms_per_pass': {('%s_M%d_N%d_K%d' % (epi_names[t[0]], t[1], t[2], t[3])): round(v['ms_per_pass'], 3)
                                            for t, v in sorted(shapes.items(), key=lambda kv: -kv[1]['ms_per_pass'])[:8]},
            'peak_source': f'MEASURED_PEAKS.json ({src})'}


def conformer_params():
    """egs/aishell/conf/conformer_baseline.yaml with the SURVEY.md 8(d) config-4 overrides (d_model 256,
    residual_dropout 0.0 because the reference applies dropout in eval mode otherwise)."""
    p = model_params()
    p['encoder_type'] = 'conformer'
    p['frontend'].update(mid_channel=256, out_channel=256)
    p['encoder'] = dict(d_model=256, d_ff=768, cov_kernel_size=5, n_heads=4, nblocks=12, pos_dropout=0.0,
                        slf_attn_dropout=0.0, ffn_dropout=0.0, residual_dropout=0.0, conv_dropout=0.0,
                        macaron_style=True, ffn_scale=0.5, conv_bias=True, activation='glu',
                        positional_encoding=True, relative_positional=True)
    p['decoder'].update(d_ff=768)
    return p


def measure_conformer(args, steps):
    """BASELINE config 4: Conformer encoder forward, 64 x 1000 frames per GPU, utterance-sharded over ranks.
    Returns the result line (rank 0) -- used both as the main line of --workload conformer and as an extra of the default run."""
    import torch.distributed as dist
    from opentransformer_b200.model import SpeechToText
    rank, world, local, dev, nccl_log = init_dist()
    torch.manual_seed(1234)
    model = SpeechToText(conformer_params()).eval().to(dev)
    B = 64
    ring = [tuple(t.to(dev) for t in synthetic_batch(B, 1000 * rank + i)) for i in range(8)]
    with torch.no_grad():
        # ~400 launches per pass: replayed from a CUDA graph (launched one by one from Python the pass is host-bound as soon
        # as several ranks share the host's cores), inputs copied into the graph's static buffers every step
        sx, sm = ring[0][0].clone(), ring[0][1].clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(max(args.warmup, 3)):
                model.encode_bf16(sx, sm)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = model.encode_bf16(sx, sm)

        def one_pass(i):
            sx.copy_(ring[i % 8][0])
            sm.copy_(ring[i % 8][1])
            graph.replay()
            return out
        for i in range(3):
            one_pass(i)
        dist_barrier(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            one_pass(i)
        e1.record()
        dist_barrier(world)
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    del graph, model, ring
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    peaks, src = measured_peaks()
    flop = 898.0e9      # SURVEY.md 8(d): ~898 GFLOP per 64-utterance batch
    ach = flop * steps / (ms * 1e-3) / 1e12
    return {'metric': 'utterances/sec (Conformer encoder forward)', 'value': B * world * steps / (ms * 1e-3),
            'unit': 'utt/s', 'n_gpus': world, 'steps': steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': 'Conformer encoder 12L d_model=256 d_ff=768 k=5 rel-pos, frontend 1->256->256, '
                                   f'{B} utt x {T_FRAMES} frames per GPU (BASELINE config 4)',
                       'parallelism': f'dp{world} (utterance sharding, no data-path collective)'},
            'roofline': {'bound': 'tensor', 'achieved': ach, 'peak': peaks.get('bf16_tflops_sustained'),
                         'unit': 'TFLOP/s', 'frac': ach / peaks.get('bf16_tflops_sustained', 1400.0),
                         'traffic': None, 'kernel': 'whole encoder pass (898 GFLOP algorithmic per batch)',
                         'peak_source': src}}


def run_conformer(args):
    import torch.distributed as dist
    line = measure_conformer(args, args.steps)
    if line is not None:
        emit(line)
    if dist.is_initialized():
        dist.destroy_process_group()
    return 0


def train_params():
    """BASELINE config 5: the config-2 model with every dropout rate 0 (the reference's residual_dropout 0.1 is stochastic;
    the B200 training path implements the deterministic network, DESIGN.md 6)."""
    p = model_params()
    for part in ('frontend', 'encoder', 'decoder'):
        for k in list(p[part]):
            if 'dropout' in k:
                p[part][k] = 0.0
    return p


def synthetic_targets(batch, seed):
    """collate_fn_with_eos_bos (data/loader.py:85-86): <S/E> ids <S/E> then PAD(0); 20-30 ids in [3, V)."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(20, 31, (batch,), generator=g)
    L = 32                                   # 30 ids + <S/E> on both sides: one step geometry for every batch
    t = torch.zeros(batch, L, dtype=torch.long)
    for b in range(batch):
        n = int(lens[b])
        t[b, 0] = 1
        t[b, 1:n + 1] = torch.randint(3, 4234, (n,), generator=g)
        t[b, n + 1] = 1
    return t


def measure_train(args, steps):
    """BASELINE config 5: one optimizer step per `step` -- SpecAugment (device) -> forward -> hand-written backward ->
    gradient all-reduce over NCCL (N > 1) -> global-norm clip + Adam.  32 utterances x 1000 frames per GPU (weak scaling:
    global batch 32 N; N = 8 is the reference's 256)."""
    import random
    import numpy as np
    import torch.distributed as dist
    from opentransformer_b200 import ops
    from opentransformer_b200.augment import spec_augment_
    from opentransformer_b200.model import SpeechToText
    from opentransformer_b200.train import FusedTrainer
    rank, world, local, dev, nccl_log = init_dist()
    torch.manual_seed(1234)                       # identical initial weights on every rank (run.py:23-33)
    model = SpeechToText(train_params()).to(dev).train()
    trainer = FusedTrainer(model, lr=1e-3, betas=(0.9, 0.98), eps=1e-9, weight_decay=1e-6, clip_grad=5.0, model_size=256,
                           warmup_steps=12000, accum_steps=1)
    random.seed(100 + rank)
    np.random.seed(100 + rank)
    RING = 8
    ring = []
    for i in range(RING):
        x, m = synthetic_batch(B_PER_GPU, 5000 * rank + i)
        ring.append((x.pin_memory(), m.pin_memory(), synthetic_targets(B_PER_GPU, 7000 * rank + i).pin_memory()))
    ring_dev = [tuple(t.to(dev) for t in item) for item in ring]
    lens = [T_FRAMES] * B_PER_GPU

    def barrier():
        dist_barrier(world)

    def step_resident(i):
        x, m, t = ring_dev[i % RING]
        xa = spec_augment_(x.clone(), lens)
        return trainer.step(xa, m, t)

    def step_e2e(i):
        xp, mp, tp = ring[i % RING]
        x = xp.to(dev, non_blocking=True)
        m = mp.to(dev, non_blocking=True)
        t = tp.to(dev, non_blocking=True)
        spec_augment_(x, lens)
        return float(trainer.step(x, m, t))        # the loss is read back every step (trainer.py:216)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    for i in range(max(args.warmup, 3)):
        step_resident(i)
    step_e2e(0)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    n0 = ops.COUNTERS['launches']
    ms = timed(step_resident, steps)
    launches = ops.COUNTERS['launches'] - n0
    ms_e2e = timed(step_e2e, steps)
    clocks = sampler.stop() if sampler else None
    final_loss = float(step_resident(0))
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    del trainer, model, ring_dev
    torch.cuda.empty_cache()
    if rank == 0:
        peaks, src = measured_peaks()
        # SURVEY.md 8(d): encoder-fwd 410.0 + teacher-forced decoder ~38.9 GFLOP per 32-utt batch; backward = 2x forward
        flop = 3.0 * (410.0e9 + 38.9e9)
        ach = flop * steps / (ms * 1e-3) / 1e12
        utt = B_PER_GPU * world * steps
        item = ring[0]
        line = {
            'metric': 'utterances/sec (training step: SpecAugment + fwd + bwd + grad all-reduce + clip + Adam)',
            'value': utt / (ms * 1e-3), 'unit': 'utt/s', 'n_gpus': world, 'steps': steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
            'data': 'synthetic',
            'config': {'workload': 'BASELINE config 5: training step, Speech-Transformer 12-enc/6-dec d_model=256, '
                                   f'{B_PER_GPU} utt x {T_FRAMES} frames per GPU, targets 20-30 tokens, label smoothing 0.1, '
                                   'SpecAugment on (2 freq + 2 time masks), Adam + Noam(256, 12000), clip 5, bf16 compute / fp32 '
                                   'master weights, all dropout rates 0',
                       'global_batch': B_PER_GPU * world, 'parallelism': f'dp{world} (one NCCL all-reduce of the flat fp32 gradient per step)',
                       'l2_policy': '8 distinct batches rotate; every step streams > 2 GB of activations / gradients'},
            'e2e': {'value': utt / (ms_e2e * 1e-3), 'unit': 'utt/s',
                    'h2d_bytes_per_step': item[0].numel() * 4 + item[1].numel() + item[2].numel() * 8, 'd2h_bytes_per_step': 4},
            'gpu_launches': launches, 'final_loss': final_loss,
            'roofline': {'bound': 'tensor', 'achieved': ach, 'peak': peaks.get('bf16_tflops_sustained'), 'unit': 'TFLOP/s',
                         'frac': ach / peaks.get('bf16_tflops_sustained', 1400.0), 'traffic': None,
                         'kernel': 'whole training step (3 x 448.9 GFLOP algorithmic per 32-utterance batch)',
                         'peak_source': src},
            'clocks': clocks}
        if nccl_log:
            line['comm'] = nccl_summary(nccl_log, world)
        return line
    return None


def run_train(args):
    import torch.distributed as dist
    line = measure_train(args, args.steps)
    if line is not None:
        emit(line)
    if dist.is_initialized():
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=96)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--ref-sample', type=int, default=2, help='utterances per CPU reference pass')
    ap.add_argument('--workload', default='transformer', choices=['transformer', 'conformer', 'train'],
                    help="'conformer' = BASELINE config 4 (encoder forward only), 'train' = config 5 (training step); "
                         "default is the headline workload")
    ap.add_argument('--lanes', type=int, default=0, help='utterance batches kept in flight per GPU (streams); 0 = auto: 3 for the '
                                                       'persistent decode kernel (48 SMs per batch), 16 for the per-step graph')
    ap.add_argument('--barrier', default='auto', choices=['auto', 'cluster', 'software'],
                    help='group barrier of the persistent decode kernel in the timed multi-lane region (auto: software when more than 8 '
                         'row groups are in flight, else thread-block clusters)')
    ap.add_argument('--decode', default='auto', choices=['auto', 'persistent', 'graph'],
                    help='decode path: one persistent launch per batch (csrc/decode_group.cu) or one CUDA-graph replay per step')
    ap.add_argument('--min-ms', type=float, default=0.0,
                    help='repeat the timed K-step region until this much device time is measured (default: time it once)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned (n-best ids, scores, executed decode steps; '
                         'rank 0) as DIR/<name>.npy, so that two builds can be compared on identical inputs')
    ap.add_argument('--no-extras', dest='extras', action='store_false',
                    help='skip the BASELINE config 4 / 5 measurements appended to the default run')
    ap.add_argument('--tile-policy', default='auto', choices=['auto', 'latency', 'throughput'],
                    help='tiling of the decode-step GEMMs (otb_set_tile_policy); auto = throughput when lanes > 1')
    ap.add_argument('--no-cpu-baseline', dest='cpu_baseline', action='store_false')
    ap.add_argument('--probe-persistent', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.probe_persistent:
        return run_probe_persistent()
    if args.dump_outputs and (args.impl != 'b200' or args.workload != 'transformer'):
        ap.error('--dump-outputs applies to the B200 path of the transformer workload')
    guard_stdout()
    if args.impl == 'reference':
        return run_reference(args)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference)')
    if args.workload == 'conformer':
        return run_conformer(args)
    if args.workload == 'train':
        return run_train(args)
    return run_b200(args)


if __name__ == '__main__':
    sys.exit(main())
