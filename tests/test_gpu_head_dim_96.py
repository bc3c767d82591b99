"""GPU parity of the 96-wide attention heads (d_model 384 with 4 heads, the shipped Conformer recipe) against a plain fp32
torch restatement on bf16-rounded operands: the tcgen05 attention kernel (padding, causal, cross, rel-pos band +
residual, log-sum-exp), the K = 96 head-view GEMMs of the rel-pos band and the KV-cached decode self-attention.
Run with -m gpu on a B200."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from opentransformer_b200 import ops
    DEV = torch.device('cuda:0')
BF = torch.bfloat16
HD = 96
torch.backends.cuda.matmul.allow_tf32 = False


def _rnd(*shape, scale=1.0, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _check(name, got, ref, tol_rel, tol_abs=0.0):
    got, ref = got.float(), ref.float()
    rel = float((got - ref).norm() / (ref.norm() + 1e-12))
    worst = float((got - ref).abs().max())
    lim = tol_abs + 8 * tol_rel * float(ref.abs().max())
    print(f'{name}: rel_l2={rel:.3e} max_abs={worst:.3e} (limit {lim:.3e})')
    assert not torch.isnan(got).any() and rel <= tol_rel and worst <= lim, name


def _heads(x, B, T, H):
    return x.float().view(B, T, H, HD).transpose(1, 2)


def _attn_ref(q, k, v, B, H, Tq, Tk, kv_len, causal, band=None):
    """softmax((q k^T + band) / sqrt(96)) v over the visible keys; returns (out [B*Tq, H*96], lse in log2 units [B,H,Tq])."""
    s = _heads(q, B, Tq, H) @ _heads(k, B, Tk, H).transpose(2, 3)
    if band is not None:
        s = s + band
    s = s / math.sqrt(HD)
    mask = (torch.arange(Tk, device=DEV)[None, :] < kv_len[:, None].long())[:, None, None, :].expand(B, H, Tq, Tk)
    if causal:
        mask = mask & torch.tril(torch.ones(Tq, Tk, dtype=torch.bool, device=DEV))[None, None]
    s = s.masked_fill(~mask, float('-inf'))
    out = (torch.softmax(s, -1) @ _heads(v, B, Tk, H)).transpose(1, 2).reshape(B * Tq, H * HD)
    return out, torch.logsumexp(s, -1) / math.log(2.0)


@pytest.mark.parametrize('B,T,lens', [(3, 249, [249, 200, 1]), (2, 300, [300, 129]), (3, 300, [1, 300, 257]),
                                      (2, 1, [1, 1])])
def test_self_attention_hd96_padding(B, T, lens):
    H = 4
    d = H * HD
    qkv = _rnd(B * T, 3 * d, seed=1).to(BF)
    kv_len = torch.tensor(lens, dtype=torch.int32, device=DEV)
    out = ops.attention(qkv, qkv, qkv, B, H, T, T, kv_len=kv_len, q_col0=0, k_col0=d, v_col0=2 * d, head_dim=HD)
    ref, _ = _attn_ref(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], B, H, T, T, kv_len, False)
    _check(f'self-attn hd96 [{B},{T},{lens}]', out, ref, 6e-3)


@pytest.mark.parametrize('B,L', [(1, 1), (3, 30), (2, 130)])
def test_causal_attention_hd96_with_lse(B, L):
    H = 4
    d = H * HD
    qkv = _rnd(B * L, 3 * d, seed=2).to(BF)
    full = torch.full((B,), L, dtype=torch.int32, device=DEV)
    out, lse = ops.attention_train(qkv, qkv, qkv, B, H, L, L, causal=True, q_col0=0, k_col0=d, v_col0=2 * d, head_dim=HD)
    ref, lse_ref = _attn_ref(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], B, H, L, L, full, True)
    _check(f'causal-attn hd96 [{B},{L}]', out, ref, 6e-3)
    _check(f'causal-attn hd96 lse [{B},{L}]', lse, lse_ref, 1e-4, 1e-3)
    plain = ops.attention(qkv, qkv, qkv, B, H, L, L, causal=True, q_col0=0, k_col0=d, v_col0=2 * d, head_dim=HD)
    assert torch.equal(plain, out)


@pytest.mark.parametrize('B,Tq,Tk', [(4, 10, 249), (3, 1, 249)])
def test_cross_attention_hd96(B, Tq, Tk):
    H = 4
    d = H * HD
    q = _rnd(B * Tq, d, seed=3).to(BF)
    kv = _rnd(B * Tk, 2 * d, seed=4).to(BF)
    g = torch.Generator().manual_seed(9)
    kv_len = torch.randint(1, Tk + 1, (B,), generator=g).to(torch.int32).to(DEV)
    out = ops.attention(q, kv, kv, B, H, Tq, Tk, kv_len=kv_len, k_col0=0, v_col0=d, head_dim=HD)
    ref, _ = _attn_ref(q, kv[:, :d], kv[:, d:], B, H, Tq, Tk, kv_len, False)
    _check(f'cross-attn hd96 [{B},{Tq},{Tk}]', out, ref, 6e-3)


def test_attention_hd96_heads_at_the_matrix_edge():
    """q, k and v as separate [M, 384] matrices: the last head's 32-column box ends at the right edge of each matrix and
    the last row tile runs past the bottom edge; the strided output lands in the middle of a wider buffer."""
    B, H, T = 3, 4, 200
    d = H * HD
    q, k, v = (_rnd(B * T, d, seed=s).to(BF) for s in (5, 6, 7))
    kv_len = torch.tensor([200, 77, 131], dtype=torch.int32, device=DEV)
    wide = torch.full((B * T, d + 128), 7.0, dtype=BF, device=DEV)
    ops.attention(q, k, v, B, H, T, T, kv_len=kv_len, out=wide[:, 64:64 + d], head_dim=HD)
    ref, _ = _attn_ref(q, k, v, B, H, T, T, kv_len, False)
    _check('edge heads hd96', wide[:, 64:64 + d], ref, 6e-3)
    assert bool((wide[:, :64] == 7.0).all()) and bool((wide[:, 64 + d:] == 7.0).all()), 'wrote outside the output view'


def test_relpos_band_and_residual_attention_hd96():
    """scores = (q k^T + BD[i, j-i+T-1]) / sqrt(96) with ragged lengths, output added to a residual (no out-projection)."""
    B, H, T = 3, 4, 150
    d = H * HD
    qkv = _rnd(B * T, 3 * d, seed=1).to(BF)
    ld = (2 * T - 1 + 3) // 4 * 4
    bd = _rnd(H, B * T, ld, scale=2.0, seed=2)
    res = _rnd(B * T, d, seed=3).to(BF)
    lens = torch.tensor([150, 90, 129], dtype=torch.int32, device=DEV)
    out = ops.attention(qkv, qkv, qkv, B, H, T, T, kv_len=lens, q_col0=0, k_col0=d, v_col0=2 * d, bd=bd, resid=res,
                        head_dim=HD)
    idx = (torch.arange(T, device=DEV)[None, :] - torch.arange(T, device=DEV)[:, None]) + (T - 1)
    full = bd.view(H, B, T, ld).permute(1, 0, 2, 3)[..., :2 * T - 1]
    band = torch.gather(full, 3, idx.view(1, 1, T, T).expand(B, H, T, T))
    ref, _ = _attn_ref(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], B, H, T, T, lens, False, band=band)
    _check('relpos-attn+resid hd96', out, ref + res.float(), 6e-3)


def test_linear_on_96_column_head_views():
    """BD_full[h] = (q+v)_h P_h^T at K = 96: the second 64-column k-block of every head view would reach 32 columns into the
    next head (or the next operand) if the TMA maps were not bounded by the view's width."""
    M, d, R = 500, 384, 497
    ext = _rnd(M, 4 * d, seed=1).to(BF)
    pp = _rnd(R, d, seed=2).to(BF)
    out = torch.empty(M, 500, device=DEV)
    for h in range(4):
        a, w = ext[:, d + HD * h: d + HD * (h + 1)], pp[:, HD * h: HD * (h + 1)]
        ops.linear(a, w, out=out)
        _check(f'head-view gemm K=96 h={h}', out[:, :R], a.float() @ w.float().t(), 2e-5, 1e-4)


@pytest.mark.parametrize('N,H,Lmax', [(12, 4, 60), (40, 4, 128)])
def test_decode_self_attention_hd96_over_steps(N, H, Lmax):
    """Several consecutive steps with a permuted ancestry table, against a torch gather restatement; the newest K/V row is
    appended to the cache at every step."""
    d = H * HD
    kc = _rnd(Lmax, N, d, seed=2).to(BF)
    vc = _rnd(Lmax, N, d, seed=3).to(BF)
    g = torch.Generator().manual_seed(4)
    anc = torch.stack([torch.stack([torch.randperm(N, generator=g) for _ in range(Lmax)], 1) for _ in range(2)])
    anc = anc.to(torch.int32).to(DEV)                                               # [2, N, Lmax]
    steps = [0, 1, 2, 45, Lmax - 1] if Lmax == 60 else [0, 31, 32, 100, Lmax - 1]
    for step in steps:
        qkv = _rnd(N, 3 * d, seed=10 + step).to(BF)
        ctrl = torch.tensor([step, 0, 0, 0], dtype=torch.int32, device=DEV)
        kc0, vc0 = kc.clone(), vc.clone()
        out = ops.decode_self_attn(qkv, kc, vc, anc, ctrl, N, H, Lmax, head_dim=HD)
        cur = anc[step & 1].long()
        ks = torch.stack([kc0[s, cur[:, s]] for s in range(step)] + [qkv[:, d:2 * d]], 1).float()
        vs = torch.stack([vc0[s, cur[:, s]] for s in range(step)] + [qkv[:, 2 * d:]], 1).float()
        q = qkv[:, :d].float().view(N, H, 1, HD)
        s = (q @ ks.view(N, step + 1, H, HD).transpose(1, 2).transpose(2, 3)) / math.sqrt(HD)
        ref = (torch.softmax(s, -1) @ vs.view(N, step + 1, H, HD).transpose(1, 2)).reshape(N, d)
        _check(f'decode self-attn hd96 N={N} step={step}', out, ref, 6e-3)
        assert torch.equal(kc[step], qkv[:, d:2 * d]) and torch.equal(vc[step], qkv[:, 2 * d:])
        assert torch.equal(kc[:step], kc0[:step]) and torch.equal(kc[step + 1:], kc0[step + 1:])
